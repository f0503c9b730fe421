"""numpy front-end of tests/stack_bq_oracle.c, the CPU restatement of the reference's stacked ball query (TEST
INFRASTRUCTURE).  The library is compiled on first use into the temporary directory (keyed by the source's hash), so
the repository tree is never written."""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stack_bq_oracle.c")
_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        digest = hashlib.sha256(open(_SRC, "rb").read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"tsmdet_stack_bq_oracle_{digest}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            # -ffp-contract=off: only the explicit fmaf() fuses (the FFMA placement nvcc chose for the reference kernel)
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-fvisibility=hidden", "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def stack_ball_query(radius: float, nsample: int, xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt):
    """ball_query_gpu.cu (stack):15-62 -> idx (M,nsample), the raw kernel output (frame-local rows, idx[:,0] == -1
    marks an empty ball; pointnet2_utils.py (stack) then zeroes those rows)."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
    new_xyz = np.ascontiguousarray(new_xyz, dtype=np.float32).reshape(-1, 3)
    nb = np.ascontiguousarray(xyz_batch_cnt, dtype=np.int32)
    mb = np.ascontiguousarray(new_xyz_batch_cnt, dtype=np.int32)
    m = new_xyz.shape[0]
    idx = np.zeros((m, nsample), dtype=np.int32)
    f32p, i32p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int32)
    lib().sbq_stack_ball_query(len(nb), m, ctypes.c_float(radius), nsample, new_xyz.ctypes.data_as(f32p),
                               mb.ctypes.data_as(i32p), xyz.ctypes.data_as(f32p), nb.ctypes.data_as(i32p),
                               idx.ctypes.data_as(i32p))
    return idx
