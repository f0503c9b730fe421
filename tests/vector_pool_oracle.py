"""numpy front-end of tests/vector_pool_oracle.c, the CPU restatement of pointnet2_stack's vector-pool functions (TEST
INFRASTRUCTURE).  The library is compiled on first use into the temporary directory (keyed by the source's hash), so
the repository tree is never written."""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

CAP = 1000
_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "vector_pool_oracle.c")
_lib = None
_f = ctypes.POINTER(ctypes.c_float)
_i = ctypes.POINTER(ctypes.c_int32)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        digest = hashlib.sha256(open(_SRC, "rb").read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"tsmdet_vector_pool_oracle_{digest}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            # -ffp-contract=off: only the explicit fmaf() fuses (the distance contraction of the stack kernels)
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-fvisibility=hidden", "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
        _lib.vpo_pool.restype = ctypes.c_longlong
    return _lib


def _f32(a, cols=3):
    return np.ascontiguousarray(a, dtype=np.float32).reshape(-1, cols)


def local_lists(xyz, xyz_cnt, new_xyz, new_cnt, d, nsample, neighbor_type):
    """-> [list of GLOBAL support rows per centre]: the first min(hits, 1000, nsample if > 0) hits in index order"""
    xyz, new_xyz = _f32(xyz), _f32(new_xyz)
    nb, mb = np.ascontiguousarray(xyz_cnt, np.int32), np.ascontiguousarray(new_cnt, np.int32)
    m = new_xyz.shape[0]
    lists = np.zeros((max(m, 1), CAP), np.int32)
    lens = np.zeros(max(m, 1), np.int32)
    lib().vpo_local_idxs(len(nb), m, xyz.ctypes.data_as(_f), nb.ctypes.data_as(_i), new_xyz.ctypes.data_as(_f),
                         mb.ctypes.data_as(_i), ctypes.c_float(d), int(nsample), int(neighbor_type),
                         lists.ctypes.data_as(_i), lens.ctypes.data_as(_i))
    return [lists[p, :lens[p]].copy() for p in range(m)]


def three_nn_local(xyz, centres, lists):
    """centres (M, G, 3), lists (per centre) -> (idx (M,G,3) int32, dist2 (M,G,3) float32), unfilled (+inf, -1)"""
    xyz = _f32(xyz)
    centres = np.ascontiguousarray(centres, np.float32)
    m, G = centres.shape[0], centres.shape[1]
    packed = np.zeros((max(m, 1), CAP), np.int32)
    lens = np.zeros(max(m, 1), np.int32)
    for p, lst in enumerate(lists):
        assert len(lst) <= CAP
        packed[p, :len(lst)] = lst
        lens[p] = len(lst)
    idx = np.zeros((m, G, 3), np.int32)
    dist2 = np.zeros((m, G, 3), np.float32)
    lib().vpo_three_nn(m, G, xyz.ctypes.data_as(_f), centres.ctypes.data_as(_f), packed.ctypes.data_as(_i),
                       lens.ctypes.data_as(_i), idx.ctypes.data_as(_i), dist2.ctypes.data_as(_f))
    return idx, dist2


def vector_pool(xyz, xyz_cnt, feats, new_xyz, new_cnt, grids, cpg, d, use_xyz, nsample, neighbor_type, pooling_type,
                max_triples=None):
    """vector_pool_wrapper on zeroed outputs -> (new_features (M, G*cpg), new_local_xyz (M, 3G), cnt (M, G),
    triples (T, 3), T); the triples in centre-then-index order, at most max_triples kept (default: all)"""
    xyz, new_xyz = _f32(xyz), _f32(new_xyz)
    feats = np.ascontiguousarray(feats, np.float32)
    nb, mb = np.ascontiguousarray(xyz_cnt, np.int32), np.ascontiguousarray(new_cnt, np.int32)
    m, (nx, ny, nz) = new_xyz.shape[0], grids
    G = nx * ny * nz
    cout = G * cpg
    def run(cap):
        nf = np.zeros((m, cout), np.float32)
        nl = np.zeros((m, 3 * G), np.float32)
        cnt = np.zeros((m, G), np.int32)
        tr = np.zeros((max(cap, 1), 3), np.int32)
        total = lib().vpo_pool(len(nb), m, xyz.ctypes.data_as(_f), nb.ctypes.data_as(_i), feats.ctypes.data_as(_f),
                               feats.shape[1], new_xyz.ctypes.data_as(_f), mb.ctypes.data_as(_i), nx, ny, nz, cout,
                               ctypes.c_float(d), int(use_xyz), int(nsample), int(neighbor_type), int(pooling_type),
                               nf.ctypes.data_as(_f), nl.ctypes.data_as(_f), cnt.ctypes.data_as(_i),
                               tr.ctypes.data_as(_i), ctypes.c_longlong(cap))
        return nf, nl, cnt, tr[:min(total, cap)], int(total)

    if max_triples is None:
        max_triples = run(0)[4]
    return run(int(max_triples))
