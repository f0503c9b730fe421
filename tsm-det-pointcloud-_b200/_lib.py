"""ctypes binding of ``libtsmdet_b200.so`` (see ``include/tsmdet_b200.h``).

No fallback of any kind: if the shared library is missing the import fails with
instructions to build it, and every non-zero status from the C ABI becomes a Python
exception (the reference would ``exit(-1)`` instead, e.g. sampling_gpu.cu:255-259).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_longlong, c_void_p

# more hardware work queues than the CUDA default of 8 (see tsmdet_b200/__init__.py: in-kernel waits of the peer gather
# must not share a queue with other pipeline lanes); only effective before the process creates its CUDA context
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_HERE = os.path.dirname(os.path.abspath(__file__))
# TSMDET_LIB: load another build of the same C ABI (instrumented builds made by scripts/; never a fallback)
LIB_PATH = os.environ.get("TSMDET_LIB") or os.path.join(_HERE, "libtsmdet_b200.so")


class TsmdetError(RuntimeError):
    def __init__(self, code: int, where: str):
        self.code = code
        msg = _lib.tsmdet_error_string(code).decode() if _lib is not None else str(code)
        super().__init__(f"{where}: {msg} (status {code})")


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            f"`python {os.path.join(_HERE, 'build.py')}` (needs nvcc; cross-compiles sm_100a without a GPU). "
            "tsmdet_b200 has no CPU / eager fallback."
        )
    return ctypes.CDLL(LIB_PATH)


_lib = None
_lib = _load()

_f = POINTER(c_float)
_i = POINTER(c_int)
_ll = POINTER(c_longlong)
_pp = POINTER(c_void_p)

# name -> argtypes (restype is always int unless listed in _RESTYPES)
SIGNATURES = {
    "tsmdet_read_status": [],
    "tsmdet_farthest_point_sampling": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_fps_chain": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                         c_int, c_void_p],
    "tsmdet_furthest_point_sampling_weights": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_furthest_point_sampling_matrix": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_furthest_point_sampling_with_weighted_dist": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                                          c_void_p],
    "tsmdet_fps_plan": [c_int, c_int, _i, _i, _i, _i],
    "tsmdet_fps_configure": [c_int],
    "tsmdet_gather_points": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_gather_points_grad": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_gather_xyz": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stage_points": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_ball_query": [c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_ball_query_dilated": [c_int, c_int, c_int, c_float, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p],
    "tsmdet_group_points": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_group_points_grad": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_group_concat": [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                            c_void_p, c_void_p],
    "tsmdet_three_nn": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_three_interpolate": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_three_interpolate_grad": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_sa_mlp_maxpool": [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_int, _i, _pp, _pp, c_void_p, c_int, c_int, c_int, c_void_p],
    "tsmdet_pointwise_mlp": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, _i, _pp, _pp, c_void_p, c_int, c_int,
                             c_int, c_void_p],
    "tsmdet_mlp_pack": [c_int, c_int, c_int, c_int, c_int, c_int, _i, _pp, _pp, c_void_p, _ll, c_void_p],
    "tsmdet_sa_mlp_maxpool_packed": [c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int, _i, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    "tsmdet_pointwise_mlp_packed": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, _i, c_void_p, c_void_p, c_int,
                                    c_int, c_void_p],
    "tsmdet_mlp_pack_p": [c_int, c_int, c_int, c_int, c_int, c_int, c_int, _i, _pp, _pp, c_void_p, _ll, c_void_p],
    "tsmdet_sa_mlp_maxpool_packed_p": [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_int, _i, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    "tsmdet_pointwise_mlp_packed_p": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, _i, c_void_p, c_void_p,
                                      c_int, c_int, c_void_p],
    "tsmdet_voxel_centroids": [c_int, c_int, c_int, c_void_p, c_void_p, c_float, c_float, c_float, c_float, c_float, c_float,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_centroid_per_voxel": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_voxel2pinds": [c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_voxel_query": [c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_voxel_query_dilated": [c_int, c_int, c_int, c_int, c_int, c_float, c_float, c_int, c_int, c_int, c_int, c_int,
                                   c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_group_points": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_group_points_grad": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p],
    "tsmdet_stack_farthest_point_sampling": [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_ball_query": [c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_int, c_void_p],
    "tsmdet_stack_feature_rows": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_three_nn": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_three_interpolate": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p],
    "tsmdet_stack_three_interpolate_grad": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_local_neighbor_idxs": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_int, c_float, c_int, c_int, c_void_p],
    "tsmdet_stack_three_nn_local": [c_int, c_int, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p],
    "tsmdet_stack_vector_three_nn": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float,
                                     c_int, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_vector_pool": [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_longlong,
                                 c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_stack_vector_pool_grad": [c_int, c_int, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p],
    "tsmdet_stack_vector_interp_planes": [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p],
    "tsmdet_points_in_boxes": [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "tsmdet_points_in_boxes_cpu": [c_int, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_roiaware_pool3d": [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_int, c_void_p],
    "tsmdet_roiaware_pool3d_grad": [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_int, c_void_p],
    "tsmdet_boxes_overlap_bev": [c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_boxes_iou_bev": [c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    "tsmdet_boxes_iou_bev_cpu": [c_int, c_void_p, c_int, c_void_p, c_void_p],
    "tsmdet_nms_gpu": [c_int, c_void_p, c_float, c_void_p, _i, c_void_p],
    "tsmdet_nms_normal_gpu": [c_int, c_void_p, c_float, c_void_p, _i, c_void_p],
    "tsmdet_nms_batch": [c_int, c_int, c_void_p, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p],
    "tsmdet_nms_normal_batch": [c_int, c_int, c_void_p, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p],
    "tsmdet_peer_put": [c_void_p, c_longlong, c_int, _pp, _pp, _pp, c_void_p, c_void_p, c_longlong, c_int, c_longlong,
                        c_longlong, c_void_p],
    "tsmdet_peer_wait": [c_void_p, c_int, c_longlong, c_int, c_longlong, c_void_p],
    "tsmdet_reload_options": [],
    "tsmdet_scratch_stats": [_ll, _ll],
    "tsmdet_scratch_trim": [],
    "tsmdet_enable_peer_access": [c_int],
}
_RESTYPES = {"tsmdet_version": c_char_p, "tsmdet_error_string": c_char_p}

for _name, _args in SIGNATURES.items():
    _fn = getattr(_lib, _name)  # AttributeError here = header and library out of sync
    _fn.argtypes = _args
    _fn.restype = c_int
_lib.tsmdet_version.restype = c_char_p
_lib.tsmdet_version.argtypes = []
_lib.tsmdet_error_string.restype = c_char_p
_lib.tsmdet_error_string.argtypes = [c_int]

EXPORTS = sorted(list(SIGNATURES) + list(_RESTYPES))


def lib() -> ctypes.CDLL:
    return _lib


def version() -> str:
    return _lib.tsmdet_version().decode()


def check(status: int, where: str) -> None:
    if status != 0:
        raise TsmdetError(status, where)


# kernels launched per C-ABI call (for bench.py's gpu_launches claim)
KERNELS_PER_CALL = {
    "tsmdet_nms_batch": 6, "tsmdet_nms_normal_batch": 3, "tsmdet_nms_gpu": 6, "tsmdet_nms_normal_gpu": 3,
    "tsmdet_boxes_overlap_bev": 3, "tsmdet_boxes_iou_bev": 3, "tsmdet_boxes_iou_bev_cpu": 0,
    "tsmdet_fps_plan": 0, "tsmdet_fps_configure": 0, "tsmdet_enable_peer_access": 0, "tsmdet_read_status": 0,
    "tsmdet_reload_options": 0, "tsmdet_scratch_stats": 0, "tsmdet_scratch_trim": 0, "tsmdet_ball_query": 3, "tsmdet_ball_query_dilated": 3, "tsmdet_sa_mlp_maxpool": 3, "tsmdet_pointwise_mlp": 2, "tsmdet_sa_mlp_maxpool_packed": 2,
    "tsmdet_pointwise_mlp_packed": 1, "tsmdet_mlp_pack": 1, "tsmdet_sa_mlp_maxpool_packed_p": 2, "tsmdet_pointwise_mlp_packed_p": 1,
    "tsmdet_mlp_pack_p": 1, "tsmdet_stack_ball_query": 4, "tsmdet_stack_three_nn": 4, "tsmdet_stack_local_neighbor_idxs": 3,
    "tsmdet_stack_vector_three_nn": 3, "tsmdet_stack_vector_pool": 3, "tsmdet_voxel_centroids": 2, "tsmdet_centroid_per_voxel": 2, "tsmdet_voxel2pinds": 2,
    "tsmdet_points_in_boxes_cpu": 0, "tsmdet_roiaware_pool3d": 2,
}
launch_count = 0


def read_status() -> int:
    """Reads and clears the per-device watchdog word (0 = clean); works after a kernel fault (host-mapped word)."""
    return int(_lib.tsmdet_read_status())


def reload_options() -> None:
    """Re-read the TSMDET_* tuning knobs from os.environ (the library reads them once, at first use)."""
    check(_lib.tsmdet_reload_options(), "tsmdet_reload_options")


def call(name: str, *args) -> None:
    """Invoke a C-ABI function and raise on a non-zero status."""
    global launch_count
    check(getattr(_lib, name)(*args), name)
    launch_count += KERNELS_PER_CALL.get(name, 1)


# --------------------------------------------------------------------------- torch glue
def ptr(t) -> c_void_p:
    """Raw device (or host) pointer of a tensor, None -> NULL."""
    if t is None:
        return c_void_p(0)
    return c_void_p(t.data_ptr())


def stream_ptr(device=None) -> c_void_p:
    import torch

    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ValueError("tsmdet_b200 ops need CUDA tensors (there is no CPU fallback)")
