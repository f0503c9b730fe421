"""Native surface of the reference's ``roiaware_pool3d_cuda`` pybind module, every function it exports, re-hosted on the
C ABI: same names / positional arguments / returns (1) as ``/root/reference/pcdet/ops/roiaware_pool3d/src/
roiaware_pool3d.cpp``."""
from __future__ import annotations

import torch

from .._lib import call, ptr, stream_ptr


def _chk(dtypes, *tensors, cuda=True):
    for t, dt in zip(tensors, dtypes):
        if t.is_cuda != cuda:
            raise ValueError("must be a CUDA tensor" if cuda else "must be a CPU tensor")
        if not t.is_contiguous():
            raise ValueError("must be a contiguous tensor")
        if t.dtype != dt:
            raise ValueError(f"must be a {dt} tensor, got {t.dtype}")
    if cuda and len({t.device for t in tensors}) > 1:
        raise ValueError("all tensors must be on the same device")


_F, _I = torch.float32, torch.int32


def forward(rois, pts, pts_feature, argmax, pts_idx_of_voxels, pooled_features, pool_method):
    """rois (R,7), pts (P,3), pts_feature (P,C) -> argmax / pooled_features (R,X,Y,Z,C), pts_idx_of_voxels (R,X,Y,Z,L);
    pool_method 0 max, 1 avg.  X, Y, Z from argmax's shape, L from pts_idx_of_voxels'."""
    _chk((_F, _F, _F, _I, _I, _F), rois, pts, pts_feature, argmax, pts_idx_of_voxels, pooled_features)
    if argmax.dim() != 5 or pts_idx_of_voxels.dim() != 5 or pooled_features.shape != argmax.shape:
        raise ValueError("argmax / pooled_features must be (R,X,Y,Z,C) and pts_idx_of_voxels (R,X,Y,Z,L)")
    _, x, y, z, c = argmax.shape
    call("tsmdet_roiaware_pool3d", rois.shape[0], pts.shape[0], pts_feature.shape[1], x, y, z,
         pts_idx_of_voxels.shape[4], ptr(rois), ptr(pts), ptr(pts_feature), ptr(argmax), ptr(pts_idx_of_voxels),
         ptr(pooled_features), int(pool_method), stream_ptr(rois.device))
    return 1


def backward(pts_idx_of_voxels, argmax, grad_out, grad_in, pool_method):
    """grad_in (P,C) (zeroed by the caller) += the scatter of grad_out (R,X,Y,Z,C)"""
    _chk((_I, _I, _F, _F), pts_idx_of_voxels, argmax, grad_out, grad_in)
    if pts_idx_of_voxels.dim() != 5 or grad_out.dim() != 5:
        raise ValueError("pts_idx_of_voxels must be (R,X,Y,Z,L) and grad_out (R,X,Y,Z,C)")
    r, x, y, z, L = pts_idx_of_voxels.shape
    call("tsmdet_roiaware_pool3d_grad", r, grad_in.shape[0], grad_out.shape[4], x, y, z, L, ptr(pts_idx_of_voxels),
         ptr(argmax), ptr(grad_out), ptr(grad_in), int(pool_method), stream_ptr(grad_out.device))
    return 1


def points_in_boxes_gpu(boxes_tensor, pts_tensor, box_idx_of_points_tensor):
    """boxes (B,T,7), pts (B,N,3) -> box_idx_of_points (B,N) int32: the first box holding the point, the pre-fill
    otherwise"""
    _chk((_F, _F, _I), boxes_tensor, pts_tensor, box_idx_of_points_tensor)
    call("tsmdet_points_in_boxes", boxes_tensor.shape[0], boxes_tensor.shape[1], pts_tensor.shape[1],
         ptr(boxes_tensor), ptr(pts_tensor), ptr(box_idx_of_points_tensor), stream_ptr(boxes_tensor.device))
    return 1


def points_in_boxes_cpu(boxes_tensor, pts_tensor, pts_indices_tensor):
    """host tensors: boxes (M,7), pts (N,3) -> pts_indices (M,N) int32, 0 / 1 per pair"""
    _chk((_F, _F, _I), boxes_tensor, pts_tensor, pts_indices_tensor, cuda=False)
    call("tsmdet_points_in_boxes_cpu", boxes_tensor.shape[0], pts_tensor.shape[0], ptr(boxes_tensor), ptr(pts_tensor),
         ptr(pts_indices_tensor))
    return 1


__all__ = ["forward", "backward", "points_in_boxes_gpu", "points_in_boxes_cpu"]
