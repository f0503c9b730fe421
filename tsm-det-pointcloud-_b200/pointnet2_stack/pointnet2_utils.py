"""``BallQuery`` / ``QueryAndGroup`` / ``GroupingOperation`` / ``StackFarthestPointSampling`` /
``FarthestPointSampling`` / ``ThreeNN`` / ``ThreeInterpolate`` of
``/root/reference/pcdet/ops/pointnet2/pointnet2_stack/pointnet2_utils.py`` on the sm_100a kernels: same signatures,
argument checks and returns (the vector-pool ops of that file are not part of this package)."""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.autograd import Function

from . import pointnet2_stack_cuda as pointnet2


class BallQuery(Function):
    """ref :10-45"""

    @staticmethod
    def forward(ctx, radius: float, nsample: int, xyz: torch.Tensor, xyz_batch_cnt: torch.Tensor,
                new_xyz: torch.Tensor, new_xyz_batch_cnt):
        """xyz (N1+N2..., 3), xyz_batch_cnt (B), new_xyz (M1+M2..., 3), new_xyz_batch_cnt (B)
        -> (idx (M1+M2..., nsample) int32 frame-local rows, empty_ball_mask (M1+M2...) bool); rows of empty balls are 0"""
        assert new_xyz.is_contiguous()
        assert new_xyz_batch_cnt.is_contiguous()
        assert xyz.is_contiguous()
        assert xyz_batch_cnt.is_contiguous()

        B = xyz_batch_cnt.shape[0]
        M = new_xyz.shape[0]
        idx = torch.zeros((M, nsample), dtype=torch.int32, device=new_xyz.device)
        pointnet2.ball_query_wrapper(B, M, radius, nsample, new_xyz, new_xyz_batch_cnt, xyz, xyz_batch_cnt, idx)
        empty_ball_mask = idx[:, 0] == -1
        idx[empty_ball_mask] = 0
        ctx.mark_non_differentiable(idx)
        ctx.mark_non_differentiable(empty_ball_mask)
        return idx, empty_ball_mask

    @staticmethod
    def backward(ctx, a=None, b=None):
        return None, None, None, None, None, None


ball_query = BallQuery.apply


class GroupingOperation(Function):
    """ref :48-103"""

    @staticmethod
    def forward(ctx, features: torch.Tensor, features_batch_cnt: torch.Tensor, idx: torch.Tensor,
                idx_batch_cnt: torch.Tensor):
        """features (N1+N2..., C), features_batch_cnt (B), idx (M1+M2..., nsample) frame-local rows, idx_batch_cnt (B)
        -> (M1+M2..., C, nsample)"""
        assert features.is_contiguous()
        assert features_batch_cnt.is_contiguous()
        assert idx.is_contiguous()
        assert idx_batch_cnt.is_contiguous()
        assert features.shape[0] == features_batch_cnt.sum(), \
            'features: %s, features_batch_cnt: %s' % (str(features.shape), str(features_batch_cnt))
        assert idx.shape[0] == idx_batch_cnt.sum(), 'idx: %s, idx_batch_cnt: %s' % (str(idx.shape), str(idx_batch_cnt))
        M, nsample = idx.size()
        N, C = features.size()
        B = idx_batch_cnt.shape[0]
        output = torch.empty((M, C, nsample), dtype=torch.float32, device=features.device)
        pointnet2.group_points_wrapper(B, M, C, nsample, features, features_batch_cnt, idx, idx_batch_cnt, output)
        ctx.for_backwards = (B, N, idx, features_batch_cnt, idx_batch_cnt)
        return output

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        B, N, idx, features_batch_cnt, idx_batch_cnt = ctx.for_backwards
        M, C, nsample = grad_out.size()
        grad_features = torch.zeros((N, C), dtype=torch.float32, device=grad_out.device)
        pointnet2.group_points_grad_wrapper(B, M, C, N, nsample, grad_out.data.contiguous(), idx, idx_batch_cnt,
                                            features_batch_cnt, grad_features)
        return grad_features, None, None, None


grouping_operation = GroupingOperation.apply


class FarthestPointSampling(Function):
    """ref :158-184 -- the dense-batch sampler under its stack-module name"""

    @staticmethod
    def forward(ctx, xyz: torch.Tensor, npoint: int):
        assert xyz.is_contiguous()
        B, N, _ = xyz.size()
        output = torch.empty((B, npoint), dtype=torch.int32, device=xyz.device)
        temp = torch.full((B, N), 1e10, dtype=torch.float32, device=xyz.device)
        pointnet2.farthest_point_sampling_wrapper(B, N, npoint, xyz, temp, output)
        return output

    @staticmethod
    def backward(xyz, a=None):
        return None, None


farthest_point_sample = furthest_point_sample = FarthestPointSampling.apply


class StackFarthestPointSampling(Function):
    """ref :187-219"""

    @staticmethod
    def forward(ctx, xyz, xyz_batch_cnt, npoint):
        """xyz (N1+N2..., 3), xyz_batch_cnt [N1, N2, ...], npoint int | list | tensor -> (sum npoint) int32 GLOBAL rows"""
        assert xyz.is_contiguous() and xyz.shape[1] == 3
        batch_size = xyz_batch_cnt.__len__()
        if not isinstance(npoint, torch.Tensor):
            if not isinstance(npoint, list):
                npoint = [npoint for i in range(batch_size)]
            npoint = torch.tensor(npoint, device=xyz.device).int()
        N, _ = xyz.size()
        temp = torch.full((N,), 1e10, dtype=torch.float32, device=xyz.device)
        output = torch.empty((int(npoint.sum().item()),), dtype=torch.int32, device=xyz.device)
        pointnet2.stack_farthest_point_sampling_wrapper(xyz, temp, xyz_batch_cnt.int().contiguous(), output,
                                                        npoint.contiguous())
        return output

    @staticmethod
    def backward(xyz, a=None):
        return None, None


stack_farthest_point_sample = StackFarthestPointSampling.apply


class QueryAndGroup(nn.Module):
    """ref :106-155"""

    def __init__(self, radius: float, nsample: int, use_xyz: bool = True):
        super().__init__()
        self.radius, self.nsample, self.use_xyz = radius, nsample, use_xyz

    def forward(self, xyz: torch.Tensor, xyz_batch_cnt: torch.Tensor, new_xyz: torch.Tensor,
                new_xyz_batch_cnt: torch.Tensor, features: torch.Tensor = None):
        """xyz (N1+N2..., 3), xyz_batch_cnt (B), new_xyz (M1+M2..., 3), new_xyz_batch_cnt (B), features (N1+N2..., C)
        -> (new_features (M1+M2..., 3+C, nsample), idx (M1+M2..., nsample))"""
        assert xyz.shape[0] == xyz_batch_cnt.sum(), 'xyz: %s, xyz_batch_cnt: %s' % (str(xyz.shape), str(new_xyz_batch_cnt))
        assert new_xyz.shape[0] == new_xyz_batch_cnt.sum(), \
            'new_xyz: %s, new_xyz_batch_cnt: %s' % (str(new_xyz.shape), str(new_xyz_batch_cnt))

        idx, empty_ball_mask = ball_query(self.radius, self.nsample, xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt)
        grouped_xyz = grouping_operation(xyz, xyz_batch_cnt, idx, new_xyz_batch_cnt)  # (M1+M2..., 3, nsample)
        grouped_xyz -= new_xyz.unsqueeze(-1)
        grouped_xyz[empty_ball_mask] = 0

        if features is not None:
            grouped_features = grouping_operation(features, xyz_batch_cnt, idx, new_xyz_batch_cnt)  # (M1+M2..., C, nsample)
            grouped_features[empty_ball_mask] = 0
            if self.use_xyz:
                new_features = torch.cat([grouped_xyz, grouped_features], dim=1)  # (M1+M2..., 3+C, nsample)
            else:
                new_features = grouped_features
        else:
            assert self.use_xyz, "Cannot have not features and not use xyz as a feature!"
            new_features = grouped_xyz
        return new_features, idx


class ThreeNN(Function):
    """ref ThreeNN (stack)"""

    @staticmethod
    def forward(ctx, unknown, unknown_batch_cnt, known, known_batch_cnt):
        """unknown (N1+N2..., 3), unknown_batch_cnt (B), known (M1+M2..., 3), known_batch_cnt (B)
        -> (dist (N1+N2..., 3) l2 distances to the three nearest known points of the same frame,
            idx (N1+N2..., 3) int32 GLOBAL known rows)"""
        assert unknown.shape.__len__() == 2 and unknown.shape[1] == 3
        assert known.shape.__len__() == 2 and known.shape[1] == 3
        assert unknown_batch_cnt.__len__() == known_batch_cnt.__len__()

        dist2 = unknown.new_zeros(unknown.shape)
        idx = unknown_batch_cnt.new_zeros(unknown.shape).int()
        pointnet2.three_nn_wrapper(unknown.contiguous(), unknown_batch_cnt.contiguous(), known.contiguous(),
                                   known_batch_cnt.contiguous(), dist2, idx)
        return torch.sqrt(dist2), idx

    @staticmethod
    def backward(ctx, a=None, b=None):
        return None, None


three_nn = ThreeNN.apply


class ThreeInterpolate(Function):
    """ref ThreeInterpolate (stack)"""

    @staticmethod
    def forward(ctx, features: torch.Tensor, idx: torch.Tensor, weight: torch.Tensor):
        """features (M1+M2..., C), idx / weight (N1+N2..., 3) -> (N1+N2..., C)"""
        assert idx.shape[0] == weight.shape[0] and idx.shape[1] == weight.shape[1] == 3

        ctx.three_interpolate_for_backward = (idx, weight, features.shape[0])
        output = features.new_zeros((idx.shape[0], features.shape[1]))
        pointnet2.three_interpolate_wrapper(features.contiguous(), idx.contiguous(), weight.contiguous(), output)
        return output

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        """grad_out (N1+N2..., C) -> grad_features (M1+M2..., C)"""
        idx, weight, M = ctx.three_interpolate_for_backward
        grad_features = grad_out.new_zeros((M, grad_out.shape[1]))
        pointnet2.three_interpolate_grad_wrapper(grad_out.contiguous(), idx.contiguous(), weight.contiguous(),
                                                 grad_features)
        return grad_features, None, None


three_interpolate = ThreeInterpolate.apply
