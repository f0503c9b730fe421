"""``BallQuery`` / ``QueryAndGroup`` / ``GroupingOperation`` / ``StackFarthestPointSampling`` /
``FarthestPointSampling`` / ``ThreeNN`` / ``ThreeInterpolate`` and the vector-pool ops
(``ThreeNNForVectorPoolByTwoStep``, ``VectorPoolWithVoxelQuery``, ``VectorPoolLocalInterpolateModule``) of
``/root/reference/pcdet/ops/pointnet2/pointnet2_stack/pointnet2_utils.py`` on the sm_100a kernels: same signatures,
argument checks and returns."""
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


class ThreeNNForVectorPoolByTwoStep(Function):
    """ref ThreeNNForVectorPoolByTwoStep: the local neighbour lists (distance max_neighbour_distance *
    neighbor_distance_multiplier, retried with a larger buffer until they fit), then the three nearest list entries of
    every sub-voxel centre."""

    @staticmethod
    def forward(ctx, support_xyz, xyz_batch_cnt, new_xyz, new_xyz_grid_centers, new_xyz_batch_cnt,
                max_neighbour_distance, nsample, neighbor_type, avg_length_of_neighbor_idxs, num_total_grids,
                neighbor_distance_multiplier):
        """support_xyz (N1+N2..., 3), xyz_batch_cnt (B), new_xyz (M1+M2..., 3), new_xyz_grid_centers (M1+M2..., G, 3),
        new_xyz_batch_cnt (B); nsample -1 = all hits; neighbor_type 1 = ball, else cube
        -> (dist (M1+M2..., G, 3), idx (M1+M2..., G, 3) int32 GLOBAL rows, -1 where unfilled, avg_length tensor)"""
        num_new_xyz = new_xyz.shape[0]
        new_xyz_grid_dist2 = new_xyz_grid_centers.new_zeros(new_xyz_grid_centers.shape)
        new_xyz_grid_idxs = new_xyz_grid_centers.new_zeros(new_xyz_grid_centers.shape).int().fill_(-1)

        while True:
            num_max_sum_points = avg_length_of_neighbor_idxs * num_new_xyz
            stack_neighbor_idxs = new_xyz_grid_idxs.new_zeros(num_max_sum_points)
            start_len = new_xyz_grid_idxs.new_zeros(num_new_xyz, 2).int()
            cumsum = new_xyz_grid_idxs.new_zeros(1)

            pointnet2.query_stacked_local_neighbor_idxs_wrapper_stack(
                support_xyz.contiguous(), xyz_batch_cnt.contiguous(), new_xyz.contiguous(),
                new_xyz_batch_cnt.contiguous(), stack_neighbor_idxs.contiguous(), start_len.contiguous(), cumsum,
                avg_length_of_neighbor_idxs, max_neighbour_distance * neighbor_distance_multiplier, nsample,
                neighbor_type)
            total = cumsum[0].item()
            avg_length_of_neighbor_idxs = total // num_new_xyz + int(total % num_new_xyz > 0)
            if total <= num_max_sum_points:
                break

        stack_neighbor_idxs = stack_neighbor_idxs[:total]
        pointnet2.query_three_nn_by_stacked_local_idxs_wrapper_stack(
            support_xyz, new_xyz, new_xyz_grid_centers, new_xyz_grid_idxs, new_xyz_grid_dist2, stack_neighbor_idxs,
            start_len, num_new_xyz, num_total_grids)
        return torch.sqrt(new_xyz_grid_dist2), new_xyz_grid_idxs, torch.tensor(avg_length_of_neighbor_idxs)

    @staticmethod
    def backward(ctx, a=None, b=None, c=None):
        return (None,) * 11


three_nn_for_vector_pool_by_two_step = ThreeNNForVectorPoolByTwoStep.apply


class VectorPoolWithVoxelQuery(Function):
    """ref VectorPoolWithVoxelQuery: per centre, the hits of its ball / cube pooled into G = nx*ny*nz sub-voxels
    (pooling_type 0: average, 1: the first hit of each sub-voxel), retried with a larger triple buffer until it fits."""

    @staticmethod
    def forward(ctx, support_xyz: torch.Tensor, xyz_batch_cnt: torch.Tensor, support_features: torch.Tensor,
                new_xyz: torch.Tensor, new_xyz_batch_cnt: torch.Tensor, num_grid_x, num_grid_y, num_grid_z,
                max_neighbour_distance, num_c_out_each_grid, use_xyz, num_mean_points_per_grid=100, nsample=-1,
                neighbor_type=0, pooling_type=0):
        """support_xyz (N1+N2..., 3), xyz_batch_cnt (B), support_features (N1+N2..., C), new_xyz (M1+M2..., 3),
        new_xyz_batch_cnt (B) -> (new_features (M1+M2..., G*num_c_out_each_grid), new_local_xyz (M1+M2..., 3G),
        num_mean_points_per_grid (1) int, point_cnt_of_grid (M1+M2..., G))"""
        assert support_xyz.is_contiguous()
        assert support_features.is_contiguous()
        assert xyz_batch_cnt.is_contiguous()
        assert new_xyz.is_contiguous()
        assert new_xyz_batch_cnt.is_contiguous()
        num_total_grids = num_grid_x * num_grid_y * num_grid_z
        num_c_out = num_c_out_each_grid * num_total_grids
        N, num_c_in = support_features.shape
        M = new_xyz.shape[0]

        assert num_c_in % num_c_out_each_grid == 0, \
            f'the input channels ({num_c_in}) should be an integral multiple of num_c_out_each_grid({num_c_out_each_grid})'

        while True:
            new_features = support_features.new_zeros((M, num_c_out))
            new_local_xyz = support_features.new_zeros((M, 3 * num_total_grids))
            point_cnt_of_grid = xyz_batch_cnt.new_zeros((M, num_total_grids))

            num_max_sum_points = num_mean_points_per_grid * M
            grouped_idxs = xyz_batch_cnt.new_zeros((num_max_sum_points, 3))

            num_cum_sum = pointnet2.vector_pool_wrapper(
                support_xyz, xyz_batch_cnt, support_features, new_xyz, new_xyz_batch_cnt, new_features, new_local_xyz,
                point_cnt_of_grid, grouped_idxs, num_grid_x, num_grid_y, num_grid_z, max_neighbour_distance, use_xyz,
                num_max_sum_points, nsample, neighbor_type, pooling_type)
            num_mean_points_per_grid = num_cum_sum // M + int(num_cum_sum % M > 0)
            if num_cum_sum <= num_max_sum_points:
                break

        grouped_idxs = grouped_idxs[:num_cum_sum]

        normalizer = torch.clamp_min(point_cnt_of_grid[:, :, None].float(), min=1e-6)
        new_features = (new_features.view(-1, num_total_grids, num_c_out_each_grid) / normalizer).view(-1, num_c_out)

        if use_xyz:
            new_local_xyz = (new_local_xyz.view(-1, num_total_grids, 3) / normalizer).view(-1, num_total_grids * 3)

        num_mean_points_per_grid = torch.Tensor([num_mean_points_per_grid]).int()
        nsample = torch.Tensor([nsample]).int()
        ctx.vector_pool_for_backward = (point_cnt_of_grid, grouped_idxs, N, num_c_in)
        ctx.mark_non_differentiable(new_local_xyz, num_mean_points_per_grid, nsample, point_cnt_of_grid)
        return new_features, new_local_xyz, num_mean_points_per_grid, point_cnt_of_grid

    @staticmethod
    def backward(ctx, grad_new_features: torch.Tensor, grad_local_xyz: torch.Tensor, grad_num_cum_sum,
                 grad_point_cnt_of_grid):
        """grad_new_features (M1+M2..., G*num_c_out_each_grid) -> grad_support_features (N1+N2..., C)"""
        point_cnt_of_grid, grouped_idxs, N, num_c_in = ctx.vector_pool_for_backward
        grad_support_features = grad_new_features.new_zeros((N, num_c_in))

        if grouped_idxs.shape[0] > 0:
            pointnet2.vector_pool_grad_wrapper(grad_new_features.contiguous(), point_cnt_of_grid, grouped_idxs,
                                               grad_support_features)

        return None, None, grad_support_features, None, None, None, None, None, None, None, None, None, None, None, None


vector_pool_with_voxel_query_op = VectorPoolWithVoxelQuery.apply


def local_interp_weights(dist: torch.Tensor) -> torch.Tensor:
    """inverse-distance weights of the three neighbours of each sub-voxel (ref VectorPoolLocalInterpolateModule.forward):
    a (+inf) slot gets weight 0, a sub-voxel without neighbours all-zero weights"""
    dist_recip = 1.0 / (dist + 1e-8)
    norm = torch.sum(dist_recip, dim=-1, keepdim=True)
    return dist_recip / torch.clamp_min(norm, min=1e-8)


class VectorPoolLocalInterpolateModule(nn.Module):
    """ref VectorPoolLocalInterpolateModule: the features at every sub-voxel centre, interpolated from its three nearest
    neighbours among the centre's local neighbours, with their 9 local offsets (``use_xyz``)."""

    def __init__(self, mlp, num_voxels, max_neighbour_distance, nsample, neighbor_type, use_xyz=True,
                 neighbour_distance_multiplier=1.0, xyz_encoding_type='concat'):
        """num_voxels [nx, ny, nz]; neighbor_type 1 = ball, else cube; nsample -1 = all neighbours, > 0 = the first
        nsample; mlp (optional): [C, ...], 9 channels are added for the offsets"""
        super().__init__()
        self.num_voxels = num_voxels
        self.num_total_grids = self.num_voxels[0] * self.num_voxels[1] * self.num_voxels[2]
        self.max_neighbour_distance = max_neighbour_distance
        self.neighbor_distance_multiplier = neighbour_distance_multiplier
        self.nsample = nsample
        self.neighbor_type = neighbor_type
        self.use_xyz = use_xyz
        self.xyz_encoding_type = xyz_encoding_type

        if mlp is not None:
            if self.use_xyz:
                mlp[0] += 9 if self.xyz_encoding_type == 'concat' else 0
            shared_mlps = []
            for k in range(len(mlp) - 1):
                shared_mlps.extend([
                    nn.Conv2d(mlp[k], mlp[k + 1], kernel_size=1, bias=False),
                    nn.BatchNorm2d(mlp[k + 1]),
                    nn.ReLU()
                ])
            self.mlp = nn.Sequential(*shared_mlps)
        else:
            self.mlp = None

        self.num_avg_length_of_neighbor_idxs = 1000

    def forward(self, support_xyz, support_features, xyz_batch_cnt, new_xyz, new_xyz_grid_centers, new_xyz_batch_cnt):
        """support_xyz (N1+N2..., 3), support_features (N1+N2..., C), xyz_batch_cnt (B), new_xyz (M1+M2..., 3),
        new_xyz_grid_centers (M1+M2..., G, 3), new_xyz_batch_cnt (B) -> ((M1+M2...)*G, C(+9) or the mlp's width)"""
        with torch.no_grad():
            dist, idx, num_avg_length_of_neighbor_idxs = three_nn_for_vector_pool_by_two_step(
                support_xyz, xyz_batch_cnt, new_xyz, new_xyz_grid_centers, new_xyz_batch_cnt,
                self.max_neighbour_distance, self.nsample, self.neighbor_type, self.num_avg_length_of_neighbor_idxs,
                self.num_total_grids, self.neighbor_distance_multiplier)
        self.num_avg_length_of_neighbor_idxs = max(self.num_avg_length_of_neighbor_idxs,
                                                   num_avg_length_of_neighbor_idxs.item())

        weight = local_interp_weights(dist)

        empty_mask = (idx.view(-1, 3)[:, 0] == -1)
        idx.view(-1, 3)[empty_mask] = 0

        interpolated_feats = three_interpolate(support_features, idx.view(-1, 3), weight.view(-1, 3))
        interpolated_feats = interpolated_feats.view(idx.shape[0], idx.shape[1], -1)  # (M1 + M2 ..., G, C)
        if self.use_xyz:
            near_known_xyz = support_xyz[idx.view(-1, 3).long()].view(-1, 3, 3)  # ((M1 + M2 ...) * G, 3, 3)
            local_xyz = (new_xyz_grid_centers.view(-1, 1, 3) - near_known_xyz).view(-1, idx.shape[1], 9)
            if self.xyz_encoding_type == 'concat':
                interpolated_feats = torch.cat((interpolated_feats, local_xyz), dim=-1)  # (M1 + M2 ..., G, C + 9)
            else:
                raise NotImplementedError

        new_features = interpolated_feats.view(-1, interpolated_feats.shape[-1])  # ((M1 + M2 ...) * G, C)
        new_features[empty_mask, :] = 0
        if self.mlp is not None:
            new_features = new_features.permute(1, 0)[None, :, :, None]  # (1, C, (M1 + M2 ...) * G, 1)
            new_features = self.mlp(new_features)
            new_features = new_features.squeeze(dim=0).squeeze(dim=-1).permute(1, 0)
        return new_features
