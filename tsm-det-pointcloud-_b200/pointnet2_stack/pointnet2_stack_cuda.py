"""Native surface of the reference's ``pointnet2_stack_cuda`` pybind module, every function it exports, re-hosted on
the C ABI: same names / positional arguments / returns as
``/root/reference/pcdet/ops/pointnet2/pointnet2_stack/src/pointnet2_api.cpp``."""
from __future__ import annotations

from .._lib import call, ptr, stream_ptr
from ..pointnet2_batch_cuda import farthest_point_sampling_wrapper  # noqa: F401  (:16, the dense-batch sampler)


def _chk(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise ValueError("must be a CUDA tensor")
        if not t.is_contiguous():
            raise ValueError("must be a contiguous tensor")


def ball_query_wrapper(B, M, radius, nsample, new_xyz, new_xyz_batch_cnt, xyz, xyz_batch_cnt, idx):
    """ref ball_query.cpp:25-45: new_xyz (M,3), xyz (N,3) stacked, counts (B) int32, idx (M,nsample) int32 zeroed by
    the caller -> frame-local rows, first hit repeated past the hits, idx[p,0] = -1 for a centre without hits"""
    _chk(new_xyz, new_xyz_batch_cnt, xyz, xyz_batch_cnt, idx)
    call("tsmdet_stack_ball_query", B, M, xyz.shape[0], float(radius), nsample, ptr(new_xyz), ptr(new_xyz_batch_cnt),
         ptr(xyz), ptr(xyz_batch_cnt), ptr(idx), None, 0, stream_ptr(xyz.device))
    return 1


def voxel_query_wrapper(M, R1, R2, R3, nsample, radius, z_range, y_range, x_range, new_xyz, xyz, new_coords,
                        point_indices, idx, cnt_unique):
    """ref voxel_query.cpp:27-46"""
    _chk(new_coords, point_indices, new_xyz, xyz)
    call("tsmdet_voxel_query", M, R1, R2, R3, nsample, float(radius), int(z_range), int(y_range), int(x_range), ptr(new_xyz),
         ptr(xyz), ptr(new_coords), ptr(point_indices), ptr(idx), ptr(cnt_unique), stream_ptr(xyz.device))
    return 1


def voxel_query_dilated_wrapper(M, R1, R2, R3, nsample, former_radius, radius, z_range, y_range, x_range, z_stride,
                                y_stride, x_stride, new_xyz, xyz, new_coords, point_indices, idx, cnt_unique, idx_cnt):
    """ref voxel_query.cpp:48-75"""
    _chk(new_coords, point_indices, new_xyz, xyz)
    call("tsmdet_voxel_query_dilated", M, R1, R2, R3, nsample, float(former_radius), float(radius), int(z_range),
         int(y_range), int(x_range), int(z_stride), int(y_stride), int(x_stride), ptr(new_xyz), ptr(xyz), ptr(new_coords),
         ptr(point_indices), ptr(idx), ptr(cnt_unique), ptr(idx_cnt), stream_ptr(xyz.device))
    return 1


def group_points_wrapper(B, M, C, nsample, features, features_batch_cnt, idx, idx_batch_cnt, out):
    """ref group_points.cpp (stack): features (N,C), idx (M,nsample) -> out (M,C,nsample)"""
    _chk(features, features_batch_cnt, idx, idx_batch_cnt, out)
    call("tsmdet_stack_group_points", B, M, C, nsample, ptr(features), ptr(features_batch_cnt), ptr(idx),
         ptr(idx_batch_cnt), ptr(out), stream_ptr(features.device))
    return 1


def group_points_grad_wrapper(B, M, C, N, nsample, grad_out, idx, idx_batch_cnt, features_batch_cnt, grad_features):
    _chk(grad_out, idx, idx_batch_cnt, features_batch_cnt, grad_features)
    call("tsmdet_stack_group_points_grad", B, M, C, N, nsample, ptr(grad_out), ptr(idx), ptr(idx_batch_cnt),
         ptr(features_batch_cnt), ptr(grad_features), stream_ptr(grad_out.device))
    return 1


def stack_farthest_point_sampling_wrapper(points, temp, xyz_batch_cnt, idx, num_sampled_points):
    """ref sampling.cpp (stack): points (N,3), temp (N) filled with 1e10, counts on the device -> idx (sum M)"""
    _chk(points, temp, xyz_batch_cnt, idx, num_sampled_points)
    call("tsmdet_stack_farthest_point_sampling", points.shape[0], xyz_batch_cnt.shape[0], ptr(points), ptr(temp),
         ptr(xyz_batch_cnt), ptr(idx), ptr(num_sampled_points), stream_ptr(points.device))
    return 1


def three_nn_wrapper(unknown, unknown_batch_cnt, known, known_batch_cnt, dist2, idx):
    """ref interpolate.cpp (stack): unknown (N,3), known (M,3) stacked, counts (B) int32 -> dist2 (N,3) squared
    distances, idx (N,3) int32 GLOBAL known rows; slots a frame with < 3 known points cannot fill are (inf, its start)"""
    _chk(unknown, unknown_batch_cnt, known, known_batch_cnt, dist2, idx)
    call("tsmdet_stack_three_nn", unknown_batch_cnt.shape[0], unknown.shape[0], known.shape[0], ptr(unknown),
         ptr(unknown_batch_cnt), ptr(known), ptr(known_batch_cnt), ptr(dist2), ptr(idx), stream_ptr(unknown.device))


def three_interpolate_wrapper(features, idx, weight, out):
    """features (M,C), idx / weight (N,3) -> out (N,C); an index outside [0, M) reads 0 (the reference reads out of
    bounds there)"""
    _chk(features, idx, weight, out)
    call("tsmdet_stack_three_interpolate", idx.shape[0], features.shape[1], features.shape[0], ptr(features), ptr(idx),
         ptr(weight), ptr(out), 0, stream_ptr(features.device))


def three_interpolate_grad_wrapper(grad_out, idx, weight, grad_features):
    """grad_out (N,C) -> grad_features (M,C) += g * w, zeroed by the caller"""
    _chk(grad_out, idx, weight, grad_features)
    call("tsmdet_stack_three_interpolate_grad", idx.shape[0], grad_out.shape[1], grad_features.shape[0], ptr(grad_out),
         ptr(idx), ptr(weight), ptr(grad_features), stream_ptr(grad_out.device))


def query_stacked_local_neighbor_idxs_wrapper_stack(support_xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt,
                                                    stack_neighbor_idxs, start_len, cumsum, avg_length_of_neighbor_idxs,
                                                    max_neighbour_distance, nsample, neighbor_type):
    """ref vector_pool.cpp: support_xyz (N,3), new_xyz (M,3) stacked, counts (B) int32 -> the first min(hits, 1000,
    nsample if > 0) hits of every centre as GLOBAL rows, placed at start_len[p] = (atomicAdd(cumsum, L), L) in
    stack_neighbor_idxs (nothing at or beyond avg_length_of_neighbor_idxs * M); cumsum (1) int32 ends as the total"""
    _chk(support_xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt, stack_neighbor_idxs, start_len, cumsum)
    call("tsmdet_stack_local_neighbor_idxs", xyz_batch_cnt.shape[0], new_xyz.shape[0], support_xyz.shape[0],
         ptr(support_xyz), ptr(xyz_batch_cnt), ptr(new_xyz), ptr(new_xyz_batch_cnt), ptr(stack_neighbor_idxs),
         ptr(start_len), ptr(cumsum), int(avg_length_of_neighbor_idxs), float(max_neighbour_distance), int(nsample),
         int(neighbor_type), stream_ptr(support_xyz.device))
    return 1


def query_three_nn_by_stacked_local_idxs_wrapper_stack(support_xyz, new_xyz, new_xyz_grid_centers, new_xyz_grid_idxs,
                                                       new_xyz_grid_dist2, stack_neighbor_idxs, start_len, M,
                                                       num_total_grids):
    """ref vector_pool.cpp: new_xyz_grid_centers (M,G,3) -> new_xyz_grid_idxs (M,G,3) int32 GLOBAL rows and
    new_xyz_grid_dist2 (M,G,3), the three nearest of each centre's list; unfilled slots are (+inf, -1)"""
    _chk(support_xyz, new_xyz, new_xyz_grid_centers, new_xyz_grid_idxs, new_xyz_grid_dist2, stack_neighbor_idxs,
         start_len)
    call("tsmdet_stack_three_nn_local", int(M), int(num_total_grids), support_xyz.shape[0], stack_neighbor_idxs.numel(),
         ptr(support_xyz), ptr(new_xyz_grid_centers), ptr(stack_neighbor_idxs), ptr(start_len), ptr(new_xyz_grid_idxs),
         ptr(new_xyz_grid_dist2), stream_ptr(support_xyz.device))
    return 1


def vector_pool_wrapper(support_xyz, xyz_batch_cnt, support_features, new_xyz, new_xyz_batch_cnt, new_features,
                        new_local_xyz, point_cnt_of_grid, grouped_idxs, num_grid_x, num_grid_y, num_grid_z,
                        max_neighbour_distance, use_xyz, num_max_sum_points, nsample, neighbor_type, pooling_type):
    """ref vector_pool.cpp: sums (average, pooling_type 0) or first hits (random choice, 1) of every sub-voxel added to
    new_features (M, G*cpg), new_local_xyz (M, 3G), point_cnt_of_grid (M,G) int32, triples (k, p, g) in grouped_idxs
    (num_max_sum_points, 3) int32 -> the exact number of triples (a Python int: reads one int back from the device)"""
    import torch

    _chk(support_xyz, xyz_batch_cnt, support_features, new_xyz, new_xyz_batch_cnt, new_features, new_local_xyz,
         point_cnt_of_grid, grouped_idxs)
    total = torch.empty((1,), dtype=torch.int32, device=support_xyz.device)
    call("tsmdet_stack_vector_pool", xyz_batch_cnt.shape[0], new_xyz.shape[0], support_xyz.shape[0],
         support_features.shape[1], new_features.shape[1], ptr(support_xyz), ptr(xyz_batch_cnt), ptr(support_features),
         ptr(new_xyz), ptr(new_xyz_batch_cnt), ptr(new_features), ptr(new_local_xyz), ptr(point_cnt_of_grid),
         ptr(grouped_idxs), int(num_grid_x), int(num_grid_y), int(num_grid_z), float(max_neighbour_distance),
         int(use_xyz), int(num_max_sum_points), int(nsample), int(neighbor_type), int(pooling_type), ptr(total), None,
         stream_ptr(support_xyz.device))
    return int(total.item())


def vector_pool_grad_wrapper(grad_new_features, point_cnt_of_grid, grouped_idxs, grad_support_features):
    """ref vector_pool.cpp: grad_support_features (N,C_in) (zeroed by the caller) += grad_new_features[p, g*cpg + i%cpg]
    * (1 / max(point_cnt_of_grid[p,g], 1)) for every triple (k, p, g) of grouped_idxs (atomic)"""
    _chk(grad_new_features, point_cnt_of_grid, grouped_idxs, grad_support_features)
    call("tsmdet_stack_vector_pool_grad", grad_new_features.shape[0], grad_support_features.shape[0],
         grad_new_features.shape[1], grad_support_features.shape[1], point_cnt_of_grid.shape[1], grouped_idxs.shape[0],
         ptr(grad_new_features), ptr(point_cnt_of_grid), ptr(grouped_idxs), ptr(grad_support_features),
         stream_ptr(grad_new_features.device))
    return 1
