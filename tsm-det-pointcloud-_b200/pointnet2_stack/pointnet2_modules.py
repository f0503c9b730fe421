"""``StackSAModuleMSG`` (:11-94) and ``StackPointnetFPModule`` of
``/root/reference/pcdet/ops/pointnet2/pointnet2_stack/pointnet2_modules.py``: the multi-scale set abstraction over
stacked (ragged) frames that the VSA module of the detection head builds (``backbones_3d/pfe/voxel_set_abstraction.py``),
and the feature propagation that stacked backbones pair with it.

Two execution modes give the same numbers within the tolerances of ``tests/parity.py``:
  ``fused=False`` (or train mode, or ``pool_method='avg_pool'``)  the reference's eager sequence: ``QueryAndGroup``
                   (stack ball query -> stacked grouping -> zeroed empty balls) -> Conv2d/BatchNorm2d/ReLU -> pool;
  ``fused=True``   (eval mode, ``max_pool``) per scale ONE ball query with global rows and hit counts, then the fused
                   SA kernel of the dense-batch module (gather + MLP + max-pool, BatchNorm folded): the stacked layout
                   seen as one cloud, xyz (1,N,3), new_xyz (1,M,3), idx (1,M,nsample), is exactly its input.
                   ``precision`` 'fp32' | 'bf16' | 'tf32' as for ``PointnetSAModuleFSMSG``.
``StackPointnetFPModule`` likewise: eager (``fused=False`` or train mode) is the reference's sequence; in eval mode the
stacked 3-NN feeds an interpolation kernel that writes the point-wise MLP's (1,C2,N) input planes, and the dense-batch
FP module's fused MLP (``pointwise_mlp``) takes them with the skip features, never materialising the concatenation.
``VectorPoolAggregationModule(MSG)`` (PV-RCNN++'s local vector representation) likewise: eager (``fused=False`` or train
mode) is the reference's sequence over the vector-pool wrappers; in eval mode one kernel writes the grouped layer's
(1, G*(3+C), M) / (1, G*(C+9), M) input planes straight from the neighbour search (``voxel_avg_pool`` /
``voxel_random_choice``: the normalised sub-voxel means; ``local_interpolation``: the sub-voxels' 3-NN without a neighbour
list, then the interpolation), with no host synchronisation; the grouped Conv1d and the post MLPs stay torch modules.
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import pointnet2_modules as _batch
from .._lib import call, ptr, stream_ptr
from . import pointnet2_utils
from .pointnet2_utils import local_interp_weights

_ROW_Q = {"bf16": 8, "tf32": 4}  # feature-row padding of the tensor-core kernels (channels)


def stack_feature_rows(features: torch.Tensor, precision: str) -> torch.Tensor:
    """features (N,C) fp32 -> (1, N, round_up(C, 8)) bf16 ('bf16') or (1, N, round_up(C, 4)) fp32 holding tf32 values
    ('tf32'): the fused SA kernels' ``feat_t`` rows, rounded as those kernels round (B,C,N) planes themselves."""
    assert features.is_cuda and features.dtype == torch.float32 and features.is_contiguous() and features.dim() == 2
    n, c = features.shape
    q = _ROW_Q[precision]
    rows = torch.empty((1, n, (c + q - 1) // q * q), dtype=torch.bfloat16 if precision == "bf16" else torch.float32,
                       device=features.device)
    call("tsmdet_stack_feature_rows", _batch.PRECISIONS[precision], n, c, ptr(features), ptr(rows),
         stream_ptr(features.device))
    return rows


class StackSAModuleMSG(nn.Module):
    """ref :11-94.  ``mlps[i]`` lists the channels WITHOUT the +3 for xyz, as in the reference's config."""

    def __init__(self, *, radii: List[float], nsamples: List[int], mlps: List[List[int]], use_xyz: bool = True,
                 pool_method: str = 'max_pool', fused: bool = True, precision: str = "fp32"):
        super().__init__()
        assert len(radii) == len(nsamples) == len(mlps)
        self.groupers = nn.ModuleList()
        self.mlps = nn.ModuleList()
        for radius, nsample, spec in zip(radii, nsamples, mlps):
            self.groupers.append(pointnet2_utils.QueryAndGroup(radius, nsample, use_xyz=use_xyz))
            spec = list(spec)
            if use_xyz:
                spec[0] += 3
            self.mlps.append(_batch.build_shared_mlp(spec, bn=True))  # [Conv2d 1x1 (no bias), BatchNorm2d, ReLU]*
        self.pool_method = pool_method
        self.use_xyz = use_xyz
        self.fused = fused
        self.precision = precision
        self._folded = None  # per scale: folded (W, b), built lazily in eval mode
        self._packed = None
        self.init_weights()

    def init_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            if isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1.0)
                nn.init.constant_(m.bias, 0)

    def train(self, mode: bool = True):
        self._folded = None
        return super().train(mode)

    def _load_from_state_dict(self, *args, **kwargs):
        self._folded = None  # the fused path must not keep running on the folds of the previous weights
        return super()._load_from_state_dict(*args, **kwargs)

    def _folded_layers(self):
        if self._folded is None:
            self._folded = [_batch.fold_conv_bn(m) for m in self.mlps]
            self._packed = None
        return self._folded

    def _packed_layers(self, c_feat: int, use_xyz: bool):
        folded = self._folded_layers()
        if self._packed is None or self._packed[0] != (c_feat, use_xyz, self.precision):
            imgs = [_batch.pack_mlp(layers, dense=False, nsample=g.nsample, c_feat=c_feat, use_xyz=use_xyz,
                                    precision=self.precision) if self.precision in ("bf16", "tf32") else None
                    for layers, g in zip(folded, self.groupers)]
            self._packed = ((c_feat, use_xyz, self.precision), imgs)
        return self._packed[1]

    def forward(self, xyz: torch.Tensor, xyz_batch_cnt: torch.Tensor, new_xyz: torch.Tensor,
                new_xyz_batch_cnt: torch.Tensor, features: torch.Tensor = None, empty_voxel_set_zeros: bool = True):
        """xyz (N1+N2..., 3), xyz_batch_cnt (B) int32, new_xyz (M1+M2..., 3), new_xyz_batch_cnt (B) int32,
        features (N1+N2..., C) | None -> (new_xyz, new_features (M1+M2..., sum of the scales' last widths))"""
        if self.fused and not self.training and self.pool_method == 'max_pool':
            return new_xyz, self._forward_fused(xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt, features)
        new_features_list = []
        for grouper, mlp in zip(self.groupers, self.mlps):
            new_features, _ = grouper(xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt, features)  # (M, C, nsample)
            new_features = new_features.permute(1, 0, 2).unsqueeze(dim=0)  # (1, C, M, nsample)
            new_features = mlp(new_features)
            if self.pool_method == 'max_pool':
                new_features = F.max_pool2d(new_features, kernel_size=[1, new_features.size(3)]).squeeze(dim=-1)
            elif self.pool_method == 'avg_pool':
                new_features = F.avg_pool2d(new_features, kernel_size=[1, new_features.size(3)]).squeeze(dim=-1)
            else:
                raise NotImplementedError
            new_features_list.append(new_features.squeeze(dim=0).permute(1, 0))  # (M, C)
        return new_xyz, torch.cat(new_features_list, dim=1)

    @torch.no_grad()
    def _forward_fused(self, xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt, features):
        assert xyz.shape[0] == xyz_batch_cnt.sum() and new_xyz.shape[0] == new_xyz_batch_cnt.sum()
        assert features is not None or self.use_xyz, "Cannot have not features and not use xyz as a feature!"
        xyz, new_xyz = xyz.contiguous(), new_xyz.contiguous()
        xyz_batch_cnt, new_xyz_batch_cnt = xyz_batch_cnt.int().contiguous(), new_xyz_batch_cnt.int().contiguous()
        n, m, b = xyz.shape[0], new_xyz.shape[0], xyz_batch_cnt.shape[0]
        c_feat = 0 if features is None else features.shape[1]
        folded = self._folded_layers()
        packed = self._packed_layers(c_feat, self.use_xyz)
        widths = [layers[-1][0].shape[0] for layers in folded]
        out = torch.empty((1, sum(widths), m), dtype=torch.float32, device=xyz.device)
        xyz1, new_xyz1 = xyz.view(1, n, 3), new_xyz.view(1, m, 3)
        inputs = {}  # what the kernels read the features from, built once per forward: planes or per-precision rows

        def feature_input(precision, img):
            if features is None:
                return None, None
            if img is not None and precision in _ROW_Q and c_feat > 4:  # packed tensor path, rows of >4 channels
                if precision not in inputs:
                    inputs[precision] = stack_feature_rows(features.contiguous(), precision)
                return None, inputs[precision]
            if "planes" not in inputs:  # (1, C, N): the fp32 kernel, and <= 4 channels read straight from planes
                inputs["planes"] = features.t().contiguous().view(1, c_feat, n)
            return inputs["planes"], None

        c0 = 0
        for grouper, layers, w, img in zip(self.groupers, folded, widths, packed):
            s = grouper.nsample
            idx = torch.empty((1, m, s), dtype=torch.int32, device=xyz.device)
            idx_cnt = torch.empty((1, m), dtype=torch.int32, device=xyz.device)
            call("tsmdet_stack_ball_query", b, m, n, float(grouper.radius), s, ptr(new_xyz), ptr(new_xyz_batch_cnt),
                 ptr(xyz), ptr(xyz_batch_cnt), ptr(idx), ptr(idx_cnt), 1, stream_ptr(xyz.device))
            precision = _batch._effective_precision(self.precision, img)
            planes, rows = feature_input(precision, img)
            _batch.sa_mlp_maxpool(xyz1, new_xyz1, planes, idx, idx_cnt, layers, out, c0, use_xyz=self.use_xyz,
                                  precision=precision, packed=img, feat_t=rows)
            c0 += w
        return out[0].t().contiguous()


def _interp_weights(dist: torch.Tensor) -> torch.Tensor:
    """inverse-distance weights of the three neighbours, normalised (ref StackPointnetFPModule.forward); 0/0 = NaN for an
    unknown point whose frame has no known points"""
    dist_recip = 1.0 / (dist + 1e-8)
    norm = torch.sum(dist_recip, dim=-1, keepdim=True)
    return dist_recip / norm


def _dense_precision(precision: str, packed) -> str:
    """The kernel an FP layer's MLP runs in: the point-wise tensor-core path takes exactly the shapes ``pack_mlp`` packs
    (it has no first-generation fallback), so an MLP without a weight image, e.g. [768,512,512], runs in the fp32 FMA
    kernel -- tighter, slower, never looser than asked for."""
    return "fp32" if packed is None else precision


class StackPointnetFPModule(nn.Module):
    """ref StackPointnetFPModule: ``mlp`` = [C2 + C1, ...], [Conv2d 1x1 (no bias), BatchNorm2d, ReLU]* (state_dict keys
    ``mlp.{3k}.weight``, ``mlp.{3k+1}.*``).  ``fused`` (eval mode only) and ``precision`` 'fp32' | 'bf16' | 'tf32' as for
    the dense-batch ``PointnetFPModule``."""

    def __init__(self, *, mlp: List[int], fused: bool = True, precision: str = "fp32"):
        super().__init__()
        self.mlp = _batch.build_shared_mlp(mlp, bn=True)
        self.fused = fused
        self.precision = precision
        self._folded = None  # folded (W, b), built lazily in eval mode
        self._packed = None

    def train(self, mode: bool = True):
        self._folded = None
        return super().train(mode)

    def _load_from_state_dict(self, *args, **kwargs):
        self._folded = None  # the fused path must not keep running on the folds of the previous weights
        return super()._load_from_state_dict(*args, **kwargs)

    def _folded_layers(self):
        if self._folded is None:
            self._folded = _batch.fold_conv_bn(self.mlp)
            self._packed = None
        return self._folded

    def _packed_layers(self, c2: int, c1: int):
        folded = self._folded_layers()
        if self._packed is None or self._packed[0] != (c2, c1, self.precision):
            img = (_batch.pack_mlp(folded, dense=True, c_feat=c2, c1=c1, precision=self.precision)
                   if self.precision in ("bf16", "tf32") else None)
            self._packed = ((c2, c1, self.precision), img)
        return self._packed[1]

    def forward(self, unknown, unknown_batch_cnt, known, known_batch_cnt, unknown_feats=None, known_feats=None):
        """unknown (N1+N2..., 3), unknown_batch_cnt (B), known (M1+M2..., 3), known_batch_cnt (B),
        unknown_feats (N1+N2..., C1) | None, known_feats (M1+M2..., C2) -> (N1+N2..., mlp[-1])"""
        if self.fused and not self.training:
            return self._forward_fused(unknown, unknown_batch_cnt, known, known_batch_cnt, unknown_feats, known_feats)
        dist, idx = pointnet2_utils.three_nn(unknown, unknown_batch_cnt, known, known_batch_cnt)
        weight = _interp_weights(dist)
        interpolated_feats = pointnet2_utils.three_interpolate(known_feats, idx, weight)
        if unknown_feats is not None:
            new_features = torch.cat([interpolated_feats, unknown_feats], dim=1)  # (N1 + N2 ..., C2 + C1)
        else:
            new_features = interpolated_feats
        new_features = new_features.permute(1, 0)[None, :, :, None]  # (1, C, N1 + N2 ..., 1)
        new_features = self.mlp(new_features)
        return new_features.squeeze(dim=0).squeeze(dim=-1).permute(1, 0)  # (N1 + N2 ..., C)

    @torch.no_grad()
    def _forward_fused(self, unknown, unknown_batch_cnt, known, known_batch_cnt, unknown_feats, known_feats):
        dist, idx = pointnet2_utils.three_nn(unknown, unknown_batch_cnt, known, known_batch_cnt)
        weight = _interp_weights(dist)  # the eager path's weights, bit for bit
        known_feats = known_feats.contiguous()
        n, (m, c2) = unknown.shape[0], known_feats.shape
        c1 = 0 if unknown_feats is None else unknown_feats.shape[1]
        planes = torch.empty((1, c2, n), dtype=torch.float32, device=unknown.device)
        call("tsmdet_stack_three_interpolate", n, c2, m, ptr(known_feats), ptr(idx), ptr(weight.contiguous()),
             ptr(planes), 1, stream_ptr(unknown.device))
        skip = None if unknown_feats is None else unknown_feats.t().contiguous().view(1, c1, n)
        packed = self._packed_layers(c2, c1)
        out = _batch.pointwise_mlp(planes, skip, self._folded, precision=_dense_precision(self.precision, packed),
                                   packed=packed)
        # a frame without known points has 0/0 weights: the eager path's rows are NaN there, whatever the MLP's ReLU
        # makes of a NaN input
        w0 = weight[:, :1]
        return torch.where(torch.isnan(w0), w0, out[0].t()).contiguous()


class VectorPoolAggregationModule(nn.Module):
    """ref VectorPoolAggregationModule: the hits of every centre's cube / ball of ``max_neighbor_distance`` reduced to
    ``num_local_voxel`` sub-voxels (``local_aggregation_type`` 'local_interpolation' | 'voxel_avg_pool' |
    'voxel_random_choice'), a grouped Conv1d per sub-voxel (``separate_local_aggregation_layer``) and ``post_mlps``.
    Same constructor, initialisation and state_dict keys; ``fused`` (eval mode only) writes the grouped layer's input
    planes in one kernel."""

    def __init__(self, input_channels, num_local_voxel=(3, 3, 3), local_aggregation_type='local_interpolation',
                 num_reduced_channels=30, num_channels_of_local_aggregation=32, post_mlps=(128,),
                 max_neighbor_distance=None, neighbor_nsample=-1, neighbor_type=0, neighbor_distance_multiplier=2.0,
                 fused: bool = True):
        super().__init__()
        self.num_local_voxel = num_local_voxel
        self.total_voxels = self.num_local_voxel[0] * self.num_local_voxel[1] * self.num_local_voxel[2]
        self.local_aggregation_type = local_aggregation_type
        assert self.local_aggregation_type in ['local_interpolation', 'voxel_avg_pool', 'voxel_random_choice']
        self.input_channels = input_channels
        self.num_reduced_channels = input_channels if num_reduced_channels is None else num_reduced_channels
        self.num_channels_of_local_aggregation = num_channels_of_local_aggregation
        self.max_neighbour_distance = max_neighbor_distance
        self.neighbor_nsample = neighbor_nsample
        self.neighbor_type = neighbor_type  # 1: ball, others: cube
        self.fused = fused

        if self.local_aggregation_type == 'local_interpolation':
            self.local_interpolate_module = pointnet2_utils.VectorPoolLocalInterpolateModule(
                mlp=None, num_voxels=self.num_local_voxel, max_neighbour_distance=self.max_neighbour_distance,
                nsample=self.neighbor_nsample, neighbor_type=self.neighbor_type,
                neighbour_distance_multiplier=neighbor_distance_multiplier)
            num_c_in = (self.num_reduced_channels + 9) * self.total_voxels
        else:
            self.local_interpolate_module = None
            num_c_in = (self.num_reduced_channels + 3) * self.total_voxels

        num_c_out = self.total_voxels * self.num_channels_of_local_aggregation

        self.separate_local_aggregation_layer = nn.Sequential(
            nn.Conv1d(num_c_in, num_c_out, kernel_size=1, groups=self.total_voxels, bias=False),
            nn.BatchNorm1d(num_c_out),
            nn.ReLU()
        )

        post_mlp_list = []
        c_in = num_c_out
        for cur_num_c in post_mlps:
            post_mlp_list.extend([
                nn.Conv1d(c_in, cur_num_c, kernel_size=1, bias=False),
                nn.BatchNorm1d(cur_num_c),
                nn.ReLU()
            ])
            c_in = cur_num_c
        self.post_mlps = nn.Sequential(*post_mlp_list)

        self.num_mean_points_per_grid = 20
        self.init_weights()

    def init_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Conv2d) or isinstance(m, nn.Conv1d):
                nn.init.kaiming_normal_(m.weight)
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)
            if isinstance(m, nn.BatchNorm2d) or isinstance(m, nn.BatchNorm1d):
                nn.init.constant_(m.weight, 1.0)
                nn.init.constant_(m.bias, 0)

    def extra_repr(self) -> str:
        return (f'radius={self.max_neighbour_distance}, local_voxels=({self.num_local_voxel}, '
                f'local_aggregation_type={self.local_aggregation_type}, '
                f'num_c_reduction={self.input_channels}->{self.num_reduced_channels}, '
                f'num_c_local_aggregation={self.num_channels_of_local_aggregation}')

    def vector_pool_with_voxel_query(self, xyz, xyz_batch_cnt, features, new_xyz, new_xyz_batch_cnt):
        use_xyz = 1
        pooling_type = 0 if self.local_aggregation_type == 'voxel_avg_pool' else 1

        new_features, new_local_xyz, num_mean_points_per_grid, point_cnt_of_grid = \
            pointnet2_utils.vector_pool_with_voxel_query_op(
                xyz, xyz_batch_cnt, features, new_xyz, new_xyz_batch_cnt,
                self.num_local_voxel[0], self.num_local_voxel[1], self.num_local_voxel[2],
                self.max_neighbour_distance, self.num_reduced_channels, use_xyz,
                self.num_mean_points_per_grid, self.neighbor_nsample, self.neighbor_type, pooling_type)
        self.num_mean_points_per_grid = max(self.num_mean_points_per_grid, num_mean_points_per_grid.item())

        num_new_pts = new_features.shape[0]
        new_local_xyz = new_local_xyz.view(num_new_pts, -1, 3)  # (M, G, 3)
        new_features = new_features.view(num_new_pts, -1, self.num_reduced_channels)  # (M, G, C)
        new_features = torch.cat((new_local_xyz, new_features), dim=-1).view(num_new_pts, -1)
        return new_features, point_cnt_of_grid

    @staticmethod
    def get_dense_voxels_by_center(point_centers, max_neighbour_distance, num_voxels):
        """point_centers (M,3) -> voxel_centers (M, G, 3), the sub-voxel centres of each centre's cube"""
        R = max_neighbour_distance
        device = point_centers.device
        x_grids = torch.arange(-R + R / num_voxels[0], R - R / num_voxels[0] + 1e-5, 2 * R / num_voxels[0], device=device)
        y_grids = torch.arange(-R + R / num_voxels[1], R - R / num_voxels[1] + 1e-5, 2 * R / num_voxels[1], device=device)
        z_grids = torch.arange(-R + R / num_voxels[2], R - R / num_voxels[2] + 1e-5, 2 * R / num_voxels[2], device=device)
        x_offset, y_offset, z_offset = torch.meshgrid(x_grids, y_grids, z_grids, indexing='ij')  # [nx, ny, nz]
        xyz_offset = torch.cat((
            x_offset.contiguous().view(-1, 1),
            y_offset.contiguous().view(-1, 1),
            z_offset.contiguous().view(-1, 1)), dim=-1
        )
        voxel_centers = point_centers[:, None, :] + xyz_offset[None, :, :]
        return voxel_centers

    def vector_pool_with_local_interpolate(self, xyz, xyz_batch_cnt, features, new_xyz, new_xyz_batch_cnt):
        """-> (M, G * (C + 9))"""
        voxel_centers = self.get_dense_voxels_by_center(
            point_centers=new_xyz, max_neighbour_distance=self.max_neighbour_distance, num_voxels=self.num_local_voxel)
        voxel_features = self.local_interpolate_module.forward(
            support_xyz=xyz, support_features=features, xyz_batch_cnt=xyz_batch_cnt,
            new_xyz=new_xyz, new_xyz_grid_centers=voxel_centers, new_xyz_batch_cnt=new_xyz_batch_cnt)
        voxel_features = voxel_features.contiguous().view(-1, self.total_voxels * voxel_features.shape[-1])
        return voxel_features

    def forward(self, xyz, xyz_batch_cnt, new_xyz, new_xyz_batch_cnt, features, **kwargs):
        """xyz (N1+N2..., 3), xyz_batch_cnt (B), new_xyz (M1+M2..., 3), new_xyz_batch_cnt (B), features (N1+N2..., C)
        -> (new_xyz, new_features (M1+M2..., post_mlps[-1]))"""
        N, C = features.shape

        assert C % self.num_reduced_channels == 0, \
            f'the input channels ({C}) should be an integral multiple of num_reduced_channels({self.num_reduced_channels})'

        features = features.view(N, -1, self.num_reduced_channels).sum(dim=1)

        if self.fused and not self.training:
            vector_features = self.input_planes(xyz, xyz_batch_cnt, features, new_xyz, new_xyz_batch_cnt)
        else:
            if self.local_aggregation_type in ['voxel_avg_pool', 'voxel_random_choice']:
                vector_features, point_cnt_of_grid = self.vector_pool_with_voxel_query(
                    xyz=xyz, xyz_batch_cnt=xyz_batch_cnt, features=features,
                    new_xyz=new_xyz, new_xyz_batch_cnt=new_xyz_batch_cnt)
            elif self.local_aggregation_type == 'local_interpolation':
                vector_features = self.vector_pool_with_local_interpolate(
                    xyz=xyz, xyz_batch_cnt=xyz_batch_cnt, features=features,
                    new_xyz=new_xyz, new_xyz_batch_cnt=new_xyz_batch_cnt)  # (M1 + M2 + ..., G * C)
            else:
                raise NotImplementedError
            vector_features = vector_features.permute(1, 0)[None, :, :]  # (1, G * C, M1 + M2 ...)

        new_features = self.separate_local_aggregation_layer(vector_features)

        new_features = self.post_mlps(new_features)
        new_features = new_features.squeeze(dim=0).permute(1, 0)
        return new_xyz, new_features

    @torch.no_grad()
    def input_planes(self, xyz, xyz_batch_cnt, features, new_xyz, new_xyz_batch_cnt):
        """The grouped layer's input (1, G * (3 + C), M) or (1, G * (C + 9), M), equal bit for bit to the eager path's
        ``vector_features.permute(1, 0)[None]``, written by one kernel after the neighbour search; no host
        synchronisation.  ``features`` (N, C) are the reduced features."""
        xyz, new_xyz = xyz.contiguous(), new_xyz.contiguous()
        xyz_batch_cnt, new_xyz_batch_cnt = xyz_batch_cnt.int().contiguous(), new_xyz_batch_cnt.int().contiguous()
        features = features.contiguous()
        (n, c), m, b = features.shape, new_xyz.shape[0], xyz_batch_cnt.shape[0]
        G = self.total_voxels
        nx, ny, nz = self.num_local_voxel
        dev = xyz.device
        if self.local_aggregation_type == 'local_interpolation':
            li = self.local_interpolate_module
            centres = self.get_dense_voxels_by_center(new_xyz, self.max_neighbour_distance, self.num_local_voxel)
            centres = centres.contiguous()
            idx = torch.empty((m, G, 3), dtype=torch.int32, device=dev)
            dist2 = torch.empty((m, G, 3), dtype=torch.float32, device=dev)
            call("tsmdet_stack_vector_three_nn", b, m, n, G, ptr(xyz), ptr(xyz_batch_cnt), ptr(new_xyz),
                 ptr(new_xyz_batch_cnt), ptr(centres), float(li.max_neighbour_distance * li.neighbor_distance_multiplier),
                 int(li.nsample), int(li.neighbor_type), ptr(idx), ptr(dist2), stream_ptr(dev))
            weight = local_interp_weights(torch.sqrt(dist2)).contiguous()  # the eager path's weights, bit for bit
            planes = torch.empty((1, G * (c + 9), m), dtype=torch.float32, device=dev)
            call("tsmdet_stack_vector_interp_planes", m, G, n, c, ptr(features), ptr(xyz), ptr(centres), ptr(idx),
                 ptr(weight), ptr(planes), stream_ptr(dev))
            return planes
        pooling_type = 0 if self.local_aggregation_type == 'voxel_avg_pool' else 1
        planes = torch.empty((1, G * (3 + self.num_reduced_channels), m), dtype=torch.float32, device=dev)
        call("tsmdet_stack_vector_pool", b, m, n, c, G * self.num_reduced_channels, ptr(xyz), ptr(xyz_batch_cnt),
             ptr(features), ptr(new_xyz), ptr(new_xyz_batch_cnt), None, None, None, None, nx, ny, nz,
             float(self.max_neighbour_distance), 1, 0, int(self.neighbor_nsample), int(self.neighbor_type), pooling_type,
             None, ptr(planes), stream_ptr(dev))
        return planes


class VectorPoolAggregationModuleMSG(nn.Module):
    """ref VectorPoolAggregationModuleMSG: ``config.NUM_GROUPS`` VectorPoolAggregationModule layers (``layer_{k}``,
    ``config.GROUP_CFG_{k}``), their features concatenated after new_xyz, then ``msg_post_mlps``."""

    def __init__(self, input_channels, config, fused: bool = True):
        super().__init__()
        self.model_cfg = config
        self.num_groups = self.model_cfg.NUM_GROUPS

        self.layers = []
        c_in = 0
        for k in range(self.num_groups):
            cur_config = self.model_cfg[f'GROUP_CFG_{k}']
            cur_vector_pool_module = VectorPoolAggregationModule(
                input_channels=input_channels, num_local_voxel=cur_config.NUM_LOCAL_VOXEL,
                post_mlps=cur_config.POST_MLPS,
                max_neighbor_distance=cur_config.MAX_NEIGHBOR_DISTANCE,
                neighbor_nsample=cur_config.NEIGHBOR_NSAMPLE,
                local_aggregation_type=self.model_cfg.LOCAL_AGGREGATION_TYPE,
                num_reduced_channels=self.model_cfg.get('NUM_REDUCED_CHANNELS', None),
                num_channels_of_local_aggregation=self.model_cfg.NUM_CHANNELS_OF_LOCAL_AGGREGATION,
                neighbor_distance_multiplier=2.0,
                fused=fused,
            )
            self.__setattr__(f'layer_{k}', cur_vector_pool_module)
            c_in += cur_config.POST_MLPS[-1]

        c_in += 3  # use_xyz

        shared_mlps = []
        for cur_num_c in self.model_cfg.MSG_POST_MLPS:
            shared_mlps.extend([
                nn.Conv1d(c_in, cur_num_c, kernel_size=1, bias=False),
                nn.BatchNorm1d(cur_num_c),
                nn.ReLU()
            ])
            c_in = cur_num_c
        self.msg_post_mlps = nn.Sequential(*shared_mlps)

    def forward(self, **kwargs):
        features_list = []
        for k in range(self.num_groups):
            cur_xyz, cur_features = self.__getattr__(f'layer_{k}')(**kwargs)
            features_list.append(cur_features)

        features = torch.cat(features_list, dim=-1)
        features = torch.cat((cur_xyz, features), dim=-1)
        features = features.permute(1, 0)[None, :, :]  # (1, C, N)
        new_features = self.msg_post_mlps(features)
        new_features = new_features.squeeze(dim=0).permute(1, 0)  # (N, C)
        return cur_xyz, new_features


def build_local_aggregation_module(input_channels, config):
    """ref build_local_aggregation_module (the VSA module's builder): ``config.NAME`` 'StackSAModuleMSG' (default) or
    'VectorPoolAggregationModuleMSG' -> (module, number of output channels)"""
    local_aggregation_name = config.get('NAME', 'StackSAModuleMSG')

    if local_aggregation_name == 'StackSAModuleMSG':
        mlps = config.MLPS
        for k in range(len(mlps)):
            mlps[k] = [input_channels] + mlps[k]
        cur_layer = StackSAModuleMSG(
            radii=config.POOL_RADIUS, nsamples=config.NSAMPLE, mlps=mlps, use_xyz=True, pool_method='max_pool',
        )
        num_c_out = sum([x[-1] for x in mlps])
    elif local_aggregation_name == 'VectorPoolAggregationModuleMSG':
        cur_layer = VectorPoolAggregationModuleMSG(input_channels=input_channels, config=config)
        num_c_out = config.MSG_POST_MLPS[-1]
    else:
        raise NotImplementedError

    return cur_layer, num_c_out
