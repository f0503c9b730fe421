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
"""
from __future__ import annotations

from typing import List

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import pointnet2_modules as _batch
from .._lib import call, ptr, stream_ptr
from . import pointnet2_utils

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
