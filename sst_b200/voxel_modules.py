"""Voxel feature encoders registered under the reference's type names (V4, V6).

    DynamicVFE          mmdet3d/models/voxel_encoders/voxel_encoder.py:92-298
    DynamicScatterVFE   mmdet3d/models/voxel_encoders/voxel_encoder.py:502-612
    DynamicVFELayer(V2) mmdet3d/models/voxel_encoders/utils.py:107-189   (parameter containers)

Eval-mode forward is ONE fused libsstb200 call (csrc/vfe.cu).  In training mode (batch-statistics BatchNorm, naiveSyncBN
across ranks, gradients) DynamicVFE runs the reference's own composition (voxel_encoder.py:229-298): the three scatters and
their gradients are libsstb200's DynamicScatter forward / backward kernels (csrc/voxel.cu), the two small Linear layers
(9->64, 128->128; 5 GFLOP, fp32 like the reference's @force_fp32), naiveSyncBN (sst_b200/norm.py, ONE all-reduce per layer) and
ReLU are torch layers under autograd.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib as L
from . import ops
from .registry import VOXEL_ENCODERS


class DynamicVFELayer(nn.Module):
    """utils.py:107-144: linear (no bias) + norm + relu; parameter names `linear.weight`, `norm.*`."""

    def __init__(self, in_channels, out_channels, norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01)):
        super().__init__()
        self.fp16_enabled = False
        self.norm = ops.build_norm_layer(norm_cfg, out_channels)[1]
        self.linear = nn.Linear(in_channels, out_channels, bias=False)


class DynamicVFELayerV2(nn.Module):
    """utils.py:147-189."""

    def __init__(self, in_channels, out_channels, norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01), act="relu",
                 dropout=0.0):
        super().__init__()
        self.fp16_enabled = False
        self.norm = ops.build_norm_layer(norm_cfg, out_channels)[1]
        self.linear = nn.Linear(in_channels, out_channels, bias=False)
        self.act_name = act
        self.dropout = nn.Dropout(p=dropout) if dropout > 0 else None


class _VfeCfg(C.Structure):
    _fields_ = [("in_channels", C.c_int32), ("num_layers", C.c_int32), ("feat_channels", C.c_int32 * 2),
                ("with_cluster_center", C.c_int32), ("with_voxel_center", C.c_int32), ("with_distance", C.c_int32),
                ("mode_max", C.c_int32), ("drop_first_voxel_per_sample", C.c_int32), ("batch_size", C.c_int32),
                ("grid_zyx", C.c_int32 * 3), ("voxel_size", C.c_float * 3), ("center_offset", C.c_float * 3),
                ("rel_dist_scaler", C.c_float), ("bn_eps", C.c_float), ("precision", C.c_int32), ("weight", C.c_void_p * 2),
                ("bn_weight", C.c_void_p * 2), ("bn_bias", C.c_void_p * 2), ("bn_mean", C.c_void_p * 2),
                ("bn_var", C.c_void_p * 2)]


L.SIGNATURES["sstb200_dynamic_vfe_forward"] = (C.c_int, [L.vp, C.POINTER(_VfeCfg), L.vp, L.vp, C.c_int, L.vp, L.vp,
                                                         L.vp, L.P_i32])
L.SIGNATURES["sstb200_dynamic_scatter_vfe_forward"] = (C.c_int, [L.vp, C.POINTER(_VfeCfg), L.vp, L.vp, C.c_int, L.vp,
                                                                 L.vp, L.vp, L.vp, L.P_i32])
L.SIGNATURES["sstb200_dynamic_scatter_vfe_forward_i32"] = (C.c_int, [L.vp, C.POINTER(_VfeCfg), L.vp, L.vp, C.c_int, L.vp, L.vp,
                                                                     L.vp, L.vp])


@VOXEL_ENCODERS.register_module()
class DynamicVFE(nn.Module):
    """voxel_encoder.py:92-298."""
    _drop_first = 1  # DynamicScatter semantics (scatter_points_cuda.cu:207-210), see DESIGN.md "reference quirks"

    def __init__(self, in_channels=4, feat_channels=[], with_distance=False, with_cluster_center=False,
                 with_voxel_center=False, voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1),
                 norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01), mode="max", fusion_layer=None,
                 return_point_feats=False):
        super().__init__()
        assert len(feat_channels) > 0
        if fusion_layer is not None:
            raise NotImplementedError("image fusion layers are outside the hot path")
        self.raw_in_channels = in_channels
        if with_cluster_center:
            in_channels += 3
        if with_voxel_center:
            in_channels += 3
        if with_distance:
            in_channels += 3  # the reference over-counts the distance channel by 2 (voxel_encoder.py:150-151)
        self.in_channels = in_channels
        self._with_distance = with_distance
        self._with_cluster_center = with_cluster_center
        self._with_voxel_center = with_voxel_center
        self.return_point_feats = return_point_feats
        self.fp16_enabled = False
        self.vx, self.vy, self.vz = voxel_size[0], voxel_size[1], voxel_size[2]
        self.x_offset = self.vx / 2 + point_cloud_range[0]
        self.y_offset = self.vy / 2 + point_cloud_range[1]
        self.z_offset = self.vz / 2 + point_cloud_range[2]
        self.point_cloud_range = point_cloud_range
        self.mode = mode
        self.rel_dist_scaler = 1.0
        self.norm_eps = norm_cfg.get("eps", 1e-5)
        chans = [self.in_channels] + list(feat_channels)
        self.vfe_layers = nn.ModuleList(self._make_layer(chans[i] * (2 if i > 0 else 1), chans[i + 1], norm_cfg)
                                        for i in range(len(chans) - 1))
        self.num_vfe = len(self.vfe_layers)
        self.feat_channels = list(feat_channels)

    def _make_layer(self, cin, cout, norm_cfg):
        return DynamicVFELayer(cin, cout, norm_cfg)

    def _canvas(self):
        """Canvas of map_voxel_center_to_point (voxel_encoder.py:199-204: round() in double) - but never smaller than the grid
        the voxeliser emits coordinates on, which is ceil((max-min)/vs) evaluated in FLOAT32 (voxelization_cuda.cu:355-357,
        DESIGN quirk Q2): with a non-integer ratio the two differ by one cell and the last voxel row would fall off the canvas."""
        import numpy as np
        r = self.point_cloud_range
        rnd = (round((r[5] - r[2]) / self.vz), round((r[4] - r[1]) / self.vy), round((r[3] - r[0]) / self.vx))
        f32 = np.float32
        cel = tuple(int(np.ceil((f32(r[3 + i]) - f32(r[i])) / f32(v))) for i, v in ((2, self.vz), (1, self.vy), (0, self.vx)))
        return tuple(max(a, b) for a, b in zip(rnd, cel))

    precision = "fp32"  # 'bf16': second VFE layer on tensor cores (bf16 operands, fp32 accumulate)

    def _cfg(self, batch_size):
        if self._with_distance:
            raise NotImplementedError("with_distance: the reference's channel count is inconsistent (+3 vs 1)")
        if self.num_vfe > 2:
            raise NotImplementedError("fused VFE supports <= 2 layers (all SST/FSD configs)")
        if self.return_point_feats:
            raise NotImplementedError("return_point_feats")
        cfg = _VfeCfg()
        cfg.in_channels = self.raw_in_channels
        cfg.num_layers = self.num_vfe
        for i, ch in enumerate(self.feat_channels):
            cfg.feat_channels[i] = ch
        cfg.with_cluster_center = int(self._with_cluster_center)
        cfg.with_voxel_center = int(self._with_voxel_center)
        cfg.with_distance = 0
        cfg.mode_max = int(self.mode == "max")
        cfg.drop_first_voxel_per_sample = self._drop_first
        cfg.batch_size = int(batch_size)
        cz, cy, cx = self._canvas()
        cfg.grid_zyx[0], cfg.grid_zyx[1], cfg.grid_zyx[2] = cz, cy, cx
        cfg.voxel_size[0], cfg.voxel_size[1], cfg.voxel_size[2] = self.vx, self.vy, self.vz
        cfg.center_offset[0], cfg.center_offset[1], cfg.center_offset[2] = self.x_offset, self.y_offset, self.z_offset
        cfg.rel_dist_scaler = float(self.rel_dist_scaler)
        cfg.bn_eps = float(self.norm_eps)
        cfg.precision = {"fp32": 0, "bf16": 1}[self.precision]
        for i, l in enumerate(self.vfe_layers):
            if not isinstance(l.norm, nn.modules.batchnorm._BatchNorm):
                raise NotImplementedError("fused VFE expects BatchNorm layers")
            cfg.weight[i] = l.linear.weight.data_ptr()
            cfg.bn_weight[i], cfg.bn_bias[i] = l.norm.weight.data_ptr(), l.norm.bias.data_ptr()
            cfg.bn_mean[i], cfg.bn_var[i] = l.norm.running_mean.data_ptr(), l.norm.running_var.data_ptr()
        return cfg

    def _check(self, features, coors):
        ops._need_cuda(features, coors)
        assert features.dtype == torch.float32 and features.shape[1] == self.raw_in_channels
        assert coors.shape[1] == 4

    # ---- training mode: the reference's composition on libsstb200's DynamicScatter ---------------------------------
    def _map_voxel_center_to_point(self, pts_coors, voxel_mean, voxel_coors):
        """voxel_encoder.py:185-225 (dense canvas of row indices; cells of dropped voxels keep index 0 like the reference)."""
        cz, cy, cx = self._canvas()
        batch_size = int(pts_coors[-1, 0]) + 1
        canvas = torch.zeros((cz * cy * cx * batch_size,), dtype=torch.long, device=voxel_mean.device)
        vc = voxel_coors.long()
        canvas[vc[:, 0] * cz * cy * cx + vc[:, 1] * cy * cx + vc[:, 2] * cx + vc[:, 3]] = torch.arange(voxel_mean.size(0), device=voxel_mean.device)
        pc = pts_coors.long()
        return voxel_mean[canvas[pc[:, 0] * cz * cy * cx + pc[:, 1] * cy * cx + pc[:, 2] * cx + pc[:, 3]]]

    def _forward_train(self, features, coors):
        """voxel_encoder.py:229-298 verbatim in structure; see the module docstring for what runs where."""
        if self._with_distance or self.return_point_feats:
            raise NotImplementedError("with_distance / return_point_feats in training mode")
        vs, pr = (self.vx, self.vy, self.vz), self.point_cloud_range
        if not hasattr(self, "_scatters"):
            self._scatters = (ops.DynamicScatter(vs, pr, self.mode != "max"), ops.DynamicScatter(vs, pr, True))
        vfe_scatter, cluster_scatter = self._scatters
        coors = coors.int()
        feats = [features]
        if self._with_cluster_center:
            voxel_mean, mean_coors = cluster_scatter(features, coors)
            points_mean = self._map_voxel_center_to_point(coors, voxel_mean, mean_coors)
            feats.append(features[:, :3] - points_mean[:, :3])
        if self._with_voxel_center:
            f_center = features.new_zeros((features.size(0), 3))
            f_center[:, 0] = features[:, 0] - (coors[:, 3].type_as(features) * self.vx + self.x_offset)
            f_center[:, 1] = features[:, 1] - (coors[:, 2].type_as(features) * self.vy + self.y_offset)
            f_center[:, 2] = features[:, 2] - (coors[:, 1].type_as(features) * self.vz + self.z_offset)
            feats.append(f_center)
        x = torch.cat(feats, dim=-1)
        voxel_feats = voxel_coors = None
        for i, vfe in enumerate(self.vfe_layers):
            point_feats = torch.relu(vfe.norm(vfe.linear(x)))      # utils.py:129-144
            voxel_feats, voxel_coors = vfe_scatter(point_feats, coors)
            if i != len(self.vfe_layers) - 1:
                x = torch.cat([point_feats, self._map_voxel_center_to_point(coors, voxel_feats, voxel_coors)], dim=1)
        return voxel_feats, voxel_coors

    def forward(self, features, coors, points=None, img_feats=None, img_metas=None):
        self._check(features, coors)
        if self.training:
            return self._forward_train(features.contiguous(), coors)
        features, coors = features.contiguous(), coors.int().contiguous()
        P, dev = features.shape[0], features.device
        if P == 0:
            return features.new_zeros((0, self.feat_channels[-1])), coors.new_zeros((0, 4))
        batch_size = int(coors[-1, 0]) + 1  # like scatter_points.py:86
        cfg = self._cfg(batch_size)
        vf = torch.empty((P, self.feat_channels[-1]), dtype=torch.float32, device=dev)
        vc = torch.empty((P, 4), dtype=torch.int32, device=dev)
        num_dev = torch.empty((1,), dtype=torch.int32, device=dev)
        num = C.c_int32(0)
        c = L.ctx(dev)
        L.check(c, L.lib().sstb200_dynamic_vfe_forward(c, C.byref(cfg), features.data_ptr(), coors.data_ptr(), P,
                                                       vf.data_ptr(), vc.data_ptr(), num_dev.data_ptr(), C.byref(num)))
        return vf[:num.value], vc[:num.value]


def _scatter_vfe_train(self, features, coors, return_inv):
    """voxel_encoder.py:551-612 as a composition: ONE voxel index (`ops.unique_rows`; unique_once or not gives the same result), segmented
    reductions with their backward kernels (`ops.segment_reduce`: mean / sum gradients gathered, max gradient to the arg-max row),
    torch Linear + (naiveSync)BatchNorm + ReLU in between - batch statistics and autograd like the reference's training mode."""
    if self.return_point_feats:
        raise NotImplementedError("return_point_feats in training mode")
    new_coors, inv = ops.unique_rows(coors)
    M = new_coors.shape[0]
    mode = "mean" if self.mode == "avg" else self.mode
    feats = [features]
    if self._with_cluster_center:
        voxel_mean, _ = ops.segment_reduce(features[:, :3].contiguous(), inv, "mean", M, want_argmax=False)
        feats.append((features[:, :3] - voxel_mean[inv]) / self.rel_dist_scaler)
    if self._with_voxel_center:
        centre = torch.stack([coors[:, 3].type_as(features) * self.vx + self.x_offset, coors[:, 2].type_as(features) * self.vy + self.y_offset,
                              coors[:, 1].type_as(features) * self.vz + self.z_offset], 1)
        feats.append(features[:, :3] - centre)
    if self._with_distance:
        feats.append(torch.norm(features[:, :3], 2, 1, keepdim=True))
    x = torch.cat(feats, dim=-1)
    voxel_feats = None
    for i, vfe in enumerate(self.vfe_layers):
        point_feats = torch.relu(vfe.norm(vfe.linear(x)))          # utils.py:147-189 (act = relu, dropout 0)
        voxel_feats, _ = ops.segment_reduce(point_feats, inv, mode, M)
        if i != len(self.vfe_layers) - 1:
            x = torch.cat([point_feats, voxel_feats[inv]], dim=1)
    return (voxel_feats, new_coors, inv) if return_inv else (voxel_feats, new_coors)


@VOXEL_ENCODERS.register_module()
class DynamicScatterVFE(DynamicVFE):
    """voxel_encoder.py:502-612 (torch.unique based: no voxel is dropped; int64 coors; returns unq_inv)."""
    _drop_first = 0

    def __init__(self, in_channels=4, feat_channels=[], with_distance=False, with_cluster_center=False,
                 with_voxel_center=False, voxel_size=(0.2, 0.2, 4), point_cloud_range=(0, -40, -3, 70.4, 40, 1),
                 norm_cfg=dict(type="BN1d", eps=1e-3, momentum=0.01), mode="max", fusion_layer=None,
                 return_point_feats=False, return_inv=True, rel_dist_scaler=1.0, unique_once=False):
        super().__init__(in_channels, feat_channels, with_distance, with_cluster_center, with_voxel_center, voxel_size,
                         point_cloud_range, norm_cfg, mode, fusion_layer, return_point_feats)
        self.rel_dist_scaler = rel_dist_scaler
        self.unique_once = unique_once

    _forward_train_scatter = _scatter_vfe_train

    def forward(self, features, coors, points=None, img_feats=None, img_metas=None, return_inv=False):
        self._check(features, coors)
        if self.training or (torch.is_grad_enabled() and features.requires_grad):
            return self._forward_train_scatter(features.contiguous(), coors.long().contiguous(), return_inv)
        features, coors = features.contiguous(), coors.long().contiguous()
        P, dev = features.shape[0], features.device
        if P == 0:
            e = (features.new_zeros((0, self.feat_channels[-1])), coors.new_zeros((0, 4)))
            return e + (coors.new_zeros((0,)),) if return_inv else e
        batch_size = int(coors[:, 0].max()) + 1
        cfg = self._cfg(batch_size)
        # coordinates may exceed the nominal canvas (e.g. virtual voxels): bound the bitmap by what is present
        hi = coors[:, 1:].amax(0).tolist()
        for i in range(3):
            cfg.grid_zyx[i] = max(cfg.grid_zyx[i], int(hi[i]) + 1)
        vf = torch.empty((P, self.feat_channels[-1]), dtype=torch.float32, device=dev)
        vc = torch.empty((P, 4), dtype=torch.int64, device=dev)
        inv = torch.empty((P,), dtype=torch.int64, device=dev)
        num_dev = torch.empty((1,), dtype=torch.int32, device=dev)
        num = C.c_int32(0)
        c = L.ctx(dev)
        L.check(c, L.lib().sstb200_dynamic_scatter_vfe_forward(
            c, C.byref(cfg), features.data_ptr(), coors.data_ptr(), P, vf.data_ptr(), vc.data_ptr(), inv.data_ptr(),
            num_dev.data_ptr(), C.byref(num)))
        if return_inv:
            return vf[:num.value], vc[:num.value], inv
        return vf[:num.value], vc[:num.value]
