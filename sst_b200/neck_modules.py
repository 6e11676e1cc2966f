"""FSD's voxel -> point neck under the reference's registered name (SURVEY 8f next-2).

    Voxel2PointScatterNeck   mmdet3d/models/necks/voxel2point_neck.py:9-62
    reorder                  mmdet3d/models/detectors/single_stage_fsd.py:253-266 (VoteSegmentor.reorder)
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib as L
from . import ops
from .registry import MODELS

NECKS = MODELS

L.SIGNATURES["sstb200_voxel2point"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, L.vp, C.c_int, C.c_int, L.vp, C.c_int, C.c_float, L.P_f32,
                                                 L.P_f32, C.c_int, C.c_int, L.vp, L.vp, L.vp, L.P_i32])
L.SIGNATURES["sstb200_voxel2point_dev"] = (C.c_int, [L.vp, L.vp, C.c_int, L.vp, L.vp, L.vp, C.c_int, L.vp, C.c_int, C.c_float, L.P_f32,
                                                     L.P_f32, C.c_int, C.c_int, L.vp, L.vp, L.vp])


@NECKS.register_module()
class Voxel2PointScatterNeck(nn.Module):
    """voxel2point_neck.py:9-62.  Returns (results [n_kept, C(+3)], pts_mask [N] bool)."""

    def __init__(self, point_cloud_range=None, voxel_size=None, with_xyz=True, normalize_local_xyz=False):
        super().__init__()
        self.point_cloud_range = point_cloud_range
        self.voxel_size = voxel_size
        self.with_xyz = with_xyz
        self.normalize_local_xyz = normalize_local_xyz

    def forward(self, points, pts_coors, voxel_feats, voxel2point_inds, voxel_padding=-1):
        assert points.size(0) == pts_coors.size(0) == voxel2point_inds.size(-1)
        ops._need_cuda(points, pts_coors, voxel_feats, voxel2point_inds)
        if voxel_feats.requires_grad and torch.is_grad_enabled():
            raise NotImplementedError("Voxel2PointScatterNeck backward is not built yet; run under no_grad()")
        points = points.float().contiguous()
        pts_coors = pts_coors.long().contiguous()
        voxel_feats = voxel_feats.float().contiguous()
        inds = voxel2point_inds.long().contiguous()
        N, Cc = points.shape[0], voxel_feats.shape[1]
        Co = Cc + (3 if self.with_xyz else 0)
        dev = points.device
        out = torch.empty((N, Co), dtype=torch.float32, device=dev)
        mask = torch.empty((N,), dtype=torch.bool, device=dev)
        num_dev = torch.empty((1,), dtype=torch.int32, device=dev)
        num = C.c_int32(0)
        vs = [float(v) for v in (self.voxel_size if self.voxel_size is not None else (1.0, 1.0, 1.0))]
        mn = [float(v) for v in (self.point_cloud_range[:3] if self.point_cloud_range is not None else (0.0, 0.0, 0.0))]
        c = L.ctx(dev)
        L.check(c, L.lib().sstb200_voxel2point(
            c, points.data_ptr(), points.shape[1], pts_coors.data_ptr(), voxel_feats.data_ptr(), voxel_feats.shape[0], Cc,
            inds.data_ptr(), N, float(voxel_padding), L.arr(C.c_float, vs), L.arr(C.c_float, mn), int(bool(self.with_xyz)),
            int(bool(self.normalize_local_xyz)), out.data_ptr(), mask.data_ptr(), num_dev.data_ptr(), C.byref(num)))
        return out[:num.value], mask


def reorder(data, shuffle_inds, keep_inds, padding=-1):
    """single_stage_fsd.py:253-266: pad dropped voxels and undo the shuffle, so that the rows line up with the voxel encoder's
    output again (pure index bookkeeping on device tensors)."""
    n, d = len(shuffle_inds), data.size(1)
    temp = data.new_full((n, d), padding)
    out = data.new_full((n, d), padding)
    temp[keep_inds] = data
    out[shuffle_inds] = temp
    return out
