"""Sync-free frame engine for the FSD segmentation front (VoteSegmentor.extract_feat, mmdet3d/models/detectors/single_stage_fsd.py:228-249):

    points --voxelize--> DynamicScatterVFE --> SimpleSparseUNet (tables + 34 sparse convolutions) --> Voxel2PointScatterNeck

It drives the same libsstb200 kernels as the registered modules, on the same tables and in the same summation order, but through the
device-count entry points (`*_dev`): every row count stays on the device and every buffer is capacity-sized, so a frame is one CUDA
graph with no host sync, no allocation and no torch op.  The plan (levels, tables, convolutions, where each output lands) is built
once on the host by walking the U-Net's module tree (`build_plan`).  The decoder's [bottom || lateral] concatenation is never
copied: the convolution producing each half writes straight into it (row pitches), and reduce_channel + add is one kernel.
"""
import ctypes as C
import math

import numpy as np
import torch
from torch import nn

from . import _lib as L
from . import engine as _engine  # noqa: F401  (prototypes of the graph helpers and sstb200_voxelize_frames)
from .neck_modules import Voxel2PointScatterNeck
from .spconv_modules import PREC, SimpleSparseUNet, SparseBasicBlock, SparseConvolution, SparseSequential, fold_bn, split_h16
from .voxel_modules import DynamicScatterVFE


class Ref:
    """Columns [col, col + ch) of a plan buffer whose rows have pitch `ld` floats; rows live on sparse level `level`."""

    def __init__(self, buf, col, ld, ch, level):
        self.buf, self.col, self.ld, self.ch, self.level = buf, col, ld, ch, level

    def __repr__(self):
        return f"Ref({self.buf}[:, {self.col}:{self.col + self.ch}] ld={self.ld} level={self.level})"


class Plan:
    """Static schedule of one SimpleSparseUNet forward over capacity-sized buffers.

    levels[l]: dict(shape, cap, parent, geom) - level 0 = the input voxels; level l > 0 = output cells of a strided convolution.
    tables[key]: dict(kind 'subm' / 'strided', lin, lout, geom, kv, want_inv) - one per indice_key, shared like indice_dict.
    buffers[name]: (level, width) - fp32 [cap(level), width]; 'in' (the voxel encoder's output) is owned by the caller.
    convs: the convolutions in execution order; steps: ('out_coors', level) / ('table', key) / ('table_inv', key) / ('conv', i) /
    ('merge', dict) in execution order."""

    def __init__(self, batch_size):
        self.B = batch_size
        self.levels, self.tables, self.buffers, self.convs, self.steps = [], {}, {}, [], []
        self.output = None

    def new_buffer(self, level, width, prefix="t"):
        name = f"{prefix}{len(self.buffers)}"
        self.buffers[name] = (level, width)
        return Ref(name, 0, width, width, level)


def _unit(m):
    """make_sparse_convmodule's SparseSequential(conv, BatchNorm1d, ReLU) -> (conv, bn, relu)"""
    mods = list(m._modules.values()) if isinstance(m, SparseSequential) else []
    if (len(mods) != 3 or not isinstance(mods[0], SparseConvolution) or not isinstance(mods[1], nn.BatchNorm1d)
            or not isinstance(mods[2], nn.ReLU)):
        raise NotImplementedError(f"the engine fuses (sparse conv, BatchNorm1d, ReLU) units only, got {m}")
    return mods[0], mods[1], True


def check_backbone(backbone):
    """Host-side validation of a U-Net for the engine (raises before any CUDA call)."""
    if not isinstance(backbone, SimpleSparseUNet):
        raise TypeError(f"backbone must be a SimpleSparseUNet, got {type(backbone).__name__}")
    if backbone.ndim != 3:
        raise NotImplementedError("the engine runs 3-D U-Nets only (ndim == 3)")
    if backbone.keep_coors_dims is not None:
        raise NotImplementedError("keep_coors_dims is not supported by the engine")
    if backbone.return_multiscale_features:
        raise NotImplementedError("return_multiscale_features=True is not supported by the engine")
    if tuple(backbone.order) != ("conv", "norm", "act"):
        raise NotImplementedError(f"order {backbone.order}: the engine fuses conv -> norm -> act")
    if backbone.training or any(m.training for m in backbone.modules()):
        raise ValueError("the engine runs eval-mode modules only (call .eval())")
    for m in backbone.modules():
        if isinstance(m, SparseConvolution):
            if m.conv1x1 or m.transposed:
                raise NotImplementedError("1x1x1 / transposed sparse convolutions are not supported by the engine")
        if isinstance(m, SparseBasicBlock) and not isinstance(m.relu, nn.ReLU):
            raise NotImplementedError("SparseBasicBlock with a non-ReLU activation")


def build_plan(backbone, batch_size, max_voxels):
    """Pure host function: walk conv_input, encoder_layers, then lateral / merge / upsample per decoder level, reusing each layer's
    own geometry (SparseConvolution._geometry) and indice_key sharing.  Capacities: level 0 = min(max_voxels, B * cells); a strided
    level = min(cap_in * prod(ceil(k / s)), B * prod(out_shape)) (the bound sstb200_spconv_out_coors enforces)."""
    check_backbone(backbone)
    B = int(batch_size)
    plan = Plan(B)
    shape0 = [int(s) for s in backbone.sparse_shape]
    plan.levels.append(dict(shape=shape0, cap=max(1, min(int(max_voxels), B * int(np.prod(shape0)))), parent=None, geom=None))
    cin = backbone.in_channels
    plan.buffers["in"] = (0, cin)

    def conv(unit, x, dst=None, residual=None):
        cv, bn, relu = unit
        if cv.in_channels != x.ch:
            raise ValueError(f"channel mismatch: {cv.in_channels} expected, {x.ch} given")
        kv = int(np.prod(cv.kernel_size))
        geom = cv._geometry(plan.levels[x.level]["shape"])
        key = cv.indice_key
        if cv.inverse:
            t = plan.tables.get(key)
            if t is None or t["kind"] != "strided" or t["lout"] != x.level or t["kv"] != kv:
                raise ValueError(f"inverse conv {key}: needs the table of its strided couple conv with the same kernel size")
            if not t["want_inv"]:
                t["want_inv"] = True
                plan.steps.append(("table_inv", key))
            lout, table = t["lin"], (key, "inv")
        elif key is not None and key in plan.tables:
            t = plan.tables[key]
            if t["kv"] != kv or t["lin"] != x.level:
                raise ValueError(f"indice_key {key} reused with a different kernel size / input level")
            lout, table = t["lout"], (key, "nbr")
        else:
            in_shape, out_shape, ks, st, pd = geom
            if cv.subm:
                lout = x.level
            else:
                per_in = int(np.prod([(k + s - 1) // s for k, s in zip(ks, st)]))
                cap = min(plan.levels[x.level]["cap"] * per_in, B * int(np.prod(out_shape)))
                plan.levels.append(dict(shape=[int(v) for v in out_shape], cap=max(1, cap), parent=x.level, geom=geom))
                lout = len(plan.levels) - 1
                plan.steps.append(("out_coors", lout))
            name = key if key is not None else f"_anonymous{len(plan.tables)}"
            plan.tables[name] = dict(kind="subm" if cv.subm else "strided", lin=x.level, lout=lout, geom=geom, kv=kv, want_inv=False)
            plan.steps.append(("table", name))
            table = (name, "nbr")
        if dst is None:
            dst = plan.new_buffer(lout, cv.out_channels)
        elif callable(dst):
            dst = dst(lout, cv.out_channels)
        if dst.level != lout or dst.ch != cv.out_channels or (residual is not None and (residual.level != lout or residual.ch != dst.ch)):
            raise ValueError("the U-Net's hand-over tensors do not line up (levels / channels)")
        plan.convs.append(dict(conv=cv, bn=bn, relu=relu, src=x, dst=dst, res=residual, table=table, kv=kv, level=lout))
        plan.steps.append(("conv", len(plan.convs) - 1))
        return dst

    cats = {}

    def bottom_of(lvl):
        """x_bottom of decoder level lvl lands in the left half of that level's [bottom || lateral] buffer"""
        def place(level, ch):
            lat = getattr(backbone, f"lateral_layer{lvl}").conv2.out_channels
            name = f"cat{lvl}"
            plan.buffers[name] = (level, ch + lat)
            cats[lvl] = (name, ch, lat, level)
            return Ref(name, 0, ch + lat, ch, level)
        return place

    x = Ref("in", 0, cin, cin, 0)
    x = conv(_unit(backbone.conv_input), x)
    stages = list(backbone.encoder_layers)
    n = len(stages)
    enc = []
    for i, stage in enumerate(stages):
        blocks = list(stage)
        for j, blk in enumerate(blocks):
            x = conv(_unit(blk), x, dst=bottom_of(n) if (i == n - 1 and j == len(blocks) - 1) else None)
        enc.append(x)
    for lvl in range(n, 0, -1):
        lat = getattr(backbone, f"lateral_layer{lvl}")
        merge = _unit(getattr(backbone, f"merge_layer{lvl}"))
        up = _unit(getattr(backbone, f"upsample_layer{lvl}"))
        name, cb, cl, level = cats[lvl]
        xl = enc[lvl - 1]
        t = conv((lat.conv1, lat.bn1, True), xl)
        conv((lat.conv2, lat.bn2, True), t, dst=Ref(name, cb, cb + cl, cl, level), residual=xl)
        full = Ref(name, 0, cb + cl, cb + cl, level)
        xm = conv(merge, full)
        if full.ch % xm.ch:
            raise ValueError("reduce_channel: concatenated channels must be a multiple of the merge layer's")
        m = plan.new_buffer(level, xm.ch)
        plan.steps.append(("merge", dict(x_merge=xm, cat=full, out=m)))
        x = conv(up, m, dst=bottom_of(lvl - 1) if lvl > 1 else None)
    plan.output = x
    if x.level != 0:
        raise ValueError("the U-Net's output is not on the input voxels")
    return plan


def _grid_f32(voxel_size, pc_range):
    """(z, y, x) grid of the voxeliser: ceil((max - min) / vs) in float32 (sstb_grid_size, voxelization_cuda.cu:355-357)"""
    f = np.float32
    return [int(np.ceil((f(pc_range[3 + i]) - f(pc_range[i])) / f(voxel_size[i]))) for i in (2, 1, 0)]


class FSDSegEngine:
    """One engine = one stream, one capacity: frames of up to `max_points` points in total, `batch_size` frames per run.
    precision ('bf16' / 'fp32_tc' / 'fp32') selects the sparse convolutions' path; the voxel encoder runs its layer 1 on the tensor
    core with 'bf16' (its own fp32 path otherwise), like DynamicScatterVFE.precision."""

    def __init__(self, voxel_size, point_cloud_range, voxel_encoder: DynamicScatterVFE, backbone: SimpleSparseUNet,
                 decode_neck: Voxel2PointScatterNeck, max_points, batch_size=1, precision="bf16", device="cuda:0", use_graph=True):
        # ---- host-side validation (before any CUDA call) ------------------------------------------------------------------------
        if precision not in PREC:
            raise ValueError(f"precision must be one of {sorted(PREC)}, got {precision!r}")
        if not isinstance(voxel_encoder, DynamicScatterVFE):
            raise TypeError(f"voxel_encoder must be a DynamicScatterVFE, got {type(voxel_encoder).__name__}")
        if not isinstance(decode_neck, Voxel2PointScatterNeck):
            raise TypeError(f"decode_neck must be a Voxel2PointScatterNeck, got {type(decode_neck).__name__}")
        if voxel_encoder.training:
            raise ValueError("the engine runs eval-mode modules only (call .eval())")
        self.vs = [float(v) for v in voxel_size]
        self.rng = [float(v) for v in point_cloud_range]
        if (not np.allclose([voxel_encoder.vx, voxel_encoder.vy, voxel_encoder.vz], self.vs, rtol=0, atol=0)
                or not np.allclose(list(voxel_encoder.point_cloud_range), self.rng, rtol=0, atol=0)):
            raise ValueError("the voxel encoder's voxel_size / point_cloud_range differ from the engine's")
        if voxel_encoder.mode != "max":
            raise NotImplementedError("the fused voxel encoder path of the engine needs mode='max'")
        if voxel_encoder.feat_channels[-1] != backbone.in_channels:
            raise ValueError(f"voxel encoder emits {voxel_encoder.feat_channels[-1]} channels, the U-Net expects {backbone.in_channels}")
        self.B, self.cap = int(batch_size), int(max_points)
        if self.B < 1 or self.cap < 1:
            raise ValueError("batch_size and max_points must be >= 1")
        grid = _grid_f32(self.vs, self.rng)
        if any(g > s for g, s in zip(grid, backbone.sparse_shape)):
            raise ValueError(f"voxel grid (z,y,x) {grid} does not fit the U-Net's sparse_shape {list(backbone.sparse_shape)}")
        self.vfe, self.bb, self.neck = voxel_encoder, backbone, decode_neck
        self.precision = precision
        self.vfe_precision = "bf16" if precision == "bf16" else "fp32"
        saved = voxel_encoder.precision
        voxel_encoder.precision = self.vfe_precision
        try:
            self.vfe_cfg = voxel_encoder._cfg(self.B)   # raises on VFE configurations the fused path does not build
        finally:
            voxel_encoder.precision = saved
        self.plan = build_plan(backbone, self.B, self.cap)
        self.F = voxel_encoder.raw_in_channels
        self.use_graph = use_graph

        # ---- device buffers (capacity-sized, allocated once) ----------------------------------------------------------------------
        self.dev = torch.device(device)
        dev, cap, plan = self.dev, self.cap, self.plan
        f32, i32 = dict(dtype=torch.float32, device=dev), dict(dtype=torch.int32, device=dev)
        self._owned = []

        def own(t):
            self._owned.append(t)
            return t
        self.points = own(torch.zeros((cap, self.F), **f32))
        self.offsets = own(torch.zeros((self.B + 1,), **i32))
        self.coors4 = own(torch.empty((cap, 4), **i32))
        self.vf = own(torch.empty((cap, backbone.in_channels), **f32))
        self.vc = own(torch.empty((cap, 4), **i32))
        self.inv = own(torch.empty((cap,), **i32))
        nl = len(plan.levels)
        self.counts = own(torch.zeros((nl + 1,), **i32))   # [0, nl): rows per level (level 0 = voxels), [nl]: kept points
        self.level_coors = [self.vc] + [own(torch.empty((lv["cap"], 4), **i32)) for lv in plan.levels[1:]]
        self.bufs = {"in": self.vf}
        for name, (lvl, width) in plan.buffers.items():
            if name != "in":
                self.bufs[name] = own(torch.empty((plan.levels[lvl]["cap"], width), **f32))
        self.nbr, self.nbr_inv = {}, {}
        for key, t in plan.tables.items():
            self.nbr[key] = own(torch.empty((plan.levels[t["lout"]]["cap"], t["kv"]), **i32))
            if t["want_inv"]:
                self.nbr_inv[key] = own(torch.empty((plan.levels[t["lin"]]["cap"], t["kv"]), **i32))
        C_out = plan.output.ch
        self.pts_feats = own(torch.empty((cap, C_out + (3 if decode_neck.with_xyz else 0)), **f32))
        self.pts_mask = own(torch.zeros((cap,), dtype=torch.bool, device=dev))
        self._weights = []
        for cv in plan.convs:
            conv, kv = cv["conv"], cv["kv"]
            w = {"w32": None, "h16": None}
            if precision == "fp32":
                w["w32"] = own(torch.empty((kv, conv.in_channels, conv.out_channels), **f32))
            else:
                w["h16"] = own(torch.empty(((1 if precision == "bf16" else 2) * kv, conv.out_channels, conv.in_channels),
                                           dtype=torch.float16, device=dev))
            w["scale"] = own(torch.empty((conv.out_channels,), **f32))
            w["shift"] = own(torch.empty((conv.out_channels,), **f32))
            self._weights.append(w)
        self.refresh_weights()
        self.buffer_bytes = sum(t.numel() * t.element_size() for t in self._owned)
        self._vs_arr, self._rng_arr = L.arr(C.c_float, self.vs), L.arr(C.c_float, self.rng)
        nvs = decode_neck.voxel_size if decode_neck.voxel_size is not None else (1.0, 1.0, 1.0)
        nmn = decode_neck.point_cloud_range[:3] if decode_neck.point_cloud_range is not None else (0.0, 0.0, 0.0)
        self._neck_vs, self._neck_mn = L.arr(C.c_float, [float(v) for v in nvs]), L.arr(C.c_float, [float(v) for v in nmn])

        self.stream = torch.cuda.Stream(device=dev)
        self.graph = None
        self.launches_per_frame = self.other_nodes_per_frame = None
        with torch.cuda.stream(self.stream):
            self._enqueue()           # warm-up: grows the arena, sets kernel attributes
            self._enqueue()
        self.stream.synchronize()
        if use_graph:
            with torch.cuda.stream(self.stream):
                lib, c = L.lib(), L.ctx(self.dev)
                L.check(c, lib.sstb200_graph_begin(c))
                try:
                    self._enqueue()
                finally:
                    ex, nk, no = C.c_void_p(), C.c_int32(0), C.c_int32(0)
                    L.check(c, lib.sstb200_graph_end(c, C.byref(ex), C.byref(nk), C.byref(no)))
                self.graph = ex
                self.launches_per_frame = nk.value
                self.other_nodes_per_frame = no.value
            self.stream.synchronize()

    def refresh_weights(self):
        """Call after the modules' parameters / BatchNorm statistics changed (load_state_dict, optimiser step): the folded BN
        scale / shift and the weight copies (fp32, or the fp16 operands of the tensor-core paths) are recomputed INTO the buffers
        the graph points at.  The voxel encoder folds its BatchNorm inside the frame and reads its parameters in place."""
        with torch.no_grad():
            for cv, w in zip(self.plan.convs, self._weights):
                conv, kv = cv["conv"], cv["kv"]
                weight = conv.weight.detach().reshape(kv, conv.in_channels, conv.out_channels)
                if w["w32"] is not None:
                    w["w32"].copy_(weight)
                else:
                    hi, lo = split_h16(weight)
                    w["h16"].copy_(hi if self.precision == "bf16" else torch.cat([hi, lo], 0))
                scale, shift = fold_bn(cv["bn"], conv.bias)
                w["scale"].copy_(scale)
                w["shift"].copy_(shift)

    # ---- everything below is stream-ordered and sync-free ----------------------------------------------------------------------
    def _cnt(self, i):
        return self.counts.data_ptr() + 4 * i

    def _ptr(self, ref):
        return self.bufs[ref.buf].data_ptr() + 4 * ref.col

    def _enqueue(self):
        lib, c = L.lib(), L.ctx(self.dev)
        plan, B = self.plan, self.B
        L.check(c, lib.sstb200_voxelize_frames(c, self.points.data_ptr(), self.cap, self.F, self.offsets.data_ptr(), B, self._vs_arr,
                                               self._rng_arr, self.coors4.data_ptr()))
        L.check(c, lib.sstb200_dynamic_scatter_vfe_forward_i32(c, C.byref(self.vfe_cfg), self.points.data_ptr(), self.coors4.data_ptr(),
                                                               self.cap, self.vf.data_ptr(), self.vc.data_ptr(), self.inv.data_ptr(),
                                                               self._cnt(0)))
        caps = [lv["cap"] for lv in plan.levels]
        i3 = lambda v: L.arr(C.c_int32, [int(x) for x in v])
        prec = PREC[self.precision]
        for kind, arg in plan.steps:
            if kind == "out_coors":
                lv = plan.levels[arg]
                p = lv["parent"]
                L.check(c, lib.sstb200_spconv_out_coors_dev(c, self.level_coors[p].data_ptr(), caps[p], self._cnt(p), B, *map(i3, lv["geom"]),
                                                            self.level_coors[arg].data_ptr(), caps[arg], self._cnt(arg)))
            elif kind in ("table", "table_inv"):
                t = plan.tables[arg]
                li, lo = t["lin"], t["lout"]
                nbr = self.nbr[arg].data_ptr() if kind == "table" else None
                inv = self.nbr_inv[arg].data_ptr() if kind == "table_inv" else None
                L.check(c, lib.sstb200_spconv_table_dev(c, self.level_coors[li].data_ptr(), caps[li], self._cnt(li),
                                                        self.level_coors[lo].data_ptr(), caps[lo], self._cnt(lo), B, *map(i3, t["geom"]),
                                                        nbr, inv))
            elif kind == "conv":
                cv, w = plan.convs[arg], self._weights[arg]
                conv = cv["conv"]
                key, which = cv["table"]
                nbr = self.nbr[key] if which == "nbr" else self.nbr_inv[key]
                res = cv["res"]
                lvl = cv["level"]
                L.check(c, lib.sstb200_spconv_forward_dev(
                    c, self._ptr(cv["src"]), cv["src"].ld, conv.in_channels, nbr.data_ptr(), caps[lvl], self._cnt(lvl), cv["kv"],
                    L.ptr(w["w32"]), L.ptr(w["h16"]), conv.out_channels, w["scale"].data_ptr(), w["shift"].data_ptr(),
                    self._ptr(res) if res is not None else None, res.ld if res is not None else 0, int(cv["relu"]), prec,
                    self._ptr(cv["dst"]), cv["dst"].ld))
            else:
                xm, cat, out = arg["x_merge"], arg["cat"], arg["out"]
                L.check(c, lib.sstb200_spconv_decoder_merge(c, self._ptr(xm), self._ptr(cat), xm.ch, cat.ch, caps[xm.level],
                                                            self._cnt(xm.level), self._ptr(out)))
        out = plan.output
        L.check(c, lib.sstb200_voxel2point_dev(c, self.points.data_ptr(), self.F, self.coors4.data_ptr(), self._ptr(out), self._cnt(0),
                                               out.ch, self.inv.data_ptr(), self.cap, -1.0, self._neck_vs, self._neck_mn,
                                               int(bool(self.neck.with_xyz)), int(bool(self.neck.normalize_local_xyz)),
                                               self.pts_feats.data_ptr(), self.pts_mask.data_ptr(), self._cnt(len(plan.levels))))

    def load_frames_device(self, points_dev, offsets_dev):
        """points_dev [P, F] fp32 (frames back to back) and offsets_dev int32 [B + 1] (row ranges of the frames), both on the device.
        Stream-ordered copy into the engine's input buffer (no sync).  Rows past offsets[B] are ignored."""
        n = points_dev.shape[0]
        if n > self.cap or offsets_dev.numel() != self.B + 1 or points_dev.shape[1] != self.F:
            raise ValueError(f"at most {self.cap} points of {self.F} features and {self.B + 1} offsets expected")
        self.stream.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(self.stream):
            self.points[:n].copy_(points_dev, non_blocking=True)
            self.offsets.copy_(offsets_dev, non_blocking=True)

    def run(self):
        """Enqueue one forward over the resident frames (graph replay) and return the engine's PERSISTENT output buffers, valid until
        the next run() on this engine (a consumer on another stream orders itself after `engine.stream`):
          pts_feats [cap, C(+3)]   rows [0, num_pts) = the neck's output (kept points, input order)
          pts_mask  [cap] bool     the neck's mask per point row (rows past the last frame: False)
          num_pts   [1] int32      kept points (device)
          voxel_feats [cap, C], voxel_coors [cap, 4] int32 (b,z,y,x), num_voxels [1] int32 (device): the U-Net's output
          unq_inv   [cap] int32    voxel row of every point (-1: no voxel)"""
        with torch.cuda.stream(self.stream):
            if self.graph is not None:
                c = L.ctx(self.dev)
                L.check(c, L.lib().sstb200_graph_launch(c, self.graph))
            else:
                self._enqueue()
        nl = len(self.plan.levels)
        return dict(pts_feats=self.pts_feats, pts_mask=self.pts_mask, num_pts=self.counts[nl:nl + 1],
                    voxel_feats=self.bufs[self.plan.output.buf], voxel_coors=self.vc, num_voxels=self.counts[0:1], unq_inv=self.inv)

    def __del__(self):
        g = getattr(self, "graph", None)
        if g is not None:
            try:
                L.lib().sstb200_graph_destroy(L.ctx(self.dev), g)
            except Exception:
                pass


def module_front(voxel_encoder, backbone, decode_neck, frames, voxel_size, point_cloud_range):
    """The same front through the registered modules (VoteSegmentor.voxelize + extract_feat): frames = list of [n_i, F] device
    tensors.  Returns (pts_feats [kept, C(+3)], pts_mask, voxel_feats, voxel_coors int64, unq_inv int64).  Syncs like the modules do."""
    from . import ops
    coors = []
    for b, pts in enumerate(frames):
        co = torch.empty((pts.shape[0], 3), dtype=torch.int32, device=pts.device)
        ops.dynamic_voxelize(pts.contiguous(), co, voxel_size, point_cloud_range)
        coors.append(torch.nn.functional.pad(co, (1, 0), value=b))
    points, coors = torch.cat(frames), torch.cat(coors).long()
    vf, vc, inv = voxel_encoder(points, coors, return_inv=True)
    x = backbone(dict(voxel_feats=vf, voxel_coors=vc))[0]
    out, mask = decode_neck(points, coors, x["voxel_feats"], inv, -1)
    return out, mask, x["voxel_feats"], vc, inv
