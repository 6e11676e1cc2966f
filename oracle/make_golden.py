"""TEST INFRASTRUCTURE - generates tests/golden/*.npz by running the UNMODIFIED reference Python
(/root/reference, through oracle/ref_shim.py) on small seeded inputs.  Run in the build container only:

    python -m oracle.make_golden

Each fixture stores inputs, the reference module's state_dict and the reference outputs, so that
tests/test_oracle_golden.py can pin oracle/sst_oracle.py against them anywhere (the GPU box has no
/root/reference).  DynamicScatter inside DynamicVFE uses the restatement (the reference has no CPU
dynamic_point_to_voxel, voxelization.h:96-108); that op is pinned separately (restated reference test +
reference CUDA build in oracle/_ref on GPU boxes).
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim, sst_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
VS = (0.32, 0.32, 6)
RNG = [-74.88, -74.88, -2, 74.88, 74.88, 4]
DROP_TRAIN = {0: {'max_tokens': 30, 'drop_range': (0, 30)}, 1: {'max_tokens': 60, 'drop_range': (30, 60)},
              2: {'max_tokens': 100, 'drop_range': (60, 100000)}}
DROP_TEST = {0: {'max_tokens': 30, 'drop_range': (0, 30)}, 1: {'max_tokens': 60, 'drop_range': (30, 60)},
             2: {'max_tokens': 100, 'drop_range': (60, 100)}, 3: {'max_tokens': 144, 'drop_range': (100, 100000)}}


def _rand_norm(m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n_, p in m.named_parameters():
            if p.dim() == 1:
                p.copy_(torch.randn(p.shape, generator=g) * 0.2 + (1.0 if "norm" in n_ and "weight" in n_ else 0.0))
            if n_.endswith("tau"):
                p.copy_(torch.rand(p.shape, generator=g) * 0.5 + 0.05)
        for n_, b in m.named_buffers():
            if "running_mean" in n_:
                b.copy_(torch.randn(b.shape, generator=g) * 0.3)
            if "running_var" in n_:
                b.copy_(torch.rand(b.shape, generator=g) + 0.5)


def _sd(m, prefix):
    return {prefix + k: v.detach().numpy() for k, v in m.state_dict().items() if v.dtype.is_floating_point}


def sst_fixture(R):
    torch.manual_seed(0)
    pts = torch.cat([O.synth_frame(5, 2500), O.synth_frame(6, 1500)])
    pts[:, :2] *= 0.2  # dense enough to populate every drop level incl. > 100 tokens
    c3 = O.dynamic_voxelize(pts, VS, RNG)
    coors = torch.cat([torch.nn.functional.pad(c3[:2500], (1, 0), value=0), torch.nn.functional.pad(c3[2500:], (1, 0), value=1)])
    vfe = R.DynamicVFE(in_channels=3, feat_channels=[16, 32], with_cluster_center=True, with_voxel_center=True, voxel_size=VS,
                       point_cloud_range=RNG, norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01)).eval()
    _rand_norm(vfe, 1)
    out = {"points": pts.numpy(), "coors": coors.numpy()}
    with torch.no_grad():
        vf, vc = vfe(pts, coors)
        out.update(vfe_feats=vf.numpy(), vfe_coors=vc.numpy(), **_sd(vfe, "vfe."))
        for tag, drop, train in (("eval", (DROP_TRAIN, DROP_TEST), False), ("train", (DROP_TRAIN, DROP_TEST), True)):
            il = R.SSTInputLayerV2(drop, (12, 12, 1), (468, 468, 1), shuffle_voxels=False, debug=True)
            il.train(train)
            info = il(vf, vc, 2)
            for i in range(2):
                out[f"{tag}.batch_win_inds_shift{i}"] = info[f"batch_win_inds_shift{i}"].numpy()
                out[f"{tag}.coors_in_win_shift{i}"] = info[f"coors_in_win_shift{i}"].numpy()
                out[f"{tag}.drop_level_shift{i}"] = info[f"voxel_drop_level_shift{i}"].numpy()
                for dl, v in info[f"flat2win_inds_shift{i}"].items():
                    if isinstance(dl, str):
                        continue
                    # the reference's inner order is implementation defined (sst_ops.py:203): the shim uses the
                    # canonical stable order, so these are comparable element-wise
                    out[f"{tag}.f2w{i}.{dl}.inds"] = v[0].numpy()
                    out[f"{tag}.f2w{i}.{dl}.pos"] = v[1][0].numpy()
                    out[f"{tag}.pos{i}.{dl}"] = info[f"pos_dict_shift{i}"][dl].numpy()
                    out[f"{tag}.mask{i}.{dl}"] = info[f"key_mask_shift{i}"][dl].numpy()
            out[f"{tag}.keep"] = info["voxel_keep_inds"].numpy()
            if tag == "eval":
                for name, lc in (("plain", {}), ("cosine", dict(cosine=True, tau_min=0.01)), ("prebn", dict(post_norm=False, use_bn=True))):
                    torch.manual_seed(3)
                    bb = R.SSTv2(d_model=[32] * 2, nhead=[4] * 2, num_blocks=2, dim_feedforward=[64] * 2, output_shape=[468, 468],
                                 num_attached_conv=0, to_bev=False, layer_cfg=lc).eval()
                    _rand_norm(bb, 4)
                    y = bb(info)[0]["voxel_feats"]
                    out[f"sst.{name}.out"] = y.numpy()
                    out.update(_sd(bb, f"sst.{name}.w."))
    np.savez_compressed(os.path.join(OUT, "sst_small.npz"), **out)
    print("sst_small", len(out), "arrays", vf.shape)


def vfe_fixture(R):
    """DynamicVFE alone at a channel pair the fused CUDA kernels are instantiated for (multiples of 32)."""
    torch.manual_seed(0)
    pts = torch.cat([O.synth_frame(25, 3000), O.synth_frame(26, 2000)])
    pts[:, :2] *= 0.3
    c3 = O.dynamic_voxelize(pts, VS, RNG)
    coors = torch.cat([torch.nn.functional.pad(c3[:3000], (1, 0), value=0), torch.nn.functional.pad(c3[3000:], (1, 0), value=1)])
    vfe = R.DynamicVFE(in_channels=3, feat_channels=[32, 64], with_cluster_center=True, with_voxel_center=True, voxel_size=VS,
                       point_cloud_range=RNG, norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01)).eval()
    _rand_norm(vfe, 31)
    with torch.no_grad():
        vf, vc = vfe(pts, coors)
    np.savez_compressed(os.path.join(OUT, "vfe_small.npz"), points=pts.numpy(), coors=coors.numpy(), feats=vf.numpy(), vcoors=vc.numpy(),
                        **_sd(vfe, "w."))
    print("vfe_small", vf.shape)


def sst_v1_fixture(R):
    """configs/sst names: SSTInputLayer (v1) + SSTv1 through the unmodified reference classes.  The dense BEV output is stored
    as its rows at the occupied cells plus its total absolute sum (everything else must be zero)."""
    torch.manual_seed(0)
    pts = torch.cat([O.synth_frame(15, 2500), O.synth_frame(16, 1500)])
    pts[:, :2] *= 0.2
    c3 = O.dynamic_voxelize(pts, VS, RNG)
    c4 = torch.cat([torch.nn.functional.pad(c3[:2500], (1, 0), value=0), torch.nn.functional.pad(c3[2500:], (1, 0), value=1)])
    vc = torch.unique(c4, dim=0).long()
    g = torch.Generator().manual_seed(21)
    vf = torch.randn(vc.shape[0], 32, generator=g)
    il = R.SSTInputLayer(drop_info=(DROP_TRAIN, DROP_TEST), shifts_list=[(0, 0), (6, 6)], window_shape=(12, 12), point_cloud_range=RNG,
                         voxel_size=VS, shuffle_voxels=False, debug=True).eval()
    bb = R.SSTv1(d_model=[32] * 2, nhead=[4] * 2, num_blocks=2, dim_feedforward=[64] * 2, output_shape=[468, 468], num_attached_conv=0,
                 debug=True, drop_info=(DROP_TRAIN, DROP_TEST), pos_temperature=10000, normalize_pos=False, window_shape=(12, 12)).eval()
    _rand_norm(bb, 14)
    with torch.no_grad():
        feat, f2w, info = il(vf, vc)
        bev = bb((feat, f2w, info))[0]
    co = info["coors"]
    rows = bev[co[:, 0], :, co[:, 2], co[:, 3]]
    out = dict(voxel_feats=vf.numpy(), voxel_coors=vc.numpy(), keep=info["voxel_keep_inds"].numpy(), coors=co.numpy(),
               bev_rows=rows.numpy(), bev_abs_sum=np.array(bev.abs().double().sum().item()), bev_shape=np.array(bev.shape),
               **{f"bwi{i}": info[f"batch_win_inds_shift{i}"].numpy() for i in range(2)},
               **{f"ciw{i}": info[f"coors_in_win_shift{i}"].numpy() for i in range(2)},
               **{f"lvl{i}": info[f"voxel_drop_level_shift{i}"].numpy() for i in range(2)}, **_sd(bb, "w."))
    np.savez_compressed(os.path.join(OUT, "sst_v1_small.npz"), **out)
    print("sst_v1_small", rows.shape, float(out["bev_abs_sum"]))


def sir_fixture(R):
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(11)
    N, G = 3000, 23
    points = torch.cat([torch.randn(N, 3, generator=g) * 10, torch.rand(N, 2, generator=g)], 1)
    feats = torch.randn(N, 27, generator=g)
    gid = torch.randint(0, G, (N,), generator=g)
    coors = torch.stack([gid % 3, gid % 2, gid], 1)
    fcl = torch.randn(N, 3, generator=g) * 2
    sir = R.SIR(num_blocks=3, in_channels=[32, 37, 37], feat_channels=[[32, 32]] * 3, rel_mlp_hidden_dims=[[16, 32] for _ in range(3)],
                norm_cfg=dict(type='LN', eps=1e-3), mode='max', xyz_normalizer=[20, 20, 4], act='gelu', unique_once=True).eval()
    _rand_norm(sir, 2)
    with torch.no_grad():
        a, b, c = sir(points, feats, coors, fcl)
    out = dict(points=points.numpy(), feats=feats.numpy(), coors=coors.numpy(), f_cluster=fcl.numpy(), out_point=a.numpy(),
               out_group=b.numpy(), out_coors=c.numpy(), **_sd(sir, "w."))
    np.savez_compressed(os.path.join(OUT, "sir_small.npz"), **out)
    print("sir_small", a.shape, b.shape)


def dsvfe_fixture(R):
    torch.manual_seed(0)
    vs, rng = (0.25, 0.25, 0.2), [-80, -80, -2, 80, 80, 4]
    pts = torch.cat([O.synth_frame(3, 3000), torch.rand(3000, 2)], 1)
    co = torch.nn.functional.pad(O.dynamic_voxelize(pts, vs, rng), (1, 0), value=0).long()
    co[1500:, 0] = 1
    m = R.DynamicScatterVFE(in_channels=5, feat_channels=[32, 32], with_cluster_center=True, with_voxel_center=True, voxel_size=vs,
                            point_cloud_range=rng, norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01), unique_once=True,
                            rel_dist_scaler=10.0).eval()
    _rand_norm(m, 7)
    with torch.no_grad():
        f, c, inv = m(pts, co, return_inv=True)
    np.savez_compressed(os.path.join(OUT, "dsvfe_small.npz"), points=pts.numpy(), coors=co.numpy(), feats=f.numpy(),
                        vcoors=c.numpy(), inv=inv.numpy(), **_sd(m, "w."))
    print("dsvfe_small", f.shape)


FSDV2 = dict(vs=(0.5, 0.5, 0.5), rng=[-40, -40, -2, 40, 40, 4], target=[12, 160, 160], C=16,
             vfe=dict(in_channels=19, feat_channels=[32, 32], with_cluster_center=True, with_voxel_center=True, rel_dist_scaler=10.0),
             ms_hiddens=[[24, 32], [16, 32], [16, 32]], ms_shapes=[[12, 160, 160], [6, 80, 80], [3, 40, 40]])


def fsdv2_inputs(seed=11, n_ori=4000, n_vir=1500, batch=2):
    """Synthetic segmentor outputs for the FSDv2 front: real points with features, sampled foreground points with centre votes."""
    g = torch.Generator().manual_seed(seed)
    C, rng = FSDV2["C"], FSDV2["rng"]
    lo, hi = torch.tensor(rng[:3], dtype=torch.float32), torch.tensor(rng[3:], dtype=torch.float32)

    def pts(n):
        return torch.cat([lo + (hi - lo) * torch.rand(n, 3, generator=g) * 0.98 + 0.01, torch.rand(n, 2, generator=g)], 1)
    origin = dict(seg_points=pts(n_ori), seg_feats=torch.randn(n_ori, C + 3, generator=g), batch_idx=torch.randint(0, batch, (n_ori,), generator=g))
    sp = pts(n_vir)
    centers = sp[:, :3] + torch.randn(n_vir, 3, generator=g) * 1.5   # votes; a few leave the range and get clipped
    centers[::97] += 100.0
    sampled = dict(seg_points=sp, center_preds=centers, seg_logits=torch.randn(n_vir, 3, generator=g), seg_feats=torch.randn(n_vir, C, generator=g),
                   batch_idx=torch.randint(0, batch, (n_vir,), generator=g))
    levels = []
    for (fin, _), shp in zip(FSDV2["ms_hiddens"], FSDV2["ms_shapes"]):
        n = 600
        cells = torch.randperm(batch * shp[0] * shp[1] * shp[2], generator=g)[:n]
        b, r = cells // (shp[0] * shp[1] * shp[2]), cells % (shp[0] * shp[1] * shp[2])
        idx = torch.stack([b, r // (shp[1] * shp[2]), (r // shp[2]) % shp[1], r % shp[2]], 1).int()
        levels.append((torch.randn(n, fin, generator=g), idx, list(shp)))
    return sampled, origin, levels


def fsdv2_front_fixture(R):
    """SingleStageFSDV2.extract_feat / multiscale_fusion / voxelize_with_batch_idx / clip_points / ms_coors_proj run from the
    reference source itself (ref_shim.reference_methods) on a stand-in `self` that carries the reference's own sub-modules; the
    backbone (sparse-conv mixer, SURVEY 8f next-1) is an identity that records what it is given."""
    import types
    torch.manual_seed(0)
    fns = ref_shim.reference_methods("mmdet3d/models/detectors/single_stage_fsd_v2.py", "SingleStageFSDV2",
                                     ["extract_feat", "multiscale_fusion", "voxelize_with_batch_idx", "clip_points", "ms_coors_proj"])
    norm = dict(type='naiveSyncBN1d', eps=1e-5, momentum=0.01)
    C = FSDV2["C"]

    class Stand(torch.nn.Module):
        pass
    for with_ms, with_mixer in ((False, False), (True, False), (True, True)):
        self = Stand()
        self.baseline_mode, self.zero_virtual_feature, self.only_virtual, self.as_rpn = False, False, False, False
        self.virtual_voxel_size, self.point_cloud_range = FSDV2["vs"], FSDV2["rng"]
        self.virtual_proj = R.sst_ops.build_mlp(C + 3 + 3 + 2, [16, 16], norm)
        self.ori_proj = R.sst_ops.build_mlp(C + 3, [16, 16], norm)
        self.voxel_encoder = R.DynamicScatterVFE(voxel_size=FSDV2["vs"], point_cloud_range=FSDV2["rng"],
                                                 norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01), unique_once=True, **FSDV2["vfe"])
        self.multiscale_cfg = dict(multiscale_levels=[0, 1, 2], projector_hiddens=FSDV2["ms_hiddens"], fusion_mode='avg',
                                   target_sparse_shape=FSDV2["target"], norm_cfg=norm) if with_ms else None
        if with_ms:
            self.ms_projectors = torch.nn.ModuleList([R.sst_ops.build_mlp(h[0], h[1:], norm) for h in FSDV2["ms_hiddens"]])
        self.eval()
        _rand_norm(self, 21)
        seen = {}

        def backbone(vf, vc, bs):
            seen.update(vf=vf.clone(), vc=vc.clone(), bs=bs)
            return vf, vc, None
        self.backbone = backbone
        if with_mixer:   # the reference's own VirtualVoxelMixer over its vendored spconv v1 (SURVEY 8f next-1): config 5 end to end
            from oracle import spconv_oracle as SO_
            torch.manual_seed(5)
            mixer = ref_shim.load_spconv().VirtualVoxelMixer(**SO_.FSDV2_MIXER).eval()
            _rand_bn(mixer, 33, wmul=5.0)   # the fused voxels are almost isolated (7k in 600k cells): little neighbour signal

            def backbone_mixer(vf, vc, bs):
                seen.update(vf=vf.clone(), vc=vc.clone(), bs=bs)
                return mixer(vf, vc, bs)
            self.backbone = backbone_mixer
        for k, f in fns.items():
            setattr(self, k, types.MethodType(f, self))
        sampled, origin, levels = fsdv2_inputs()
        ms = [types.SimpleNamespace(features=f, indices=i, spatial_shape=s) for f, i, s in levels] if with_ms else None
        with torch.no_grad():
            out = self.extract_feat({k: v.clone() for k, v in sampled.items()}, {k: v.clone() for k, v in origin.items()}, None, ms)
            coors = self.voxelize_with_batch_idx(torch.cat([origin["seg_points"][:, :3], self.clip_points(sampled["center_preds"].clone(), FSDV2["rng"])]),
                                                 torch.cat([origin["batch_idx"], sampled["batch_idx"]]))
        tag = "mixer" if with_mixer else ("ms" if with_ms else "plain")
        extra = {"mix." + k: v.numpy() for k, v in mixer.state_dict().items()} if with_mixer else {}
        np.savez_compressed(os.path.join(OUT, f"fsdv2_front_{tag}.npz"), **extra, coors=coors.numpy(), backbone_feats=seen["vf"].numpy(),
                            backbone_coors=seen["vc"].numpy(), batch_size=np.array(seen["bs"]), virtual_feats=out["virtual_feats"].numpy(),
                            virtual_coors=out["virtual_coors"].numpy(), virtual_centers=out["virtual_centers"].numpy(),
                            **{f"sampled.{k}": v.numpy() for k, v in sampled.items()}, **{f"origin.{k}": v.numpy() for k, v in origin.items()},
                            **{f"ms{i}.{n}": (np.array(a) if n == "shape" else a.numpy()) for i, lv in enumerate(levels)
                               for n, a in zip(("features", "indices", "shape"), lv)},
                            **_sd(self, "w."))
        print("fsdv2_front", tag, seen["vf"].shape, out["virtual_feats"].shape)


def scatter_fixture():
    """Seeded restatement of tests/test_models/test_voxel_encoder/test_dynamic_scatter.py:56-84: expected values are the
    brute-force per-voxel loop the reference test itself uses as ground truth."""
    g = torch.Generator().manual_seed(0)
    feats = torch.rand(20000, 3, generator=g) * 100 - 50
    coors = torch.randint(-1, 20, (20000, 3), generator=g, dtype=torch.int32)
    ref_coors = coors.unique(dim=0, sorted=True)
    ref_coors = ref_coors[ref_coors.min(dim=-1).values >= 0]
    mean = torch.stack([feats[coors.eq(rc).all(dim=-1)].mean(dim=0) for rc in ref_coors])
    mx = torch.stack([feats[coors.eq(rc).all(dim=-1)].max(dim=0).values for rc in ref_coors])
    np.savez_compressed(os.path.join(OUT, "dynamic_scatter.npz"), feats=feats.numpy(), coors=coors.numpy(),
                        ref_coors=ref_coors.numpy(), ref_mean=mean.numpy(), ref_max=mx.numpy())
    print("dynamic_scatter", ref_coors.shape)


def neck_fixture(R):
    """Voxel2PointScatterNeck (necks/voxel2point_neck.py:28-62) through the unmodified reference class."""
    g = torch.Generator().manual_seed(5)
    N, M, C = 3000, 400, 16
    pts = O.synth_frame(3, N, extra_dims=1)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0).long()
    vf = torch.randn(M, C, generator=g)
    vf[::7] = -1.0
    inds = torch.randint(0, M, (N,), generator=g)
    out = {"points": pts.numpy(), "coors": coors.numpy(), "voxel_feats": vf.numpy(), "inds": inds.numpy()}
    for name, (xyz, norm) in {"xyz": (True, False), "xyznorm": (True, True), "noxyz": (False, False)}.items():
        neck = R.Voxel2PointScatterNeck(point_cloud_range=RNG, voxel_size=VS, with_xyz=xyz, normalize_local_xyz=norm).eval()
        r, m = neck(pts, coors, vf, inds)
        out[f"out_{name}"], out[f"mask_{name}"] = r.numpy(), m.numpy()
    np.savez_compressed(os.path.join(OUT, "neck_small.npz"), **out)
    print("neck", out["out_xyz"].shape)


def hard_voxelize_fixture():
    """voxel_layer.hard_voxelize through the reference's own C++ (oracle/_ref, built from voxelization_cpu.cpp unmodified)."""
    from oracle import build_ref
    ref = build_ref.load_module() or (build_ref.build() and build_ref.load_module())
    pts = O.synth_frame(41, 6000, extra_dims=1)
    pts[::13, 0] += 500.0
    out = {"points": pts.numpy()}
    for name, (mp, mv) in {"roomy": (16, 6000), "capped": (3, 150)}.items():
        voxels = torch.zeros((mv, mp, 4))
        coors = torch.zeros((mv, 3), dtype=torch.int32)
        npts = torch.zeros((mv,), dtype=torch.int32)
        n = ref.hard_voxelize(pts, voxels, coors, npts, list(VS), list(RNG), mp, mv, 3)
        out[f"voxels_{name}"], out[f"coors_{name}"], out[f"npts_{name}"] = voxels[:n].numpy(), coors[:n].numpy(), npts[:n].numpy()
        out[f"cfg_{name}"] = np.array([mp, mv])
    np.savez_compressed(os.path.join(OUT, "hard_voxelize.npz"), **out)
    print("hard_voxelize", out["voxels_roomy"].shape, out["voxels_capped"].shape)


def _rand_bn(m, seed, wmul=2.0):
    """BatchNorm statistics / affine parameters that keep the signal alive through ~25 layers (weights in [0.5, 1.5])"""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.running_mean.copy_(torch.randn(mod.num_features, generator=g) * 0.2)
                mod.running_var.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
                mod.weight.copy_(torch.rand(mod.num_features, generator=g) + 0.5)
                mod.bias.copy_(torch.randn(mod.num_features, generator=g) * 0.2)
        for p in m.parameters():
            if p.dim() == 5:   # spconv's default init (kaiming_uniform, a = sqrt 5) shrinks the signal ~3x per layer
                p.mul_(wmul)


def _sort_rows(feats, coors):
    c = coors.long()
    order = torch.argsort(((c[:, 0] * 4096 + c[:, 1]) * 4096 + c[:, 2]) * 4096 + c[:, 3])
    return feats[order], coors[order]


def spconv_fixture():
    """SURVEY 8f next-1: the reference's vendored spconv v1 layers (mmdet3d/ops/spconv/conv.py over oracle/_ref/sparse_conv_ext_ref*.so,
    built from its own C++ sources) and its SimpleSparseUNet / VirtualVoxelMixer classes (middle_encoders/sparse_unet.py), eval mode.
    Rows of strided-conv outputs are stored sorted by coordinate (spconv's own order is hash-insertion order)."""
    from oracle import spconv_oracle as SO
    S = ref_shim.load_spconv()
    out = {}
    feats, coors = SO.synth_sparse(11, 2, (9, 20, 24), 400, 8)
    out["l_feats"], out["l_coors"], out["l_shape"] = feats.numpy(), coors.numpy(), np.array([9, 20, 24])
    torch.manual_seed(21)
    for name, (ks, st, pd) in {"a": (3, 2, 1), "b": (3, 2, (0, 1, 1)), "c": ((3, 1, 1), (2, 1, 1), 0)}.items():
        conv = S.SparseConv3d(8, 12, ks, stride=st, padding=pd, bias=False, indice_key="k")
        inv = S.SparseInverseConv3d(12, 8, ks, indice_key="k", bias=False)
        with torch.no_grad():
            y = conv(S.SparseConvTensor(feats, coors, [9, 20, 24], 2))
            z = inv(y)
        yf, yc = _sort_rows(y.features, y.indices)
        out[f"conv_{name}_cfg"] = np.array(list(conv.kernel_size) + list(conv.stride) + list(conv.padding))
        out[f"conv_{name}_w"], out[f"conv_{name}_out"], out[f"conv_{name}_coors"] = conv.weight.detach().numpy(), yf.numpy(), yc.numpy()
        out[f"conv_{name}_shape"] = np.array(list(y.spatial_shape))
        out[f"inv_{name}_w"], out[f"inv_{name}_out"] = inv.weight.detach().numpy(), z.features.numpy()
        assert torch.equal(z.indices, coors)
    sub = S.SubMConv3d(8, 12, 3, padding=0, bias=True, indice_key="s")
    with torch.no_grad():
        y = sub(S.SparseConvTensor(feats, coors, [9, 20, 24], 2))
    out["subm_w"], out["subm_b"], out["subm_out"] = sub.weight.detach().numpy(), sub.bias.detach().numpy(), y.features.numpy()
    np.savez_compressed(os.path.join(OUT, "spconv_layers.npz"), **out)

    out = {}
    torch.manual_seed(3)
    net = S.SimpleSparseUNet(**SO.SP_UNET, return_multiscale_features=True).eval()
    _rand_bn(net, 5)
    feats, coors = SO.synth_sparse(4, 2, (9, 32, 32), 500, 8)
    with torch.no_grad():
        r = net(dict(voxel_feats=feats, voxel_coors=coors))[0]
    assert torch.equal(r["voxel_coors"], coors)
    out["unet_feats"], out["unet_coors"], out["unet_out"] = feats.numpy(), coors.numpy(), r["voxel_feats"].numpy()
    for i, d in enumerate(r["decoder_features"]):
        f, c = _sort_rows(d.features, d.indices)
        out[f"unet_ms{i}_f"], out[f"unet_ms{i}_c"] = f.numpy(), c.numpy()
    for k, v in net.state_dict().items():
        out["unet_sd." + k] = v.numpy()
    torch.manual_seed(7)
    mix = S.VirtualVoxelMixer(**SO.SP_MIXER).eval()
    _rand_bn(mix, 9)
    feats, coors = SO.synth_sparse(8, 3, (8, 24, 24), 300, 8)
    with torch.no_grad():
        rf, rc, _ = mix(feats, coors, 3)
    assert torch.equal(rc, coors)
    out["mixer_feats"], out["mixer_coors"], out["mixer_out"] = feats.numpy(), coors.numpy(), rf.numpy()
    for k, v in mix.state_dict().items():
        out["mixer_sd." + k] = v.numpy()
    np.savez_compressed(os.path.join(OUT, "spconv_unet.npz"), **out)
    print("spconv", out["unet_out"].shape, out["mixer_out"].shape)



def fsd_cluster_fixture():
    """SURVEY 8f next-3: find_connected_componets / ClusterAssigner from the reference's own source (single_stage_fsd.py:47-81, 922-999)."""
    from oracle import fsd_oracle as FO
    RF = ref_shim.reference_functions("mmdet3d/models/detectors/single_stage_fsd.py",
                                      ["filter_almost_empty", "find_connected_componets", "modify_cluster_by_class", "ClusterAssigner"])
    out = {}
    pts, bidx = FO.synth_centres(3, 3, 700)
    g = torch.Generator().manual_seed(1)
    perm = torch.randperm(pts.shape[0], generator=g)   # samples interleaved: the numbering still goes sample by sample
    out["cc_points"], out["cc_batch"] = pts.numpy(), bidx.numpy()
    out["cc_points_mixed"], out["cc_batch_mixed"] = pts[perm].numpy(), bidx[perm].numpy()
    for d in (0.1, 0.6, 2.0):
        out[f"cc_labels_{d}"] = RF["find_connected_componets"](pts, bidx, d).numpy()
        out[f"cc_labels_mixed_{d}"] = RF["find_connected_componets"](pts[perm], bidx[perm], d).numpy()
    cfg = dict(cluster_voxel_size=dict(Car=(0.3, 0.3, 6), Cyclist=(0.2, 0.2, 6), Pedestrian=(0.05, 0.05, 6)), min_points=2,
               point_cloud_range=[-80, -80, -2, 80, 80, 4], connected_dist=dict(Car=0.6, Cyclist=0.4, Pedestrian=0.1),
               class_names=['Car', 'Cyclist', 'Pedestrian'])
    ca = RF["ClusterAssigner"](**cfg)
    ca.num_classes = 3
    ca.train()
    pts_l, b_l = [], []
    for i, blob in enumerate((0.5, 0.3, 0.08)):
        p, b = FO.synth_centres(10 + i, 2, 1500, blob=blob)
        # coordinates on a 1/64 m lattice: per-voxel sums are then exact in fp32 and fp64 alike, so the voxel centres (scatter_v2 'avg')
        # do not depend on the summation order / accumulator width of the implementation under test
        pts_l.append(torch.round(p * 64) / 64)
        b_l.append(b)
    inds, masks = ca(pts_l, b_l, origin_points=[None] * 3)
    for i in range(3):
        out[f"ca_points{i}"], out[f"ca_batch{i}"] = pts_l[i].numpy(), b_l[i].numpy()
        out[f"ca_inds{i}"], out[f"ca_mask{i}"] = inds[i].numpy(), masks[i].numpy()
    np.savez_compressed(os.path.join(OUT, "fsd_cluster.npz"), **out)
    print("fsd_cluster", {k: int(out[k].max()) + 1 for k in out if k.startswith("cc_labels_")})


# ---- reference pins: what tests/test_oracle_*_vs_reference.py, test_ref_voxel_layer.py and test_host_logic.py compare with ----------
# Stored as compact records (oracle/golden_io.py): digests where the tests demand bit equality, seeded row samples + projections where
# they allow a tolerance.  Weights are regenerated from seeds on both sides (golden_io.seeded_state), inputs by the functions below.
SST_VS = VS
PIN_DROP_TEST = DROP_TEST


def pin_dsvfe_points():
    g = torch.Generator().manual_seed(17)
    vs, rng = (0.25, 0.25, 0.2), [-80, -80, -2, 80, 80, 4]
    pts = torch.cat([torch.cat([O.synth_frame(3 + b, 3000), torch.rand(3000, 2, generator=g)], 1) for b in range(2)])
    co = torch.cat([torch.nn.functional.pad(O.dynamic_voxelize(pts[b * 3000:(b + 1) * 3000], vs, rng), (1, 0), value=b)
                    for b in range(2)]).long()
    return pts, co, vs, rng


def pin_neck_inputs():
    g = torch.Generator().manual_seed(5)
    N, M, C = 5000, 700, 16
    pts = O.synth_frame(3, N, extra_dims=1)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0).long()
    vf = torch.randn(M, C, generator=g)
    vf[::7] = -1.0  # dropped voxels are padded rows
    inds = torch.randint(0, M, (N,), generator=g)
    return pts, coors, vf, inds


def pin_sir_inputs():
    N, G = 3000, 40
    g = torch.Generator().manual_seed(2)
    points = torch.cat([torch.randn(N, 3, generator=g) * 10, torch.rand(N, 2, generator=g)], 1)
    feats = torch.randn(N, 27, generator=g)
    gid = torch.randint(0, G, (N,), generator=g)
    coors = torch.stack([gid % 3, torch.zeros_like(gid), gid], 1)
    fcl = torch.randn(N, 3, generator=g) * 2
    return points, feats, coors, fcl


def sst_pins_fixture(R):
    from oracle import golden_io as GI
    out = {}
    vfe_kw = dict(in_channels=3, with_cluster_center=True, with_voxel_center=True, voxel_size=VS, point_cloud_range=RNG,
                  norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01))
    bb_kw = dict(d_model=[64], nhead=[4], num_blocks=1, dim_feedforward=[128], output_shape=[468, 468], num_attached_conv=0, to_bev=False)
    # config 1: 20k points, DynamicVFE -> SSTInputLayerV2 -> one SSTv2 block
    pts = O.synth_frame(1000, 20000)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0)
    vfe = R.DynamicVFE(feat_channels=[64, 64], **vfe_kw).eval()
    il = R.SSTInputLayerV2(DROP_TEST, (12, 12, 1), (468, 468, 1), shuffle_voxels=False, debug=True, mute=True).eval()
    bb = R.SSTv2(**bb_kw).eval()
    out["config1.vfe_spec"], out["config1.bb_spec"] = GI.state_spec(vfe), GI.state_spec(bb)
    GI.load_seeded(vfe, out["config1.vfe_spec"], 101)
    GI.load_seeded(bb, out["config1.bb_spec"], 102)
    with torch.no_grad():
        vf_r, vc_r = vfe(pts, coors)
        info_r = il(vf_r, vc_r, 1)
        out_r = bb(info_r)[0]["voxel_feats"]
    GI.record(out, "config1.vc", vc_r, exact=True)
    GI.record(out, "config1.vf", vf_r)
    for i in range(2):
        for k in (f"batch_win_inds_shift{i}", f"coors_in_win_shift{i}", f"voxel_drop_level_shift{i}"):
            GI.record(out, f"config1.{k}", info_r[k], exact=True)
    GI.record(out, "config1.out", out_r)
    # state-dict keys and shapes of the reference classes
    from sst_b200 import flagship as fl
    cfg = fl.sst_cfg(num_blocks=2)
    r_vfe = R.DynamicVFE(**{k: v for k, v in cfg['voxel_encoder'].items() if k != 'type'})
    r_bb = R.SSTv2(**{k: v for k, v in cfg['backbone'].items() if k != 'type'})
    lc = dict(cosine=True, non_shared_tau=True, use_bn=True)
    r_cos = R.SSTv2(d_model=[32], nhead=[4], num_blocks=1, dim_feedforward=[64], num_attached_conv=0, to_bev=False, layer_cfg=lc)
    for name, m in (("vfe", r_vfe), ("bb", r_bb), ("cosine", r_cos)):
        out[f"keys.{name}"] = {k: list(v.shape) for k, v in m.state_dict().items()}
    # Voxel2PointScatterNeck
    pts_n, coors_n, vf_n, inds_n = pin_neck_inputs()
    for with_xyz, norm in ((True, False), (True, True), (False, False)):
        neck = R.Voxel2PointScatterNeck(point_cloud_range=RNG, voxel_size=VS, with_xyz=with_xyz, normalize_local_xyz=norm).eval()
        r_out, r_mask = neck(pts_n, coors_n, vf_n, inds_n)
        GI.record(out, f"neck.{with_xyz}.{norm}.out", r_out, exact=True)
        GI.record(out, f"neck.{with_xyz}.{norm}.mask", r_mask, exact=True)
    # gradients of DynamicVFE -> SSTInputLayerV2 -> SSTv2 (eval-mode BN, one block)
    pts = O.synth_frame(1000, 6000)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0)
    vfe = R.DynamicVFE(feat_channels=[32, 64], **vfe_kw).eval()
    bb = R.SSTv2(**bb_kw).eval()
    out["grad.vfe_spec"], out["grad.bb_spec"] = GI.state_spec(vfe), GI.state_spec(bb)
    GI.load_seeded(vfe, out["grad.vfe_spec"], 103)
    GI.load_seeded(bb, out["grad.bb_spec"], 104)
    p_r = pts.clone().requires_grad_(True)
    vf_r, vc_r = vfe(p_r, coors)
    out_r = bb(il(vf_r, vc_r, 1))[0]["voxel_feats"]
    out_r.square().mean().backward()
    GI.record(out, "grad.points", p_r.grad)
    for pre, m in (("vfe.", vfe), ("bb.", bb)):
        for k, v in m.named_parameters():
            GI.record(out, "grad." + pre + k, v.grad, rows=4)
    # SIR gradients
    m = R.SIR(num_blocks=2, in_channels=[32, 37], feat_channels=[[32, 32], [32, 32]], rel_mlp_hidden_dims=[[16, 32], [16, 32]],
              norm_cfg=dict(type='LN', eps=1e-3), mode='max', xyz_normalizer=[20, 20, 4], act='gelu', unique_once=True).eval()
    out["sir.spec"] = GI.state_spec(m)
    GI.load_seeded(m, out["sir.spec"], 105)
    points, feats, coors_s, fcl = pin_sir_inputs()
    f_r = feats.clone().requires_grad_(True)
    a, b, _ = m(points, f_r, coors_s, fcl)
    (a.square().mean() + b.square().mean()).backward()
    GI.record(out, "sir.feats", f_r.grad)
    for k, p in m.named_parameters():
        GI.record(out, "sir." + k, p.grad, rows=4)
    # DynamicVFE in train(): outputs, gradients, running buffers after the step
    vfe = R.DynamicVFE(feat_channels=[32, 64], **vfe_kw).train()
    out["train.spec"] = GI.state_spec(vfe)
    GI.load_seeded(vfe, out["train.spec"], 106)
    p_r = pts.clone().requires_grad_(True)
    vf_r, vc_r = vfe(p_r, coors)
    vf_r.square().mean().backward()
    GI.record(out, "train.vc", vc_r, exact=True)
    GI.record(out, "train.vf", vf_r)
    GI.record(out, "train.points", p_r.grad)
    for k, p in vfe.named_parameters():
        GI.record(out, "train." + k, p.grad, rows=4)
    sd = vfe.state_dict()
    for k in ("vfe_layers.0.norm.running_mean", "vfe_layers.0.norm.running_var"):
        GI.record(out, "train." + k, sd[k])
    # DynamicScatterVFE in train()
    pts_d, co_d, vs, rng = pin_dsvfe_points()
    m = R.DynamicScatterVFE(in_channels=5, feat_channels=[32, 32], with_cluster_center=True, with_voxel_center=True, voxel_size=vs,
                            point_cloud_range=rng, norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01), unique_once=True,
                            rel_dist_scaler=10.0).train()
    out["dsvfe.spec"] = GI.state_spec(m)
    GI.load_seeded(m, out["dsvfe.spec"], 107)
    x = pts_d.clone().requires_grad_(True)
    vf, vc, inv = m(x, co_d, return_inv=True)
    probe = torch.randn(vf.shape, generator=torch.Generator().manual_seed(1))
    (vf * probe).sum().backward()
    GI.record(out, "dsvfe.vc", vc, exact=True)
    GI.record(out, "dsvfe.inv", inv, exact=True)
    GI.record(out, "dsvfe.vf", vf)
    GI.record(out, "dsvfe.points", x.grad)
    for k, p in m.named_parameters():
        GI.record(out, "dsvfe." + k, p.grad, rows=4)
    GI.save(os.path.join(OUT, "ref_sst_pins.npz"), out)
    print("ref_sst_pins", len(out), "arrays")


def fsd_pins_fixture():
    from oracle import fsd_oracle as FO, golden_io as GI
    RF = ref_shim.reference_functions("mmdet3d/models/detectors/single_stage_fsd.py",
                                      ["filter_almost_empty", "find_connected_componets", "find_connected_componets_single_batch",
                                       "modify_cluster_by_class", "ClusterAssigner"])
    out = {}
    pts, bidx = FO.synth_centres(3, 3, 700)
    for d in (0.1, 0.6, 2.0):
        GI.record(out, f"cc.{d}", RF["find_connected_componets"](pts, bidx, d), exact=True)
        GI.record(out, f"cc_single.{d}", RF["find_connected_componets_single_batch"](pts[:700], bidx[:700], d), exact=True)
    ca = RF["ClusterAssigner"](**FSD_CA_CFG)
    ca.num_classes = 3
    ca.train()
    pts_l, b_l = pin_cluster_inputs()
    inds, masks = ca(pts_l, b_l, origin_points=[None] * 3)
    for i in range(3):
        GI.record(out, f"ca.class{i}", inds[i][:, 0].long(), exact=True)
        GI.record(out, f"ca.inds{i}", inds[i][:, 1:].int(), exact=True)
        GI.record(out, f"ca.mask{i}", masks[i], exact=True)
    ca.eval()
    m0 = b_l[0] == 0
    inds1, _ = ca([pts_l[0][m0]], [b_l[0][m0]], origin_points=[None])
    GI.record(out, "ca.eval_inds", inds1[0][:, 1:].int(), exact=True)
    GI.save(os.path.join(OUT, "ref_fsd_pins.npz"), out)
    print("ref_fsd_pins", len(out), "arrays")


FSD_CA_CFG = dict(cluster_voxel_size=dict(Car=(0.3, 0.3, 6), Cyclist=(0.2, 0.2, 6), Pedestrian=(0.05, 0.05, 6)), min_points=2,
                  point_cloud_range=[-80, -80, -2, 80, 80, 4], connected_dist=dict(Car=0.6, Cyclist=0.4, Pedestrian=0.1),
                  class_names=['Car', 'Cyclist', 'Pedestrian'])


def pin_cluster_inputs():
    from oracle import fsd_oracle as FO
    pts_l, b_l = [], []
    for i, blob in enumerate((0.5, 0.3, 0.08)):
        p, b = FO.synth_centres(10 + i, 2, 1500, blob=blob)
        order = torch.argsort(b, stable=True)
        pts_l.append(p[order])
        b_l.append(b[order])
    return pts_l, b_l


SPCONV_PIN_CONV = [(3, 2, 1), (3, 2, (0, 1, 1)), ((3, 1, 1), (2, 1, 1), 0), (2, 2, 0)]
SPCONV_PIN_SUBM = [(3, 1), ((3, 1, 1), (1, 0, 0)), (3, 0), (3, (0, 1, 1))]
SPCONV_PIN_UNET = dict(in_channels=8, sparse_shape=[9, 32, 32], order=('conv', 'norm', 'act'),
                       norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01), base_channels=8, output_channels=16,
                       encoder_channels=((8,), (8, 8, 8), (16, 16, 16), (16, 16, 16)),
                       encoder_paddings=((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1)),
                       decoder_channels=((16, 16, 16), (16, 16, 8), (8, 8, 8), (8, 8, 8)), decoder_paddings=((1, 1), (1, 0), (0, 0), (0, 1)))
SPCONV_PIN_MIXER = dict(in_channels=8, sparse_shape=[8, 24, 24], norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01), base_channels=8,
                        output_channels=12, encoder_channels=((8,), (8, 8), (8, 8)), encoder_paddings=((1,), (1, 1), (1, 1)),
                        decoder_channels=((8, 8, 8), (8, 8, 8), (8, 8, 8)), decoder_paddings=((1, 1), (1, 1), (1, 1)))


def spconv_pins_fixture():
    """The reference's vendored spconv v1 layers and sparse U-Nets with seeded weights (rows of strided outputs sorted by coordinate)."""
    from oracle import golden_io as GI, spconv_oracle as SO
    S = ref_shim.load_spconv()
    out = {}
    feats, coors = SO.synth_sparse(1, 2, (9, 20, 24), 300, 8)
    for i, (ks, stride, padding) in enumerate(SPCONV_PIN_CONV):
        conv = S.SparseConv3d(8, 12, ks, stride=stride, padding=padding, bias=False, indice_key="k")
        inv = S.SparseInverseConv3d(12, 6, ks, indice_key="k", bias=False)
        GI.load_seeded(conv, GI.state_spec(conv), 200 + i)
        GI.load_seeded(inv, GI.state_spec(inv), 210 + i)
        with torch.no_grad():
            y = conv(S.SparseConvTensor(feats, coors, [9, 20, 24], 2))
            z = inv(y)
        yf, yc = _sort_rows(y.features, y.indices)
        out[f"conv{i}.geometry"] = [list(conv.kernel_size), list(conv.stride), list(conv.padding)]
        out[f"conv{i}.spatial_shape"] = [int(v) for v in y.spatial_shape]
        GI.record(out, f"conv{i}.coors", yc.int(), exact=True)
        GI.record(out, f"conv{i}.out", yf, rows=GI.MIN_ROWS)
        GI.record(out, f"conv{i}.inv_coors", z.indices, exact=True)
        GI.record(out, f"conv{i}.inv_out", z.features, rows=GI.MIN_ROWS)
    feats, coors = SO.synth_sparse(2, 2, (7, 18, 18), 250, 8)
    for i, (ks, padding) in enumerate(SPCONV_PIN_SUBM):
        conv = S.SubMConv3d(8, 10, ks, padding=padding, bias=True, indice_key="s")
        GI.load_seeded(conv, GI.state_spec(conv), 220 + i)
        with torch.no_grad():
            y = conv(S.SparseConvTensor(feats, coors, [7, 18, 18], 2))
        out[f"subm{i}.kernel_size"] = list(conv.kernel_size)
        GI.record(out, f"subm{i}.coors", y.indices, exact=True)
        GI.record(out, f"subm{i}.out", y.features, rows=GI.MIN_ROWS)
    net = S.SimpleSparseUNet(**SPCONV_PIN_UNET, return_multiscale_features=True).eval()
    out["unet.spec"] = GI.state_spec(net)
    GI.load_seeded(net, out["unet.spec"], 230)
    feats, coors = SO.synth_sparse(4, 2, (9, 32, 32), 500, 8)
    with torch.no_grad():
        r = net(dict(voxel_feats=feats, voxel_coors=coors))[0]
    GI.record(out, "unet.coors", r["voxel_coors"], exact=True)
    GI.record(out, "unet.out", r["voxel_feats"], rows=GI.MIN_ROWS)
    out["unet.n_levels"] = len(r["decoder_features"])
    for i, d in enumerate(r["decoder_features"]):
        f, c = _sort_rows(d.features, d.indices)
        GI.record(out, f"unet.ms{i}.coors", c.int(), exact=True)
        GI.record(out, f"unet.ms{i}.out", f, rows=GI.MIN_ROWS)
    net = S.VirtualVoxelMixer(**SPCONV_PIN_MIXER).eval()
    out["mixer.spec"] = GI.state_spec(net)
    GI.load_seeded(net, out["mixer.spec"], 240)
    feats, coors = SO.synth_sparse(8, 3, (8, 24, 24), 300, 8)
    with torch.no_grad():
        rf, rc, rshape = net(feats, coors, 3)
    GI.record(out, "mixer.coors", rc, exact=True)
    out["mixer.spatial_shape"] = [int(v) for v in rshape]
    GI.record(out, "mixer.out", rf, rows=GI.MIN_ROWS)
    GI.save(os.path.join(OUT, "ref_spconv_pins.npz"), out)
    print("ref_spconv_pins", len(out), "arrays")


VOXEL_PIN_CASES = [(VS, RNG), ((0.25, 0.25, 0.2), [-80, -80, -2, 80, 80, 4]), ((0.1, 0.1, 0.15), [-51.2, -51.2, -5, 51.2, 51.2, 3])]
HV_PIN_CASES = [  # (P, F, voxel_size, range, max_points, max_voxels)
    (20000, 4, (0.32, 0.32, 6), [-74.88, -74.88, -2, 74.88, 74.88, 4], 32, 20000),
    (20000, 4, (0.32, 0.32, 6), [-74.88, -74.88, -2, 74.88, 74.88, 4], 5, 300),       # both caps bite
    (30000, 5, (0.5, 0.5, 0.25), [-40, -40, -3, 40, 40, 1], 10, 16000),               # 3-D grid
    (7, 3, (1.0, 1.0, 1.0), [0, 0, 0, 4, 4, 4], 2, 3),
    (150000, 4, (0.32, 0.32, 6), [-74.88, -74.88, -2, 74.88, 74.88, 4], 32, 32000),
]


def pin_voxel_points():
    pts = O.synth_frame(11, 40000)
    pts[::7, 0] += 200.0
    pts[::11, 1] -= 300.0
    return pts


def pin_hv_points(P, F):
    pts = O.synth_frame(300 + P, P, extra_dims=F - 3)
    pts[::13, 0] += 500.0  # out of range -> clamped by this fork's voxeliser
    return pts


def voxel_layer_pins_fixture():
    """The reference's own C++ dynamic_voxelize / hard_voxelize (voxelization_cpu.cpp, compiled unmodified into oracle/_ref)."""
    from oracle import build_ref, golden_io as GI
    ref = build_ref.load_module() or (build_ref.build() and build_ref.load_module())
    out = {}
    pts = pin_voxel_points()
    for i, (vs, rng) in enumerate(VOXEL_PIN_CASES):
        co = torch.zeros((pts.shape[0], 3), dtype=torch.int32)
        ref.dynamic_voxelize(pts, co, list(vs), list(rng), 3)
        GI.record(out, f"dyn{i}.coors", co, exact=True)
    for i, (P, F, vs, rng, mp, mv) in enumerate(HV_PIN_CASES):
        pts = pin_hv_points(P, F)
        voxels = torch.zeros((mv, mp, F))
        coors = torch.zeros((mv, 3), dtype=torch.int32)
        npts = torch.zeros((mv,), dtype=torch.int32)
        n = ref.hard_voxelize(pts, voxels, coors, npts, list(vs), list(rng), mp, mv, 3)
        out[f"hv{i}.n"] = int(n)
        GI.record(out, f"hv{i}.voxels", voxels[:n], exact=True)
        GI.record(out, f"hv{i}.coors", coors[:n], exact=True)
        GI.record(out, f"hv{i}.npts", npts[:n], exact=True)
    GI.save(os.path.join(OUT, "ref_voxel_layer_pins.npz"), out)
    print("ref_voxel_layer_pins", len(out), "arrays")


SCATTER_PIN_CASES = [(150000, 128, 0), (200000, 3, -1), (5000, 64, -1), (17, 5, 0)]
VOXEL_CUDA_PIN_SIZES = [1, 20000, 150000]


def pin_scatter_inputs(P, C, lo):
    """feats, coors and output-gradient generator of one dynamic-scatter case (CPU tensors; for the sweep-sized cases the coors come from
    the oracle's voxeliser, oracle.sst_oracle.dynamic_voxelize, so that they do not depend on the implementation under test)."""
    g = torch.Generator().manual_seed(P + C)
    feats = torch.rand(P, C, generator=g) * 100 - 50
    if P >= 100000:
        pts = O.synth_frame(5, P)
        coors = O.dynamic_voxelize(pts, VS, RNG)
    else:
        coors = torch.randint(lo, 20, (P, 3), generator=g, dtype=torch.int32)
    return feats, coors, g


def pin_voxel_cuda_points(P):
    pts = O.synth_frame(77 + P, P)
    pts[::5, 0] += 300.0
    return pts


def ref_cuda_pins_fixture(out_dir=OUT):
    """The reference's own CUDA dynamic_voxelize and dynamic_point_to_voxel_forward / backward (voxelization_cuda.cu,
    scatter_points_cuda.cu, compiled unmodified into oracle/_ref) on a GPU: `python -m oracle.make_golden cuda-pins [DIR]`."""
    from oracle import build_ref, golden_io as GI
    ref = build_ref.load_module()
    assert ref is not None, "oracle/_ref/voxel_layer_ref*.so not built"
    dev = torch.device("cuda:0")
    out = {}
    for P in VOXEL_CUDA_PIN_SIZES:
        pts = pin_voxel_cuda_points(P).to(dev)
        r = torch.zeros((P, 3), dtype=torch.int32, device=dev)
        ref.dynamic_voxelize(pts, r, list(VS), list(RNG), 3)
        GI.record(out, f"voxelize{P}", r, exact=True)
    for reduce in ("max", "mean", "sum"):
        for P, C, lo in SCATTER_PIN_CASES:
            feats, coors, g = pin_scatter_inputs(P, C, lo)
            feats, coors = feats.to(dev), coors.to(dev)
            r_f, r_c, r_m, r_n = ref.dynamic_point_to_voxel_forward(feats, coors, reduce)
            key = f"scatter.{reduce}.{P}.{C}"
            GI.record(out, key + ".coors", r_c, exact=True)
            GI.record(out, key + ".map", r_m, exact=True)
            GI.record(out, key + ".count", r_n, exact=True)
            GI.record(out, key + ".feats", r_f, exact=reduce == "max")
            grad = torch.randn(r_f.shape, generator=g).to(dev)
            r_g = torch.zeros_like(feats)
            ref.dynamic_point_to_voxel_backward(r_g, grad, feats, r_f, r_m, r_n, reduce)
            GI.record(out, key + ".grad", r_g)
    torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    GI.save(os.path.join(out_dir, "ref_cuda_pins.npz"), out)
    print("ref_cuda_pins", len(out), "arrays")


REF_CONFIG_DIRS = ("configs/sst", "configs/sst_refactor", "configs/fsd", "configs/fsdv2")


def reference_configs_fixture():
    """The `model` dict of every config under configs/sst (v1 names), configs/sst_refactor, configs/fsd and configs/fsdv2, as parsed by the
    stand-in Config loader (inheritance resolved), written as Python literals."""
    import glob
    from sst_b200.config import Config
    files = sorted(f for d in REF_CONFIG_DIRS for f in glob.glob(os.path.join(ref_shim.REF_ROOT, d, "*.py")))
    # configs/sst/to_be_done_do_not_use.py inherits from a _base_ file that does not exist in the reference tree: mmcv cannot load it either
    files = [f for f in files if not f.endswith("to_be_done_do_not_use.py")]
    models = {os.path.relpath(f, ref_shim.REF_ROOT): _plain(Config.fromfile(f).get("model", {})) for f in files}
    names = sorted(models)
    np.savez_compressed(os.path.join(OUT, "reference_configs.npz"), files=np.array(names), models=np.array([repr(models[k]) for k in names]))
    print("reference_configs", len(models), "files")


def _plain(v):
    if isinstance(v, dict):
        return {k: _plain(x) for k, x in v.items()}
    if isinstance(v, (list, tuple)):
        return type(v)(_plain(x) for x in v)
    return v


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if "cuda-pins" in sys.argv[1:]:   # on a GPU machine that has oracle/_ref
        args = [a for a in sys.argv[1:] if a != "cuda-pins"]
        ref_cuda_pins_fixture(args[0] if args else OUT)
        sys.exit(0)
    if "pins" in sys.argv[1:]:   # only the reference pins
        sst_pins_fixture(ref_shim.load())
        fsd_pins_fixture()
        spconv_pins_fixture()
        voxel_layer_pins_fixture()
        reference_configs_fixture()
        sys.exit(0)
    if "fsdv2" in sys.argv[1:]:
        fsdv2_front_fixture(ref_shim.load())
        sys.exit(0)
    if "spconv" in sys.argv[1:] or "fsd" in sys.argv[1:]:   # only the next-1 / next-3 fixtures
        if "spconv" in sys.argv[1:]:
            spconv_fixture()
        if "fsd" in sys.argv[1:]:
            fsd_cluster_fixture()
        sys.exit(0)
    R = ref_shim.load()
    sst_fixture(R)
    sst_v1_fixture(R)
    vfe_fixture(R)
    sir_fixture(R)
    dsvfe_fixture(R)
    fsdv2_front_fixture(R)
    scatter_fixture()
    neck_fixture(R)
    hard_voxelize_fixture()
    spconv_fixture()
    fsd_cluster_fixture()
    sst_pins_fixture(R)
    fsd_pins_fixture()
    spconv_pins_fixture()
    voxel_layer_pins_fixture()
    reference_configs_fixture()
