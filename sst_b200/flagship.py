"""Factory for the BASELINE.json configurations (config dicts = the reference's own, e.g.
configs/sst_refactor/sst_waymoD5_1x_3class_8heads_v2.py:8-72), shared by bench.py, smoke() and the tests."""
import math

import torch

from .registry import build_backbone, build_middle_encoder, build_voxel_encoder
from . import sst_modules, voxel_modules  # noqa: F401  (registers the types)

VOXEL_SIZE = (0.32, 0.32, 6)
WINDOW_SHAPE = (12, 12, 1)
PC_RANGE = [-74.88, -74.88, -2, 74.88, 74.88, 4]
DROP_TRAIN = {0: {'max_tokens': 30, 'drop_range': (0, 30)}, 1: {'max_tokens': 60, 'drop_range': (30, 60)},
              2: {'max_tokens': 100, 'drop_range': (60, 100000)}}
DROP_TEST = {0: {'max_tokens': 30, 'drop_range': (0, 30)}, 1: {'max_tokens': 60, 'drop_range': (30, 60)},
             2: {'max_tokens': 100, 'drop_range': (60, 100)}, 3: {'max_tokens': 144, 'drop_range': (100, 100000)}}


def sst_cfg(d_model=128, nhead=8, dim_ff=256, num_blocks=6, in_channels=3):
    return dict(
        voxel_encoder=dict(type='DynamicVFE', in_channels=in_channels, feat_channels=[64, d_model], with_distance=False,
                           voxel_size=VOXEL_SIZE, with_cluster_center=True, with_voxel_center=True,
                           point_cloud_range=PC_RANGE, norm_cfg=dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01)),
        middle_encoder=dict(type='SSTInputLayerV2', window_shape=WINDOW_SHAPE, sparse_shape=(468, 468, 1),
                            shuffle_voxels=False, debug=True, drop_info=(DROP_TRAIN, DROP_TEST), pos_temperature=10000,
                            normalize_pos=False, mute=True),
        backbone=dict(type='SSTv2', d_model=[d_model] * num_blocks, nhead=[nhead] * num_blocks, num_blocks=num_blocks,
                      dim_feedforward=[dim_ff] * num_blocks, output_shape=[468, 468], num_attached_conv=0, to_bev=False,
                      debug=True),
    )


def build_sst(cfg=None, seed=0, randomize_norm=True):
    """Random-init modules (torch.manual_seed(seed) + the modules' own init, xavier for SSTv2).  BN running stats and
    affine norm parameters are perturbed so that every term of the arithmetic is exercised."""
    cfg = cfg or sst_cfg()
    torch.manual_seed(seed)
    vfe = build_voxel_encoder(cfg['voxel_encoder']).eval()
    il = build_middle_encoder(cfg['middle_encoder']).eval()
    bb = build_backbone(cfg['backbone']).eval()
    if randomize_norm:
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            for m in (vfe, bb):
                for n_, p in m.named_parameters():
                    if p.dim() == 1:
                        p.copy_(torch.randn(p.shape, generator=g) * 0.1 + (1.0 if 'norm' in n_ and 'weight' in n_ else 0.0))
                for n_, b in m.named_buffers():
                    if 'running_mean' in n_:
                        b.copy_(torch.randn(b.shape, generator=g) * 0.3)
                    if 'running_var' in n_:
                        b.copy_(torch.rand(b.shape, generator=g) + 0.5)
    return vfe, il, bb


def synth_frame(seed, P=150000, extra_dims=0, sigma=0.04):
    """The seeded "64-beam ring" synthetic sweep of SURVEY.md 8(d): beam ~ U{0..63}; r0 = 2.5*(74/2.5)^(beam/63);
    r = r0 + sigma*N(0,1); theta ~ U[0,2pi); z ~ U[-2,4); extra dims ~ U[0,1).  CPU tensor [P, 3+extra_dims] fp32."""
    g = torch.Generator().manual_seed(seed)
    beam = torch.randint(0, 64, (P,), generator=g).float()
    r = 2.5 * (74.0 / 2.5) ** (beam / 63.0) + sigma * torch.randn(P, generator=g)
    th = torch.rand(P, generator=g) * (2 * math.pi)
    z = torch.rand(P, generator=g) * 6.0 - 2.0
    cols = [r * torch.cos(th), r * torch.sin(th), z] + [torch.rand(P, generator=g) for _ in range(extra_dims)]
    return torch.stack(cols, dim=1).contiguous()


# ---- SURVEY 8f next-1: the FSD segmentation backbone (configs/fsd/fsd_waymoD1_1x.py:39-51) ---------------------------------------
FSD_UNET = dict(type="SimpleSparseUNet", in_channels=64, sparse_shape=[32, 640, 640], order=("conv", "norm", "act"),
                norm_cfg=dict(type="naiveSyncBN1d", eps=1e-3, momentum=0.01), base_channels=64, output_channels=128,
                encoder_channels=((64,), (64, 64, 64), (64, 64, 64), (128, 128, 128), (256, 256, 256)),
                encoder_paddings=((1,), (1, 1, 1), (1, 1, 1), ((0, 1, 1), 1, 1), (1, 1, 1)),
                decoder_channels=((256, 256, 128), (128, 128, 64), (64, 64, 64), (64, 64, 64), (64, 64, 64)),
                decoder_paddings=((1, 1), (1, 0), (1, 0), (0, 0), (0, 1)))


def fsd_sweep_voxels(seed=1000, points=150000, channels=64, shuffle=False):
    """A synthetic sweep voxelised on the configs/fsd segmentation grid (0.2 m, [32, 640, 640]): ([M, channels] fp32, [M, 4] int32
    (b,z,y,x)) on the CPU, rows in lexicographic order (what the voxel encoder hands over) unless shuffled."""
    pts = synth_frame(seed, points)
    lo = torch.tensor([-64.0, -64.0, -3.2])
    c = ((pts[:, :3] - lo) / 0.2).floor().long()[:, [2, 1, 0]]
    ok = (c[:, 0] >= 0) & (c[:, 0] < 32) & (c[:, 1] >= 0) & (c[:, 1] < 640) & (c[:, 2] >= 0) & (c[:, 2] < 640)
    c = torch.unique(c[ok], dim=0)
    g = torch.Generator().manual_seed(seed)
    if shuffle:
        c = c[torch.randperm(c.shape[0], generator=g)]
    coors = torch.cat([torch.zeros((c.shape[0], 1), dtype=torch.long), c], 1).int()
    return torch.randn((coors.shape[0], channels), generator=g), coors


def fsd_unet_bench(dev, reps=5, precisions=("bf16", "fp32_tc", "fp32")):
    """SimpleSparseUNet forward (tables + 34 convolution launches + glue) on one sweep, CUDA events on the current stream."""
    from . import spconv_modules as SP
    torch.manual_seed(0)
    net = build_backbone(dict(FSD_UNET)).to(dev).eval()
    feats, coors = fsd_sweep_voxels()
    info = dict(voxel_feats=feats.to(dev), voxel_coors=coors.to(dev))
    rec = {"workload": "SimpleSparseUNet, configs/fsd backbone shape, 150k-point sweep at 0.2 m, eval, batch 1", "voxels": int(coors.shape[0])}
    with torch.no_grad():
        for prec in precisions:
            SP.set_spconv_precision(net, prec)
            for _ in range(2):
                net(info)
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                net(info)
            b.record()
            torch.cuda.synchronize(dev)
            ms = a.elapsed_time(b) / reps
            rec[{"bf16": "f16_tcgen05", "fp32_tc": "fp32_split_tcgen05", "fp32": "fp32_ffma"}[prec]] = {"ms_per_sweep": ms, "sweeps_per_s": 1e3 / ms}
    return rec


def sir_bench(dev, reps=5, precisions=("bf16", "fp32")):
    """BASELINE config 3: FSD `SIR` (3 blocks, 150k points, 256 groups; configs/fsd/fsd_waymoD1_1x.py:92-103) forward, CUDA events on the
    current stream.  Same synthetic inputs as tools/sir_kernels.py / SURVEY 8(d)."""
    from .sir_modules import SIR
    N, G = 150000, 256
    g = torch.Generator().manual_seed(3)
    sp = torch.cat([torch.randn(N, 3, generator=g) * 10, torch.rand(N, 2, generator=g)], 1).to(dev)
    sf = torch.randn(N, 79, generator=g).to(dev)
    gid = torch.randint(0, G, (N,), generator=g)
    sc = torch.stack([gid % 3, torch.zeros_like(gid), gid], 1).to(dev)
    fcl = (torch.randn(N, 3, generator=g) * 2).to(dev)
    torch.manual_seed(0)
    sir = SIR(num_blocks=3, in_channels=[84, 133, 133], feat_channels=[[128, 128]] * 3, rel_mlp_hidden_dims=[[16, 32]] * 3,
              norm_cfg=dict(type="LN", eps=1e-3), mode="max", xyz_normalizer=[20, 20, 4], act="gelu", unique_once=True).eval().to(dev)
    flops = sum(2 * N * (3 * 16 + 16 * 32 + 32 * c + c * 128 + 256 * 128) for c in (84, 133, 133))   # SURVEY 8(d)
    rec = {"workload": "config3: FSD SIR, 3 blocks, 150k points, 256 groups, forward", "gflop": flops / 1e9}
    with torch.no_grad():
        for prec in precisions:
            sir.precision = prec
            for _ in range(2):
                sir(sp, sf, sc, fcl)
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                sir(sp, sf, sc, fcl)
            b.record()
            torch.cuda.synchronize(dev)
            ms = a.elapsed_time(b) / reps
            rec["bf16_tcgen05" if prec == "bf16" else "fp32_ffma"] = {"ms": ms, "tflops": flops / ms / 1e9}
    return rec


# ---- the configs/fsd segmentation front (configs/fsd/fsd_waymoD1_1x.py:7-58): voxel encoder -> U-Net -> voxel-to-point neck ----------
FSD_SEG_VOXEL_SIZE = (0.25, 0.25, 0.2)
FSD_PC_RANGE = [-80, -80, -2, 80, 80, 4]
FSD_VFE = dict(type="DynamicScatterVFE", in_channels=5, feat_channels=[64, 64], voxel_size=FSD_SEG_VOXEL_SIZE, with_cluster_center=True,
               with_voxel_center=True, point_cloud_range=FSD_PC_RANGE, norm_cfg=dict(type="naiveSyncBN1d", eps=1e-3, momentum=0.01),
               unique_once=True)
FSD_NECK = dict(type="Voxel2PointScatterNeck", voxel_size=FSD_SEG_VOXEL_SIZE, point_cloud_range=FSD_PC_RANGE)


def build_fsd_front(vfe_cfg=None, unet_cfg=None, neck_cfg=None, seed=0):
    """(DynamicScatterVFE, SimpleSparseUNet, Voxel2PointScatterNeck) in eval mode, random init (torch.manual_seed(seed)) with the
    BatchNorm statistics perturbed so that the folded scale / shift are not the identity."""
    from . import neck_modules, spconv_modules  # noqa: F401  (registers the types)
    from .registry import MODELS
    torch.manual_seed(seed)
    vfe = MODELS.build(dict(vfe_cfg or FSD_VFE)).eval()
    unet = build_backbone(dict(unet_cfg or FSD_UNET)).eval()
    neck = MODELS.build(dict(neck_cfg or FSD_NECK))
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for m in list(vfe.modules()) + list(unet.modules()):
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.2)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.weight.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.num_features, generator=g) * 0.1)
    return vfe, unet, neck
