"""B200: FSDSegEngine (sst_b200/fsd_engine.py) - the FSD segmentation front as one CUDA graph - against the registered module chain
DynamicScatterVFE -> SimpleSparseUNet -> Voxel2PointScatterNeck (bit-identical: same kernels, same tables, same summation order) and,
at a small geometry, against the oracle chain."""
import pytest
import torch

from oracle import spconv_oracle as SO
from oracle import sst_oracle as O
from sst_b200 import flagship as fl
from sst_b200.fsd_engine import FSDSegEngine, module_front
from sst_b200.spconv_modules import set_spconv_precision

pytestmark = pytest.mark.gpu

PRECISIONS = ("bf16", "fp32_tc", "fp32")


def _frames(seeds, sizes):
    g = torch.Generator().manual_seed(sum(seeds))
    return [torch.cat([fl.synth_frame(s, n), torch.rand(n, 2, generator=g)], 1) for s, n in zip(seeds, sizes)]


def _load(eng, frames, dev):
    pts = torch.cat(frames).to(dev)
    offs = torch.tensor([0] + [int(f.shape[0]) for f in frames], dtype=torch.int32).cumsum(0).int().to(dev)
    eng.load_frames_device(pts, offs)


def _modules(vfe, unet, neck, frames, precision, dev, vs=fl.FSD_SEG_VOXEL_SIZE, rng=fl.FSD_PC_RANGE):
    vfe.precision = "bf16" if precision == "bf16" else "fp32"
    set_spconv_precision(unet, precision)
    with torch.no_grad():
        return module_front(vfe, unet, neck, [f.to(dev) for f in frames], vs, rng)


def _assert_same(eng_out, ref, n_points):
    out, mask, uf, vc, inv = ref
    torch.cuda.synchronize()
    M, K = int(eng_out["num_voxels"].item()), int(eng_out["num_pts"].item())
    assert M == vc.shape[0] and K == out.shape[0]
    assert torch.equal(eng_out["voxel_coors"][:M].long(), vc)
    assert torch.equal(eng_out["unq_inv"][:n_points].long(), inv)
    assert bool((eng_out["unq_inv"][n_points:] == -1).all())
    assert torch.equal(eng_out["voxel_feats"][:M], uf)
    assert torch.equal(eng_out["pts_mask"][:n_points], mask) and not bool(eng_out["pts_mask"][n_points:].any())
    assert torch.equal(eng_out["pts_feats"][:K], out)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_engine_matches_the_module_chain(cuda, precision):
    """configs/fsd shapes, B = 2, two seeds: bit-identical voxel coordinates, unq_inv, U-Net features, neck output, mask and counts."""
    vfe, unet, neck = fl.build_fsd_front(seed=1)
    vfe, unet = vfe.to(cuda), unet.to(cuda)
    eng = FSDSegEngine(fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE, vfe, unet, neck, max_points=2 * 60000, batch_size=2, precision=precision,
                       device=cuda)
    assert eng.graph is not None and eng.launches_per_frame > 34
    for seeds in ((11, 12), (13, 14)):
        frames = _frames(seeds, (60000, 45000))
        _load(eng, frames, cuda)
        got = eng.run()
        _assert_same(got, _modules(vfe, unet, neck, frames, precision, cuda), 105000)


def test_engine_matches_the_oracle_chain(cuda):
    """the small geometry of test_fsd_segmentation_front_pipeline: engine vs the oracle chain (pinned to the reference)."""
    from sst_b200 import registry
    vs, rng = (0.5, 0.5, 0.375), [-40, -40, -2, 40, 40, 4]
    norm = dict(type='naiveSyncBN1d', eps=1e-3, momentum=0.01)
    unet_cfg = dict(in_channels=64, sparse_shape=[16, 160, 160], norm_cfg=norm, base_channels=64, output_channels=64,
                    encoder_channels=((64,), (64, 64, 64), (64, 64, 64)), encoder_paddings=((1,), (1, 1, 1), (1, 1, 1)),
                    decoder_channels=((64, 64, 64), (64, 64, 64), (64, 64, 64)), decoder_paddings=((1, 1), (1, 0), (0, 1)))
    vfe, unet, neck = fl.build_fsd_front(vfe_cfg=dict(fl.FSD_VFE, voxel_size=vs, point_cloud_range=rng),
                                         unet_cfg=dict(unet_cfg, type="SimpleSparseUNet"),
                                         neck_cfg=dict(fl.FSD_NECK, voxel_size=vs, point_cloud_range=rng), seed=2)
    P = 6000
    frames = [torch.cat([O.synth_frame(7 + b, P) * torch.tensor([0.5, 0.5, 1.0]), torch.rand(P, 2, generator=torch.Generator().manual_seed(b))], 1)
              for b in range(2)]
    pts = torch.cat(frames)
    co = torch.cat([torch.nn.functional.pad(O.dynamic_voxelize(f, vs, rng), (1, 0), value=b) for b, f in enumerate(frames)]).long()
    vf_r, vc_r, inv_r = O.dynamic_scatter_vfe_forward(pts, co, dict(vfe.state_dict()), vs, rng, 2)
    uf_r, _ = SO.sparse_unet_forward(unet.state_dict(), vf_r, vc_r.int(), 2, unet_cfg["sparse_shape"], unet_cfg["encoder_channels"],
                                     unet_cfg["encoder_paddings"], unet_cfg["decoder_channels"], unet_cfg["decoder_paddings"])
    out_r, mask_r = O.voxel2point_neck(pts, co, uf_r, inv_r, vs, rng)
    for precision, rtol, atol in (("fp32", 1e-3, 1e-4), ("bf16", 1e-2, 1e-2)):
        eng = FSDSegEngine(vs, rng, vfe.to(cuda), unet.to(cuda), neck, max_points=2 * P, batch_size=2, precision=precision, device=cuda)
        _load(eng, frames, cuda)
        got = eng.run()
        torch.cuda.synchronize()
        M, K = int(got["num_voxels"].item()), int(got["num_pts"].item())
        assert torch.equal(got["voxel_coors"][:M].cpu().long(), vc_r) and torch.equal(got["unq_inv"].cpu().long(), inv_r)
        scale = float(uf_r.abs().max())
        torch.testing.assert_close(got["voxel_feats"][:M].cpu(), uf_r, rtol=rtol, atol=atol * scale)
        assert torch.equal(got["pts_mask"].cpu(), mask_r) and K == out_r.shape[0]
        torch.testing.assert_close(got["pts_feats"][:K].cpu(), out_r, rtol=rtol, atol=atol * max(scale, 1.0))


def test_replay_with_varying_point_counts(cuda):
    """One engine, three batches of different sizes (one frame much smaller than the other): each equals a fresh module run, two
    replays of the same input are identical and the torch allocator does not move."""
    vfe, unet, neck = fl.build_fsd_front(seed=3)
    vfe, unet = vfe.to(cuda), unet.to(cuda)
    eng = FSDSegEngine(fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE, vfe, unet, neck, max_points=150000, batch_size=2, precision="bf16",
                       device=cuda)
    for seeds, sizes in (((21, 22), (70000, 3000)), ((23, 24), (2000, 90000)), ((25, 26), (40000, 50000))):
        frames = _frames(seeds, sizes)
        _load(eng, frames, cuda)
        got = eng.run()
        _assert_same(got, _modules(vfe, unet, neck, frames, "bf16", cuda), sum(sizes))
    torch.cuda.synchronize()
    mem = torch.cuda.memory_allocated()
    first = eng.run()
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == mem
    first = {k: v.clone() for k, v in first.items()}
    second = eng.run()
    torch.cuda.synchronize()
    for k in first:
        assert torch.equal(first[k], second[k]), k


@pytest.mark.parametrize("precision", ("bf16", "fp32"))
def test_refresh_weights_after_load_state_dict(cuda, precision):
    vfe, unet, neck = fl.build_fsd_front(seed=4)
    vfe, unet = vfe.to(cuda), unet.to(cuda)
    eng = FSDSegEngine(fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE, vfe, unet, neck, max_points=80000, batch_size=1, precision=precision,
                       device=cuda)
    g = torch.Generator().manual_seed(5)
    for m in (vfe, unet):
        sd = m.state_dict()
        new = {k: (v + 0.05 * torch.randn(v.shape, generator=g).to(v.device) if v.is_floating_point() and "running_var" not in k
                   else (v * 1.5 if "running_var" in k else v)) for k, v in sd.items()}
        m.load_state_dict(new)
    eng.refresh_weights()
    frames = _frames((31,), (80000,))
    _load(eng, frames, cuda)
    got = eng.run()
    _assert_same(got, _modules(vfe, unet, neck, frames, precision, cuda), 80000)


def test_capture_reports_launches(cuda):
    vfe, unet, neck = fl.build_fsd_front(seed=6)
    eng = FSDSegEngine(fl.FSD_SEG_VOXEL_SIZE, fl.FSD_PC_RANGE, vfe.to(cuda), unet.to(cuda), neck, max_points=20000, batch_size=1,
                       precision="bf16", device=cuda, use_graph=True)
    assert eng.graph is not None
    assert eng.launches_per_frame >= 34 + 5 and eng.other_nodes_per_frame >= 0 and eng.buffer_bytes > 0
    print(f"[fsd engine] {eng.launches_per_frame} kernel nodes + {eng.other_nodes_per_frame} other nodes per frame, "
          f"{eng.buffer_bytes / 2**20:.0f} MiB of buffers")
