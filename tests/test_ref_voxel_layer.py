"""The reference's OWN voxel_layer (mmdet3d/ops/voxel/src/*.cpp,*.cu, compiled unmodified for sm_100a by oracle/build_ref.py) as the
checker, through what it returned on seeded inputs (tests/golden/ref_voxel_layer_pins.npz: its C++ on the CPU, `python -m oracle.make_golden
pins`; tests/golden/ref_cuda_pins.npz: its CUDA kernels on a B200, `python -m oracle.make_golden cuda-pins`):

  * CPU (not gpu): pins oracle.dynamic_voxelize / hard_voxelize to the reference C++ (voxelization_cpu.cpp:7-142).
  * GPU: libsstb200 vs the reference CUDA kernels - `dynamic_voxelize_gpu` (voxelization_cuda.cu:332-375) and
    `dynamic_point_to_voxel_forward/backward_gpu` (scatter_points_cuda.cu:183-303); indices bit-exact.

test_speed_vs_reference_cuda times the reference kernels themselves and runs only where oracle/_ref was built."""
import os

import pytest
import torch

from oracle import build_ref, golden_io as GI, make_golden as MG, sst_oracle as O

VS = (0.32, 0.32, 6)
RNG = [-74.88, -74.88, -2, 74.88, 74.88, 4]


GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def Z():
    return GI.load(os.path.join(GOLDEN, "ref_voxel_layer_pins.npz"))


@pytest.fixture(scope="module")
def ZC():
    return GI.load(os.path.join(GOLDEN, "ref_cuda_pins.npz"))


@pytest.fixture(scope="module")
def ref():
    try:
        m = build_ref.load_module()
    except Exception as e:  # e.g. a torch ABI mismatch
        pytest.skip(f"oracle/_ref not loadable: {e}")
    if m is None:
        pytest.skip("oracle/_ref/voxel_layer_ref.so not built")
    return m


@pytest.mark.parametrize("voxel_size,rng", MG.VOXEL_PIN_CASES)
def test_oracle_voxelize_equals_reference_cpp(Z, voxel_size, rng):
    case = MG.VOXEL_PIN_CASES.index((voxel_size, rng))
    GI.check(Z, f"dyn{case}.coors", O.dynamic_voxelize(MG.pin_voxel_points(), voxel_size, rng))


@pytest.mark.gpu
@pytest.mark.parametrize("P", MG.VOXEL_CUDA_PIN_SIZES)
def test_voxelize_vs_reference_cuda(cuda, ZC, P):
    from sst_b200 import ops
    pts = MG.pin_voxel_cuda_points(P).to(cuda)
    g = torch.zeros((P, 3), dtype=torch.int32, device=cuda)
    ops.dynamic_voxelize(pts, g, VS, RNG, 3)
    GI.check(ZC, f"voxelize{P}", g)


@pytest.mark.gpu
@pytest.mark.parametrize("reduce", ["max", "mean", "sum"])
@pytest.mark.parametrize("P,C,lo", MG.SCATTER_PIN_CASES)
def test_dynamic_scatter_vs_reference_cuda(cuda, ZC, reduce, P, C, lo):
    """Forward + backward against what the reference CUDA op (sorted unique + atomics) returned for the same inputs on a B200."""
    from sst_b200 import ops
    feats, coors, g = MG.pin_scatter_inputs(P, C, lo)
    feats, coors = feats.to(cuda), coors.to(cuda)
    key = f"scatter.{reduce}.{P}.{C}"
    g_f, g_c, g_m, g_n = ops.dynamic_point_to_voxel_forward(feats, coors, reduce)
    GI.check(ZC, key + ".coors", g_c)
    GI.check(ZC, key + ".map", g_m)
    GI.check(ZC, key + ".count", g_n)
    # the reference accumulates with fp32 atomics in arbitrary order
    GI.check(ZC, key + ".feats", g_f, rtol=1e-5, atol=2e-3 if reduce == "sum" else 1e-4)
    grad = torch.randn(g_f.shape, generator=g).to(cuda)
    g_g = torch.zeros_like(feats)
    ops.dynamic_point_to_voxel_backward(g_g, grad, feats, g_f, g_m, g_n, reduce)
    GI.check(ZC, key + ".grad", g_g, rtol=1e-6, atol=1e-6)


@pytest.mark.gpu
def test_speed_vs_reference_cuda(cuda, ref):
    """SURVEY 8(d): "also time the reference CUDA voxel_layer built for sm_100a - the in-tree GPU kernel to beat for V1/V2".
    Same device tensors, CUDA events, L2 flushed before every call, median of 15.  The gate is deliberately loose (2x); the
    measured ratios are printed (run with -s) and written to gpurun_out/ref_cuda_timing.json when that directory exists."""
    import json
    import os
    from sst_b200 import ops
    P, C = 150000, 128
    pts = O.synth_frame(1000, P).to(cuda)
    coors = ops.Voxelization(VS, RNG, -1)(pts)
    feats = torch.randn(P, C, device=cuda)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=cuda)

    def timed(fn, iters=15):
        ts = []
        for i in range(iters + 2):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b) * 1e3)
        return sorted(ts)[len(ts) // 2]

    out = {}
    rc = torch.zeros((P, 3), dtype=torch.int32, device=cuda)
    gc = torch.zeros((P, 3), dtype=torch.int32, device=cuda)
    out["dynamic_voxelize"] = dict(reference_us=timed(lambda: ref.dynamic_voxelize(pts, rc, list(VS), list(RNG), 3)),
                                   ours_us=timed(lambda: ops.dynamic_voxelize(pts, gc, VS, RNG, 3)))
    for red in ("max", "mean"):
        ds = ops.DynamicScatter(VS, RNG, red == "mean")
        out[f"dynamic_scatter_{red}_C{C}"] = dict(
            reference_us=timed(lambda: ref.dynamic_point_to_voxel_forward(feats, coors, red)),
            ours_us=timed(lambda: ds(feats, coors)))
    for k, v in out.items():
        v["speedup"] = v["reference_us"] / v["ours_us"]
        print(f"{k}: reference CUDA {v['reference_us']:.1f} us, libsstb200 {v['ours_us']:.1f} us, x{v['speedup']:.1f}")
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if os.path.isdir(d):
        json.dump(out, open(os.path.join(d, "ref_cuda_timing.json"), "w"), indent=1)
    assert out["dynamic_scatter_max_C128"]["speedup"] > 2.0 and out["dynamic_scatter_mean_C128"]["speedup"] > 2.0


@pytest.mark.parametrize("P,F,vs,rng,mp,mv", MG.HV_PIN_CASES[:-1])
def test_oracle_hard_voxelize_equals_reference_cpp(Z, P, F, vs, rng, mp, mv):
    """Pins oracle.hard_voxelize to the reference's own `hard_voxelize_cpu` (voxelization_cpu.cpp:43-142)."""
    case = MG.HV_PIN_CASES.index((P, F, vs, rng, mp, mv))
    ov, oc, on = O.hard_voxelize(MG.pin_hv_points(P, F), vs, rng, mp, mv)
    assert ov.shape[0] == Z[f"hv{case}.n"]
    GI.check(Z, f"hv{case}.coors", oc)
    GI.check(Z, f"hv{case}.npts", on)
    GI.check(Z, f"hv{case}.voxels", ov)


@pytest.mark.gpu
@pytest.mark.parametrize("P,F,vs,rng,mp,mv", MG.HV_PIN_CASES)
def test_hard_voxelize_vs_reference(cuda, Z, P, F, vs, rng, mp, mv):
    """libsstb200 `Voxelization(max_num_points > 0)` against the reference CPU implementation (bit-exact: pure data movement)."""
    from sst_b200 import ops
    case = MG.HV_PIN_CASES.index((P, F, vs, rng, mp, mv))
    layer = ops.Voxelization(vs, rng, mp, mv).eval()
    gv, gc, gn = layer(MG.pin_hv_points(P, F).to(cuda))
    assert gv.shape[0] == Z[f"hv{case}.n"]
    GI.check(Z, f"hv{case}.coors", gc)
    GI.check(Z, f"hv{case}.npts", gn)
    GI.check(Z, f"hv{case}.voxels", gv)
