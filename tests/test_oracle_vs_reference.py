"""CPU: pins the oracle to what the reference's own Python (unmodified, through oracle/ref_shim.py) computed on seeded inputs with seeded
weights - outputs, gradients and state-dict layouts recorded in tests/golden/ref_sst_pins.npz by `python -m oracle.make_golden pins`."""
import os

import pytest
import torch

from oracle import golden_io as GI, make_golden as MG, sst_oracle as O

VS = (0.32, 0.32, 6)
RNG = [-74.88, -74.88, -2, 74.88, 74.88, 4]
DROP_TEST = {0: {'max_tokens': 30, 'drop_range': (0, 30)}, 1: {'max_tokens': 60, 'drop_range': (30, 60)},
             2: {'max_tokens': 100, 'drop_range': (60, 100)}, 3: {'max_tokens': 144, 'drop_range': (100, 100000)}}


@pytest.fixture(scope="module")
def Z():
    return GI.load(os.path.join(os.path.dirname(__file__), "golden", "ref_sst_pins.npz"))


def test_config1_path(Z):
    """BASELINE config 1: 20k points, DynamicScatter + 1 SRA block d=64 h=4 on CPU (reference plumbing)."""
    pts = O.synth_frame(1000, 20000)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0)
    wv, wb = GI.seeded_state(Z["config1.vfe_spec"], 101), GI.seeded_state(Z["config1.bb_spec"], 102)
    vf_o, vc_o = O.dynamic_vfe_forward(pts, coors, wv, VS, RNG, 2)
    GI.check(Z, "config1.vc", vc_o)
    GI.check(Z, "config1.vf", vf_o, rtol=1e-6, atol=1e-6)
    info_o = O.input_layer_v2(vf_o, vc_o, DROP_TEST, (12, 12, 1), (468, 468, 1))
    for i in range(2):
        for k in (f"batch_win_inds_shift{i}", f"coors_in_win_shift{i}", f"voxel_drop_level_shift{i}"):
            GI.check(Z, f"config1.{k}", info_o[k])
    out_o = O.sstv2_forward(info_o, wb, [4], 1)
    GI.check(Z, "config1.out", out_o, rtol=1e-5, atol=1e-6)


def test_state_dict_keys_match_reference(Z):
    """The registered modules are checkpoint-compatible: same state-dict keys and shapes as the reference's."""
    from sst_b200 import flagship as fl
    cfg = fl.sst_cfg(num_blocks=2)
    vfe, il, bb = fl.build_sst(cfg)
    from sst_b200.sst_modules import SSTv2
    lc = dict(cosine=True, non_shared_tau=True, use_bn=True)
    o = SSTv2(d_model=[32], nhead=[4], num_blocks=1, dim_feedforward=[64], num_attached_conv=0, to_bev=False, layer_cfg=lc)
    for name, ours in (("vfe", vfe), ("bb", bb), ("cosine", o)):
        assert {k: list(v.shape) for k, v in ours.state_dict().items()} == Z[f"keys.{name}"], name


@pytest.mark.parametrize("with_xyz,norm", [(True, False), (True, True), (False, False)])
def test_voxel2point_neck(Z, with_xyz, norm):
    """oracle.voxel2point_neck vs the unmodified reference Voxel2PointScatterNeck (necks/voxel2point_neck.py:28-62)."""
    pts, coors, vf, inds = MG.pin_neck_inputs()
    o_out, o_mask = O.voxel2point_neck(pts, coors, vf, inds, VS, RNG, with_xyz, norm)
    GI.check(Z, f"neck.{with_xyz}.{norm}.out", o_out)
    GI.check(Z, f"neck.{with_xyz}.{norm}.mask", o_mask)


def test_oracle_gradients_match_reference(Z):
    """The oracle is differentiable torch code, so autograd through it is the checker for the backward kernels: parameter and input
    gradients of DynamicVFE -> SSTInputLayerV2 -> SSTv2 (eval-mode BN, one block) against the reference's autograd."""
    pts = O.synth_frame(1000, 6000)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0)
    vfe_spec, bb_spec = Z["grad.vfe_spec"], Z["grad.bb_spec"]
    wv = {k: v.requires_grad_("running" not in k) for k, v in GI.seeded_state(vfe_spec, 103).items()}
    wb = {k: v.requires_grad_(True) for k, v in GI.seeded_state(bb_spec, 104).items()}
    p_o = pts.clone().requires_grad_(True)
    vf_o, vc_o = O.dynamic_vfe_forward(p_o, coors, wv, VS, RNG, 2)
    info_o = O.input_layer_v2(vf_o, vc_o, DROP_TEST, (12, 12, 1), (468, 468, 1))
    out_o = O.sstv2_forward(info_o, wb, [4], 1)
    out_o.square().mean().backward()
    GI.check(Z, "grad.points", p_o.grad, rtol=1e-4, atol=1e-7)
    names = [k[len("grad."):] for k in Z["meta"] if k.startswith(("grad.vfe.", "grad.bb."))]
    assert names
    for k in names:
        w = wv[k[4:]] if k.startswith("vfe.") else wb[k[3:]]
        GI.check(Z, "grad." + k, w.grad, rtol=2e-4, atol=1e-7)


def test_oracle_sir_gradients_match_reference(Z):
    """Same for FSD's SIR (point-group MLP + pooling): oracle autograd == reference autograd."""
    points, feats, coors, fcl = MG.pin_sir_inputs()
    w = {k: v.requires_grad_(True) for k, v in GI.seeded_state(Z["sir.spec"], 105).items()}
    f_o = feats.clone().requires_grad_(True)
    ao, bo, _ = O.sir_forward(points, f_o, coors, fcl, w, 2, 3, 2, [20, 20, 4])
    (ao.square().mean() + bo.square().mean()).backward()
    GI.check(Z, "sir.feats", f_o.grad, rtol=1e-4, atol=1e-7)
    names = [k for k in w if "sir." + k in Z["meta"]]
    assert len(names) == len(w), f"parameters without a reference record: {sorted(set(w) - set(names))}"
    for k in names:
        GI.check(Z, "sir." + k, w[k].grad, rtol=2e-4, atol=1e-7)


def test_training_mode_vfe_matches_reference(Z):
    """DynamicVFE in TRAIN mode (naiveSyncBN1d batch statistics, single process) - outputs, input / parameter gradients and the
    running-buffer update of one step against the reference."""
    pts = O.synth_frame(1000, 6000)
    coors = torch.nn.functional.pad(O.dynamic_voxelize(pts, VS, RNG), (1, 0), value=0)
    w0 = GI.seeded_state(Z["train.spec"], 106)
    w = {k: v.clone().requires_grad_("running" not in k) for k, v in w0.items()}
    p_o = pts.clone().requires_grad_(True)
    vf_o, vc_o = O.dynamic_vfe_forward(p_o, coors, w, VS, RNG, 2, training=True)
    vf_o.square().mean().backward()
    GI.check(Z, "train.vc", vc_o)
    GI.check(Z, "train.vf", vf_o, rtol=1e-5, atol=1e-6)
    GI.check(Z, "train.points", p_o.grad, rtol=1e-4, atol=1e-7)
    for k in w:
        if "running" not in k:
            GI.check(Z, "train." + k, w[k].grad, rtol=2e-4, atol=1e-7)
    # running buffers after the step (layer 0 sees the decorated points): nn.BatchNorm1d update with the unbiased variance
    with torch.no_grad():
        ls = [pts]
        vmean, mcoors = O.dynamic_scatter_module(pts, coors, True)
        ls.append(pts[:, :3] - vmean[O._canvas_lookup(coors, mcoors, RNG, VS)][:, :3])
        ls.append(O._center_offsets(pts, coors, VS, RNG))
        y0 = torch.nn.functional.linear(torch.cat(ls, 1), w0["vfe_layers.0.linear.weight"])
        rm, rv = O.bn_running_update(y0, w0["vfe_layers.0.norm.running_mean"], w0["vfe_layers.0.norm.running_var"], 0.01)
    GI.check(Z, "train.vfe_layers.0.norm.running_mean", rm, rtol=1e-5, atol=1e-7)
    GI.check(Z, "train.vfe_layers.0.norm.running_var", rv, rtol=1e-5, atol=1e-7)


def test_dynamic_scatter_vfe_training_mode_matches_reference(Z):
    """DynamicScatterVFE in train() (batch-statistics BatchNorm, autograd through scatter_v2): outputs and gradients of the oracle's
    training=True restatement against the reference class - the checker of the product's training composition"""
    pts, co, vs, rng = MG.pin_dsvfe_points()
    w = {k: v.requires_grad_("running" not in k) for k, v in GI.seeded_state(Z["dsvfe.spec"], 107).items()}
    x2 = pts.clone().requires_grad_(True)
    of, oc, oinv = O.dynamic_scatter_vfe_forward(x2, co, w, vs, rng, 2, rel_dist_scaler=10.0, training=True)
    GI.check(Z, "dsvfe.vc", oc)
    GI.check(Z, "dsvfe.inv", oinv)
    GI.check(Z, "dsvfe.vf", of, rtol=1e-4, atol=1e-5)
    probe = torch.randn(of.shape, generator=torch.Generator().manual_seed(1))
    (of * probe).sum().backward()
    GI.check(Z, "dsvfe.points", x2.grad, rtol=1e-3, atol=1e-5)
    names = [k for k in w if "running" not in k]
    assert names and all("dsvfe." + k in Z["meta"] for k in names), "parameters without a reference record"
    for k in names:
        GI.check(Z, "dsvfe." + k, w[k].grad, rtol=1e-3, atol=1e-4 * Z["meta"]["dsvfe." + k]["abs_max"] + 1e-7)
