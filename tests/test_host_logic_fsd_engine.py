"""CPU: the FSD segmentation engine's static plan (sst_b200/fsd_engine.py build_plan) against the oracle's geometry, and its host-side
validation (every rejected configuration raises before any CUDA call - these tests run without a GPU)."""
import copy

import pytest
import torch

from oracle import spconv_oracle as SO
from sst_b200 import flagship
from sst_b200.fsd_engine import FSDSegEngine, build_plan
from sst_b200.registry import build_backbone


@pytest.fixture(scope="module")
def unet():
    torch.manual_seed(0)
    return build_backbone(dict(flagship.FSD_UNET)).eval()


def test_plan_has_the_34_convolutions(unet):
    plan = build_plan(unet, 2, 300000)
    assert len(plan.convs) == 34
    # one table per indice_key (shared like indice_dict); every inverse conv runs on the transposed table of its strided couple
    assert sorted(plan.tables) == sorted([f"subm{i}" for i in range(1, 6)] + [f"spconv{i}" for i in range(2, 6)])
    inverse = [cv for cv in plan.convs if cv["conv"].inverse]
    assert len(inverse) == 4 and all(cv["table"][1] == "inv" for cv in inverse)
    assert all(plan.tables[f"spconv{i}"]["want_inv"] for i in range(2, 6))
    assert [s[0] for s in plan.steps].count("merge") == 5
    assert plan.output.level == 0 and plan.output.ch == flagship.FSD_UNET["decoder_channels"][-1][-1]


def test_level_shapes_follow_conv_output_size(unet):
    plan = build_plan(unet, 1, 150000)
    shape = list(flagship.FSD_UNET["sparse_shape"])
    assert plan.levels[0]["shape"] == shape
    for i, lv in enumerate(plan.levels[1:], start=1):
        pad = flagship.FSD_UNET["encoder_paddings"][i][0]
        pad = list(pad) if isinstance(pad, (list, tuple)) else [pad] * 3
        shape = SO.conv_output_size(shape, [3] * 3, [2] * 3, pad)
        assert lv["shape"] == shape, (i, lv["shape"], shape)


def test_level_capacities_bound_the_real_row_counts(unet):
    feats, coors = flagship.fsd_sweep_voxels()
    plan = build_plan(unet, 1, coors.shape[0])
    rows = coors
    for lv in plan.levels[1:]:
        in_shape, out_shape, ks, st, pd = lv["geom"]
        rows = SO.out_coors(rows, 1, in_shape, ks, st, pd)
        assert list(out_shape) == lv["shape"]
        assert rows.shape[0] <= lv["cap"], (lv["shape"], rows.shape[0], lv["cap"])
    # the hand-over buffers have the capacity of their level
    for name, (level, width) in plan.buffers.items():
        assert 0 <= level < len(plan.levels) and width % 4 == 0


def test_concatenation_halves_are_written_in_place(unet):
    plan = build_plan(unet, 1, 1000)
    for lvl in range(1, 6):
        cat = f"cat{lvl}"
        writers = [cv for cv in plan.convs if cv["dst"].buf == cat]
        assert len(writers) == 2                       # x_bottom (left) and the lateral block (right)
        left, right = sorted(writers, key=lambda cv: cv["dst"].col)
        assert left["dst"].col == 0 and right["dst"].col == left["dst"].ch and right["dst"].ld == left["dst"].ld == plan.buffers[cat][1]
        assert right["res"] is not None                # SparseBasicBlock's identity


def _front():
    return flagship.build_fsd_front()


def _engine(vfe, unet, neck, **kw):
    args = dict(voxel_size=flagship.FSD_SEG_VOXEL_SIZE, point_cloud_range=flagship.FSD_PC_RANGE, voxel_encoder=vfe, backbone=unet,
                decode_neck=neck, max_points=1000, device="cuda:0")
    args.update(kw)
    return FSDSegEngine(**args)


def _rejects(exc, **kw):
    vfe, unet, neck = _front()
    mutate = kw.pop("mutate", None)
    if mutate is not None:
        vfe, unet, neck = mutate(vfe, unet, neck)
    with pytest.raises(exc):
        _engine(vfe, unet, neck, **kw)


def test_rejects_training_mode():
    _rejects(ValueError, mutate=lambda v, u, n: (v, u.train(), n))
    _rejects(ValueError, mutate=lambda v, u, n: (v.train(), u, n))


def test_rejects_unsupported_unet_options():
    def keep(v, u, n):
        u.keep_coors_dims = [0, 2, 3]
        return v, u, n

    def multiscale(v, u, n):
        u.return_multiscale_features = True
        return v, u, n
    _rejects(NotImplementedError, mutate=keep)
    _rejects(NotImplementedError, mutate=multiscale)
    cfg2d = dict(flagship.FSD_UNET, ndim=2, sparse_shape=[640, 640])
    _rejects(NotImplementedError, mutate=lambda v, u, n: (v, build_backbone(cfg2d).eval(), n))


def test_rejects_a_grid_outside_the_sparse_shape():
    small = dict(flagship.FSD_UNET, sparse_shape=[32, 320, 320])
    _rejects(ValueError, mutate=lambda v, u, n: (v, build_backbone(small).eval(), n))


def test_rejects_unsupported_voxel_encoders():
    from sst_b200.registry import MODELS
    dist = dict(flagship.FSD_VFE, with_distance=True)
    _rejects(NotImplementedError, mutate=lambda v, u, n: (MODELS.build(dist).eval(), u, n))
    avg = dict(flagship.FSD_VFE, mode="avg")
    _rejects(NotImplementedError, mutate=lambda v, u, n: (MODELS.build(avg).eval(), u, n))
    other = dict(flagship.FSD_VFE, voxel_size=(0.2, 0.2, 0.2))
    _rejects(ValueError, mutate=lambda v, u, n: (MODELS.build(other).eval(), u, n))
    narrow = dict(flagship.FSD_VFE, feat_channels=[64, 32])
    _rejects(ValueError, mutate=lambda v, u, n: (MODELS.build(narrow).eval(), u, n))


def test_rejects_bad_arguments():
    _rejects(ValueError, precision="fp16")
    _rejects(TypeError, mutate=lambda v, u, n: (v, u, copy.deepcopy(v)))
