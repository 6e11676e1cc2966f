"""CPU: host-side logic of the package (no GPU, no compute calls): registry builds from the reference's own config dicts,
positional table vs the oracle, drop-possibility check, lazy reference-layout dicts."""
import os

import pytest
import torch

from oracle import sst_oracle as O


def test_registry_builds_flagship_and_deepcopies_lists():
    from sst_b200 import flagship as fl, registry
    vfe, il, bb = fl.build_sst(fl.sst_cfg(num_blocks=2))
    assert len(bb.block_list) == 2 and bb.block_list[0].encoder_list[1].win_attn.self_attn.in_proj_weight.shape == (384, 128)
    # aliasing trap of SIRLayer (voxel_encoder.py:665): `[[16, 32]] * 3` shares one list object
    cfg = dict(type='SIR', num_blocks=3, in_channels=[84, 133, 133], feat_channels=[[128, 128]] * 3,
               rel_mlp_hidden_dims=[[16, 32]] * 3, norm_cfg=dict(type='LN', eps=1e-3), mode='max', xyz_normalizer=[20, 20, 4],
               act='gelu', unique_once=True)
    sir = registry.build_backbone(cfg)
    assert [tuple(b.rel_mlp[2][0].weight.shape) for b in sir.block_list] == [(84, 32), (133, 32), (133, 32)]
    assert cfg['rel_mlp_hidden_dims'][0] == [16, 32], "config must not be mutated"
    assert sir.block_list[0].vfe_layers[1].linear.weight.shape == (128, 256)


def test_pos_table_matches_oracle():
    from sst_b200.sst_modules import _pos_table
    for ws, d in (((12, 12, 1), 128), ((12, 12), 64), ((10, 10, 4), 96)):
        tab, ndim, maxw, L = _pos_table(ws, d, 10000, False)
        g = torch.Generator().manual_seed(0)
        w3 = ws if len(ws) == 3 else (ws[0], ws[1], 1)
        ciw = torch.stack([torch.randint(0, w3[2], (200,), generator=g), torch.randint(0, w3[1], (200,), generator=g),
                           torch.randint(0, w3[0], (200,), generator=g)], 1)
        ref = O.pos_embed_flat(ciw, ws, d, 10000, False)
        parts = [tab[a][ciw[:, 2 - a]] for a in range(ndim)]
        got = torch.cat(parts, 1)
        got = torch.cat([got, got.new_zeros(200, d - got.shape[1])], 1)
        assert torch.equal(got, ref)


def test_may_drop_host_check():
    from sst_b200 import flagship as fl
    from sst_b200.sst_modules import SSTInputLayerV2
    il = SSTInputLayerV2((fl.DROP_TRAIN, fl.DROP_TEST), (12, 12, 1), (468, 468, 1), mute=True)
    il.eval().set_drop_info()
    assert not il._may_drop()          # test drop_info keeps 144 = the whole 12x12 window
    il2 = SSTInputLayerV2((fl.DROP_TRAIN, fl.DROP_TEST), (12, 12, 1), (468, 468, 1), mute=True).train()
    il2.set_drop_info()
    assert il2._may_drop()             # training drop_info caps windows at 100 tokens


def test_lazy_dict_materialises_once():
    from sst_b200.sst_modules import _LazyDict
    calls = []
    d = _LazyDict(lambda: calls.append(1) or {0: "a", "voxel_drop_level": "b"})
    assert not calls
    assert 0 in d and d[0] == "a" and list(d.keys()) == [0, "voxel_drop_level"] and len(d) == 2
    assert len(calls) == 1


def test_reference_configs_load_and_build_unchanged():
    """The model dicts of configs/sst (v1 names), configs/sst_refactor, configs/fsd and configs/fsdv2 (the reference's files as parsed by the
    stand-in Config loader, tests/golden/reference_configs.npz, `python -m oracle.make_golden pins`): every hot-path module they name builds
    from the unmodified dict (SURVEY 8b)."""
    import ast
    import numpy as np
    from sst_b200 import registry
    from sst_b200.config import find_hot_path_modules
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_configs.npz"))
    files, models = [str(f) for f in z["files"]], [ast.literal_eval(str(m)) for m in z["models"]]
    assert len(files) >= 11 and sum(f.startswith("configs/sst/") for f in files) >= 5
    built = {}
    for f, model in zip(files, models):
        for path, node in find_hot_path_modules(model, registry.MODELS):
            try:
                m = registry.MODELS.build(node)
            except NotImplementedError as e:   # declared gaps (e.g. fusion layers) must be explicit
                built.setdefault("unsupported", []).append((os.path.basename(f), path, str(e)))
                continue
            built.setdefault(node["type"], 0)
            built[node["type"]] += 1
            assert sum(p.numel() for p in m.parameters()) >= 0
    for t in ("DynamicVFE", "SSTInputLayer", "SSTv1", "SSTInputLayerV2", "SSTv2", "DynamicScatterVFE", "SIR", "Voxel2PointScatterNeck",
              "SimpleSparseUNet", "VirtualVoxelMixer"):
        assert built.get(t, 0) >= 1, f"no config exercised {t}: {built}"
    assert not built.get("unsupported"), built.get("unsupported")


def test_config_loader_base_chain_and_delete(tmp_path):
    """Config.fromfile resolves a two-level `_base_` chain (list and string forms, relative paths), merges nested dicts key by key,
    replaces a dict marked `_delete_=True`, and keeps what the leaf file defines last."""
    from sst_b200.config import Config
    (tmp_path / "_base_").mkdir()
    (tmp_path / "_base_" / "model.py").write_text(
        "voxel_size = (0.32, 0.32, 6)\n"
        "model = dict(type='DynamicVoxelNet', voxel_encoder=dict(type='DynamicVFE', in_channels=3, feat_channels=[64, 128]),\n"
        "             backbone=dict(type='SSTv2', d_model=[128] * 6, nhead=[8] * 6, num_blocks=6))\n")
    (tmp_path / "mid.py").write_text(
        "_base_ = ['./_base_/model.py']\n"
        "model = dict(backbone=dict(num_blocks=2), neck=dict(type='SECONDFPN', in_channels=[128]))\n")
    (tmp_path / "leaf.py").write_text(
        "_base_ = './mid.py'\n"
        "import math\n"
        "voxel_size = (0.25, 0.25, 0.2)\n"
        "model = dict(voxel_encoder=dict(feat_channels=[32, 32]), neck=dict(_delete_=True, type='Voxel2PointScatterNeck'))\n")
    cfg = Config.fromfile(str(tmp_path / "leaf.py"))
    assert cfg["voxel_size"] == (0.25, 0.25, 0.2) and "math" not in cfg and "_base_" not in cfg
    m = cfg.model
    assert m.type == "DynamicVoxelNet"
    assert m["voxel_encoder"] == dict(type='DynamicVFE', in_channels=3, feat_channels=[32, 32])
    assert m["backbone"] == dict(type='SSTv2', d_model=[128] * 6, nhead=[8] * 6, num_blocks=2)
    assert m["neck"] == dict(type='Voxel2PointScatterNeck')
    with pytest.raises(AttributeError):
        m.no_such_key


def test_product_synth_frame_equals_oracle_generator():
    """bench.py draws its sweeps from sst_b200.flagship.synth_frame; the oracle's generator (SURVEY 8d) is the checker."""
    from sst_b200 import flagship as fl
    for seed, P, extra in ((1000, 5000, 0), (3, 777, 2)):
        assert torch.equal(fl.synth_frame(seed, P, extra), O.synth_frame(seed, P, extra))


def test_strict_config_walk_rejects_missing_hot_path_types():
    """find_hot_path_modules cannot pass by skipping: a reference hot-path type that is not registered is an error, every
    type the reference registers from a hot-path file IS registered, and the dead `SST` name resolves but refuses to build."""
    from sst_b200 import registry, norm  # noqa: F401
    from sst_b200.config import REFERENCE_HOT_PATH_TYPES, find_hot_path_modules
    for t in REFERENCE_HOT_PATH_TYPES:
        assert (t in registry.NORM_LAYERS) if t.startswith("naiveSyncBN") else (t in registry.MODELS), t
    empty = registry.Registry("empty")
    with pytest.raises(KeyError):
        find_hot_path_modules({"backbone": {"type": "SSTv1"}}, empty)
    assert find_hot_path_modules({"backbone": {"type": "SomethingElse"}}, empty) == []
    with pytest.raises(NotImplementedError):
        registry.MODELS.build({"type": "SST"})
    bn = registry.NORM_LAYERS.get("naiveSyncBN3d")(4).eval()
    x = torch.randn(2, 4, 3, 3, 3)
    torch.testing.assert_close(bn(x), torch.nn.functional.batch_norm(x, bn.running_mean, bn.running_var, bn.weight, bn.bias, False, 0.1, bn.eps))
