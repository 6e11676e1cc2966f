"""CPU: pins oracle/spconv_oracle.py (dense restatement of the sparse convolutions, SURVEY 8f next-1) against the reference's own vendored
spconv v1 - its Python layers imported unmodified through oracle/ref_shim.load_spconv(), its C++ sources compiled unmodified by
oracle/build_ref.py - and its SimpleSparseUNet / VirtualVoxelMixer classes, run with seeded weights on seeded inputs.  What the reference
returned is recorded in tests/golden/ref_spconv_pins.npz by `python -m oracle.make_golden pins`."""
import os

import pytest
import torch

from oracle import golden_io as GI, make_golden as MG, spconv_oracle as SO


@pytest.fixture(scope="module")
def Z():
    return GI.load(os.path.join(os.path.dirname(__file__), "golden", "ref_spconv_pins.npz"))


def _by_coor(feats, coors):
    """rows sorted lexicographically by coordinate (the reference's SparseConv output order is hash-insertion order)"""
    c = coors.long()
    key = ((c[:, 0] * 4096 + c[:, 1]) * 4096 + c[:, 2]) * 4096 + c[:, 3]
    order = torch.argsort(key)
    return feats[order], coors[order]


@pytest.mark.parametrize("ks,stride,padding", MG.SPCONV_PIN_CONV)
def test_sparse_conv_and_inverse_match_reference(Z, ks, stride, padding):
    case = MG.SPCONV_PIN_CONV.index((ks, stride, padding))
    feats, coors = SO.synth_sparse(1, 2, (9, 20, 24), 300, 8)
    ks, stride, padding = Z[f"conv{case}.geometry"]
    w = GI.seeded_state([("weight", [*ks, 8, 12])], 200 + case)["weight"]
    wi = GI.seeded_state([("weight", [*ks, 12, 6])], 210 + case)["weight"]
    of, oc, oshape = SO.sparse_conv(feats, coors, 2, [9, 20, 24], w, stride, padding)
    assert oshape == Z[f"conv{case}.spatial_shape"]
    GI.check(Z, f"conv{case}.coors", oc)          # oracle order is lexicographic
    GI.check(Z, f"conv{case}.out", of, rtol=1e-4, atol=1e-5)
    # the neighbour table regrouped from the reference's index pairs
    nbr = SO.neighbour_table(coors, oc, 2, [9, 20, 24], ks, stride, padding)
    torch.testing.assert_close(SO.indice_conv(feats, nbr, w), of, rtol=1e-4, atol=1e-5)
    zi = SO.inverse_conv(of, oc, 2, oshape, coors, [9, 20, 24], wi, stride, padding)
    GI.check(Z, f"conv{case}.inv_coors", coors)   # the inverse conv restores the couple conv's input rows, in order
    GI.check(Z, f"conv{case}.inv_out", zi, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("ks,padding", MG.SPCONV_PIN_SUBM)
def test_subm_conv_matches_reference(Z, ks, padding):
    """incl. layers built with padding != k//2: the index generation centres every SubM conv (spconv_ops.h:74-78)"""
    case = MG.SPCONV_PIN_SUBM.index((ks, padding))
    feats, coors = SO.synth_sparse(2, 2, (7, 18, 18), 250, 8)
    ks = Z[f"subm{case}.kernel_size"]
    wb = GI.seeded_state([("weight", [*ks, 8, 10]), ("bias", [10])], 220 + case)
    GI.check(Z, f"subm{case}.coors", coors)
    o = SO.subm_conv(feats, coors, 2, [7, 18, 18], wb["weight"], wb["bias"])
    GI.check(Z, f"subm{case}.out", o, rtol=1e-4, atol=1e-5)
    nbr = SO.neighbour_table(coors, coors, 2, [7, 18, 18], ks, [1, 1, 1], [k // 2 for k in ks])
    GI.check(Z, f"subm{case}.out", SO.indice_conv(feats, nbr, wb["weight"], shift=wb["bias"]), rtol=1e-4, atol=1e-5)


def test_simple_sparse_unet_matches_reference(Z):
    U = MG.SPCONV_PIN_UNET
    sd = GI.seeded_state(Z["unet.spec"], 230)
    feats, coors = SO.synth_sparse(4, 2, (9, 32, 32), 500, 8)
    f, c, ms = SO.sparse_unet_forward(sd, feats, coors, 2, U["sparse_shape"], U["encoder_channels"], U["encoder_paddings"],
                                      U["decoder_channels"], U["decoder_paddings"], return_multiscale=True)
    assert torch.equal(c, coors)
    GI.check(Z, "unet.coors", coors)
    GI.check(Z, "unet.out", f, rtol=1e-3, atol=1e-4)
    assert len(ms) == Z["unet.n_levels"] == 4
    for i, (mf, mc) in enumerate(ms):
        of, oc = _by_coor(mf, mc)
        GI.check(Z, f"unet.ms{i}.coors", oc.int())
        GI.check(Z, f"unet.ms{i}.out", of, rtol=1e-3, atol=1e-4)


def test_virtual_voxel_mixer_matches_reference(Z):
    """the mixer's conv_out is SubM kernel 3 / padding 0 on a fresh indice key - still a centred conv"""
    cfg = MG.SPCONV_PIN_MIXER
    sd = GI.seeded_state(Z["mixer.spec"], 240)
    feats, coors = SO.synth_sparse(8, 3, (8, 24, 24), 300, 8)
    f, c = SO.sparse_unet_forward(sd, feats, coors, 3, cfg["sparse_shape"], cfg["encoder_channels"], cfg["encoder_paddings"],
                                  cfg["decoder_channels"], cfg["decoder_paddings"], mixer_out=True)
    GI.check(Z, "mixer.coors", coors)
    assert Z["mixer.spatial_shape"] == cfg["sparse_shape"]
    GI.check(Z, "mixer.out", f, rtol=1e-3, atol=1e-4)
