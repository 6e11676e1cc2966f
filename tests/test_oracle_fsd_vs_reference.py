"""CPU: oracle/fsd_oracle.py (FSD instance grouping, SURVEY 8f next-3) against what the reference's own functions and ClusterAssigner class
(compiled from mmdet3d/models/detectors/single_stage_fsd.py, unmodified source, by oracle/ref_shim.reference_functions) returned on the
same seeded inputs - recorded bit-exactly in tests/golden/ref_fsd_pins.npz by `python -m oracle.make_golden pins`."""
import os

import pytest
import torch

from oracle import fsd_oracle as FO, golden_io as GI, make_golden as MG


@pytest.fixture(scope="module")
def Z():
    return GI.load(os.path.join(os.path.dirname(__file__), "golden", "ref_fsd_pins.npz"))


@pytest.mark.parametrize("dist", [0.1, 0.6, 2.0])
def test_connected_components_match_reference(Z, dist):
    pts, bidx = FO.synth_centres(3, 3, 700)
    GI.check(Z, f"cc.{dist}", FO.find_connected_components(pts, bidx, dist))
    GI.check(Z, f"cc.{dist}", FO.connected_components_large(pts, bidx, dist))
    GI.check(Z, f"cc_single.{dist}", FO.find_connected_components(pts[:700], torch.zeros(700, dtype=torch.int32), dist))


def test_cluster_assigner_matches_reference(Z):
    cfg = MG.FSD_CA_CFG
    pts_l, b_l = MG.pin_cluster_inputs()   # the batched scipy branch of ClusterAssigner in train() (single_stage_fsd.py:984-985)
    for i, name in enumerate(cfg["class_names"]):
        o_inds, o_mask = FO.cluster_assigner_single_class(pts_l[i], b_l[i], cfg["cluster_voxel_size"][name], 2, cfg["point_cloud_range"],
                                                          cfg["connected_dist"][name])
        GI.check(Z, f"ca.mask{i}", o_mask)
        GI.check(Z, f"ca.class{i}", torch.full((o_inds.shape[0],), i, dtype=torch.long))
        GI.check(Z, f"ca.inds{i}", o_inds.int())
    m0 = b_l[0] == 0   # eval branch: find_connected_componets_single_batch on a one-sample batch
    o_inds, _ = FO.cluster_assigner_single_class(pts_l[0][m0], b_l[0][m0], cfg["cluster_voxel_size"]["Car"], 2, cfg["point_cloud_range"], 0.6,
                                                 single_batch=True)
    GI.check(Z, "ca.eval_inds", o_inds.int())
