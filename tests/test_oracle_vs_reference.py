"""The oracle restatements against outputs of the reference modules themselves, stored under tests/golden/
(tests/golden/make_golden.py regenerates them from the reference tree)."""
import numpy as np
import pytest
import torch

from helpers import GOLDEN, checksum, loftr_module_case, pose_case, spsg_real_cases
from oracle import build_ref, loftr_oracle, pose_solver_oracle as po


def test_pose_solver_module_matches_oracle():
    """The reference's FeatureMatchingModel (precomputed matches) with the metric essential-matrix and the PnP solver."""
    G = np.load(GOLDEN + "/pose_solver_reference.npz")
    c = pose_case(1)
    assert checksum(c["kpts0"], c["kpts1"], c["depth0"], c["depth1"]) == pytest.approx(float(G["c1_checksum"]), rel=0, abs=1e-6)
    for solver in ("EssentialMatrixMetric", "PNP"):
        if solver == "PNP":
            Ro, to, no = po.pnp_solver(c["kpts0"], c["kpts1"], c["depth0"], c["K_color0"], c["K_color1"], 1000, 3, 0.9999)
        else:
            Ro, to, no = po.essential_matrix_metric_solver(c["kpts0"], c["kpts1"], c["depth0"], c["depth1"],
                                                           c["K_color0"], c["K_color1"], 2.0, 0.9999, 0.1)
        np.testing.assert_allclose(G[f"c1_{solver}_R"], np.float32(Ro), atol=1e-6)
        np.testing.assert_allclose(G[f"c1_{solver}_t"], np.float32(to).ravel(), atol=1e-6)
        assert int(G[f"c1_{solver}_inliers"]) == no


def test_loftr_module_matches_oracle():
    G = np.load(GOLDEN + "/loftr_module_reference.npz")
    sd = loftr_oracle.make_state_dict(3)
    i0, i1 = loftr_module_case()
    assert checksum(i0.numpy(), i1.numpy()) == pytest.approx(float(G["checksum"]), abs=1e-6)
    with torch.no_grad():
        o = loftr_oracle.loftr_forward(i0, i1, sd, {"thr": 0.0}, True)
    np.testing.assert_array_equal(o["i_ids"].numpy(), G["i_ids"])
    np.testing.assert_array_equal(o["j_ids"].numpy(), G["j_ids"])
    torch.testing.assert_close(torch.from_numpy(G["conf_matrix"]), o["conf"], rtol=1e-5, atol=1e-12)
    torch.testing.assert_close(torch.from_numpy(G["mkpts1_f"]), o["mkpts1_f"], atol=2e-4, rtol=0)


@pytest.mark.skipif(not build_ref.available(), reason="the reference's pretrained SuperPoint / SuperGlue weights are not staged in oracle/_ref")
def test_spsg_modules_match_oracle_with_real_weights():
    """The pretrained SuperPoint/SuperGlue weights on the reference README's known-answer ScanNet pair
    (SuperGlue/README.md:121-127): identical keypoints, descriptors and matches."""
    from oracle import spsg_oracle as so
    G = np.load(GOLDEN + "/spsg_real_reference.npz")
    wdir = build_ref.weights_dir()
    sp_sd = torch.load(wdir + "/superpoint_v1.pth", map_location="cpu")
    sg_sd = torch.load(wdir + "/superglue_indoor.pth", map_location="cpu")
    name, i0, i1 = spsg_real_cases()[0]
    assert name == "readme"
    assert checksum(i0.numpy(), i1.numpy()) == pytest.approx(float(G["readme_checksum"]), rel=1e-6)
    with torch.no_grad():
        k0, s0, d0 = so.superpoint(i0, sp_sd)
        k1, s1, d1 = so.superpoint(i1, sp_sd)
        m0, ms0 = so.superglue(k0, s0, d0, k1, s1, d1, 480, 640, sg_sd)
    np.testing.assert_array_equal(k0.numpy(), G["readme_keypoints0"])
    np.testing.assert_array_equal(k1.numpy(), G["readme_keypoints1"])
    np.testing.assert_allclose(d0[::8, ::4].numpy(), G["readme_descriptors0_sample"], atol=1e-6, rtol=0)
    np.testing.assert_array_equal(m0.numpy(), G["readme_matches0"])
    assert int((m0 > -1).sum()) > 100
    # the stored scores may come from a CPU with other vector instructions: after 18 attention layers and 20 Sinkhorn
    # iterations in fp32 they differ by up to 1.0e-5 across such hosts (they are bit-identical on the host that made them)
    np.testing.assert_allclose(ms0.numpy(), G["readme_matching_scores0"], atol=2e-5, rtol=0)
