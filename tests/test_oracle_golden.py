"""Pins the oracle restatements (oracle/) against vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py imports it from /root/reference in the build container). CPU only."""
import numpy as np
import pytest
import torch

from helpers import GOLDEN, POSE_CASES, checksum, loftr_case, pose_case
from oracle import loftr_oracle, pose_solver_oracle as po

G = np.load(GOLDEN + "/pose_solver_reference.npz")
GL = np.load(GOLDEN + "/loftr_reference.npz")


@pytest.mark.parametrize("ci", range(len(POSE_CASES)))
def test_pose_solver_oracle_reproduces_reference(ci):
    c = pose_case(ci)
    assert checksum(c["kpts0"], c["kpts1"], c["depth0"], c["depth1"]) == pytest.approx(float(G[f"c{ci}_checksum"]), rel=0, abs=1e-6), \
        "synthetic input drifted from the one the golden vectors were generated on"
    args = (c["kpts0"], c["kpts1"])
    K0, K1 = c["K_color0"], c["K_color1"]
    R, t, n, mask = po.essential_matrix_solver(*args, K0, K1, 2.0, 0.9999)
    np.testing.assert_allclose(np.float32(R), G[f"c{ci}_EssentialMatrix_R"], atol=1e-6, equal_nan=True)
    np.testing.assert_allclose(np.float32(t).ravel(), G[f"c{ci}_EssentialMatrix_t"], atol=1e-6, equal_nan=True)
    assert n == int(G[f"c{ci}_EssentialMatrix_inliers"])
    if mask is not None:
        np.testing.assert_array_equal(mask.ravel().astype(np.uint8), G[f"c{ci}_emat_mask"])
    R, t, n = po.essential_matrix_metric_solver(*args, c["depth0"], c["depth1"], K0, K1, 2.0, 0.9999, 0.1)
    np.testing.assert_allclose(np.float32(R), G[f"c{ci}_EssentialMatrixMetric_R"], atol=1e-6, equal_nan=True)
    np.testing.assert_allclose(np.float32(t).ravel(), G[f"c{ci}_EssentialMatrixMetric_t"], atol=1e-6, equal_nan=True)
    assert n == int(G[f"c{ci}_EssentialMatrixMetric_inliers"])
    R, t, n = po.pnp_solver(*args, c["depth0"], K0, K1, 1000, 3, 0.9999)
    np.testing.assert_allclose(np.float32(R), G[f"c{ci}_PNP_R"], atol=1e-6, equal_nan=True)
    np.testing.assert_allclose(np.float32(t).ravel(), G[f"c{ci}_PNP_t"], atol=1e-6, equal_nan=True)
    assert n == int(G[f"c{ci}_PNP_inliers"])


@pytest.mark.parametrize("ci", range(2))
def test_loftr_oracle_reproduces_reference(ci):
    i0, i1, thr = loftr_case(ci)
    assert checksum(i0.numpy(), i1.numpy()) == pytest.approx(float(GL[f"c{ci}_checksum"]), abs=1e-6)
    sd = loftr_oracle.make_state_dict(0)
    with torch.no_grad():
        o = loftr_oracle.loftr_forward(i0, i1, sd, {"thr": thr}, True)
    np.testing.assert_allclose(o["conf"][0, ::7, ::5].numpy(), GL[f"c{ci}_conf_sample"], rtol=1e-5, atol=1e-12)
    np.testing.assert_array_equal(o["i_ids"].numpy(), GL[f"c{ci}_i_ids"])   # integer outputs: bit-exact
    np.testing.assert_array_equal(o["j_ids"].numpy(), GL[f"c{ci}_j_ids"])
    np.testing.assert_allclose(o["mconf"].numpy(), GL[f"c{ci}_mconf"], rtol=1e-5)
    np.testing.assert_array_equal(o["mkpts0_f"].numpy(), GL[f"c{ci}_mkpts0_f"])
    np.testing.assert_allclose(o["mkpts1_f"].numpy(), GL[f"c{ci}_mkpts1_f"], atol=2e-4)  # pixels
    np.testing.assert_allclose(o["expec_f"].numpy(), GL[f"c{ci}_expec_f"], atol=1e-4)


def test_spsg_oracle_reproduces_reference():
    """SuperPoint + SuperGlue restatement vs the reference modules (synthetic seeded weights)."""
    from mfr_b200 import spsg, synth
    from oracle import spsg_oracle as so
    GS = np.load(GOLDEN + "/spsg_reference.npz")
    p = synth.make_pair(5)
    g0 = synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0
    i0 = torch.from_numpy(g0[40:280, 30:350].copy())[None, None]
    i1 = torch.from_numpy(g0[48:288, 46:366].copy())[None, None]
    assert checksum(i0.numpy(), i1.numpy()) == pytest.approx(float(GS["checksum"]), abs=1e-6)
    sp, sg = spsg.synthetic_state_dicts(0)
    cfg = {"max_keypoints": 256, "match_threshold": 0.0}
    with torch.no_grad():
        k0, s0, d0 = so.superpoint(i0, sp, cfg)
        k1, s1, d1 = so.superpoint(i1, sp, cfg)
        m0, ms0, _, Z = so.superglue(k0, s0, d0, k1, s1, d1, 240, 320, sg, cfg, return_scores=True)
    np.testing.assert_array_equal(k0.numpy(), GS["keypoints0"])      # integer-valued keypoints: exact
    np.testing.assert_array_equal(k1.numpy(), GS["keypoints1"])
    np.testing.assert_allclose(s0.numpy(), GS["scores0"], rtol=1e-5)
    np.testing.assert_allclose(d0[::8, ::4].numpy(), GS["descriptors0_sample"], atol=1e-5)
    # integer matches: exact, except where the mutual-nearest-neighbour decision is a float32 tie. With random weights a
    # row or column of the log-assignment can hold two entries a few ulps apart (column 26 here: 1.9e-6), and the fp32
    # network rounds differently on CPUs with other vector instruction sets than the one the vectors were made on.
    dec = _decided(Z, 1e-5)
    assert dec.mean() > 0.97
    np.testing.assert_array_equal(m0.numpy()[dec], GS["matches0"][dec])
    np.testing.assert_allclose(ms0.numpy()[dec], GS["matching_scores0"][dec], atol=1e-5)


def _decided(Z, eps):
    """Rows of a SuperGlue log-assignment matrix (with dustbins) whose mutual-nearest-neighbour decision holds under
    perturbations below eps: the two best entries of the row, and of the column holding the row's best, differ by more."""
    P = Z[:-1, :-1]
    r2, c2 = P.topk(2, dim=1).values, P.topk(2, dim=0).values
    return (((r2[:, 0] - r2[:, 1]) > eps) & ((c2[0] - c2[1])[P.argmax(1)] > eps)).numpy()
