"""The metrics oracle (oracle/metrics_oracle.py) against the reference's OWN tests for this code
(benchmark/test_metrics.py: properties of trans_err / rot_err / reproj_err and the known-answer vectors of
test_projection, replayed here with seeded randomness), and against stored outputs of the reference module itself on
random poses (tests/golden/make_golden.py; transforms3d, which the reference imports, is stood in for there by the
oracle's restatement of its four quaternion helpers)."""
import numpy as np
import pytest

from helpers import GOLDEN, METRICS_K, metrics_cases, metrics_checksum
from oracle import metrics_oracle as mo

K0 = METRICS_K


def _rq(rng):
    return mo.euler2quat(*rng.uniform(0, 2 * np.pi, 3))


def test_reference_test_vectors_projection():            # benchmark/test_metrics.py:188-199
    xyz = np.array(((10, 20, 30), (10, 30, 50), (-20, -15, 5), (-20, -50, 10)), dtype=np.float32)
    uv = np.array(((1 / 3, 2 / 3), (1 / 5, 3 / 5), (-4, -3), (-2, -5)), dtype=np.float32)
    assert np.allclose(uv, mo.project(xyz, np.eye(3)))
    uv = np.array(((1 / 3, 2 / 3), (1 / 5, 3 / 5), (0, 0), (0, 0)), dtype=np.float32)
    assert np.allclose(uv, mo.project(xyz, np.eye(3), img_size=(5, 5)))


def test_reference_properties():
    rng = np.random.default_rng(0)
    for _ in range(50):
        t0, d = rng.normal(5, 10, 3), rng.normal(5, 10, 3)          # test_t_err_tinvariance
        q = _rq(rng)
        m = mo.pose_metrics(q, t0, q, t0 + d, K0, 540, 720)
        assert np.isclose(m["trans_err"], np.linalg.norm(d))
        axis = rng.uniform(-1, 1, 3); ang = rng.uniform(-np.pi, np.pi)      # test_rot_err_raxis
        qres = mo.axangle2quat(axis, ang)
        assert np.isclose(mo.quat_angle_error(label=mo.qmult(q, qres), pred=q), abs(np.degrees(ang)), rtol=1e-5, atol=1e-8)
        q1 = _rq(rng)                                                       # test_r_err_mat
        Rres = mo.quat2mat(q1) @ mo.quat2mat(q).T
        assert np.isclose(np.degrees(np.arccos(np.clip((np.trace(Rres) - 1) / 2, -1, 1))), mo.quat_angle_error(label=q1, pred=q))
    q, t = _rq(rng), rng.normal(0, 10, 3)                                   # test_reproj_error_identity
    assert np.isclose(mo.reprojection_error(q, t, q, t, np.eye(3), 1, 1), 0)
    for scale in np.logspace(-1, -9, 9):                                    # test_r_err_small
        q = _rq(rng); ang = rng.uniform(-np.pi, np.pi) * scale
        e = mo.quat_angle_error(label=mo.qmult(q, mo.axangle2quat(rng.uniform(-1, 1, 3), ang)), pred=q)
        assert np.isclose(e, abs(np.degrees(ang)), rtol=0.1 * scale, atol=0.1 * scale)


def test_precision_recall_small_case():
    # 4 estimates + 1 failure; confidences 9, 7, 7, 2; true positives 1, 0, 1, 1
    prec, rec, ap = mo.precision_recall([7, 9, 2, 7], [0, 1, 1, 1], 1)
    assert np.allclose(rec, [0.8, 0.6, 0.2, 0.0]) and np.allclose(prec, [0.75, 2 / 3, 1.0, 1.0])
    assert np.isclose(ap, 0.2 * 0.75 + 0.4 * 2 / 3 + 0.2 * 1.0)


def test_oracle_equals_reference_module():
    """benchmark/metrics.py MetricManager and benchmark/utils.py precision_recall of the reference, stored in
    tests/golden/metrics_reference.npz, against the oracle on the same 40 seeded poses."""
    G = np.load(GOLDEN + "/metrics_reference.npz")
    cases = metrics_cases()
    assert metrics_checksum(cases) == pytest.approx(float(G["checksum"]), rel=1e-12)
    ours = {k: [] for k in ("trans_err", "rot_err", "reproj_err", "confidence")}
    for qg, tg, qe, te_, conf in cases:
        m = mo.pose_metrics(qg, tg, qe, te_, K0, 540, 720)
        for k in ("trans_err", "rot_err", "reproj_err"):
            ours[k].append(m[k])
        ours["confidence"].append(conf)
    for k in ours:
        assert np.allclose(G[k], ours[k], rtol=1e-10, atol=1e-10), k
    tp = (np.array(ours["trans_err"]) < 0.25) * (np.array(ours["rot_err"]) < 5)
    b = mo.precision_recall(ours["confidence"], tp, 3)
    assert np.allclose(G["precision"], b[0]) and np.allclose(G["recall"], b[1]) and np.isclose(G["ap"], b[2])
