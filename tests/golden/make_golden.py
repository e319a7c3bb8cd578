"""Generates the committed golden vectors by running the UNMODIFIED reference modules
(imported from /root/reference with the shims of oracle/ref_import.py) on seeded synthetic inputs.
Run in the build container:  python tests/golden/make_golden.py
Inputs are regenerated from their seeds at test time (mfr_b200.synth, oracle.loftr_oracle.make_state_dict
are deterministic); an input checksum is stored next to the reference outputs to detect drift.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import mfr_b200  # noqa: E402,F401
from helpers import METRICS_K, loftr_module_case, metrics_cases, metrics_checksum, spsg_real_cases  # noqa: E402
from mfr_b200 import synth  # noqa: E402
from oracle import ref_import, loftr_oracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

POSE_CASES = [  # seed, n, inlier_ratio, noise_px
    (11, 400, 0.6, 0.3), (12, 800, 0.5, 0.5), (13, 300, 0.8, 0.0), (14, 1000, 0.4, 1.0),
    (15, 4, 1.0, 0.0), (16, 600, 0.7, 0.2),
]
GOLD_H, GOLD_W = 720, 540
GOLD_K = np.array([[600.0, 0, 269.5], [0, 600.0, 359.5], [0, 0, 1]])


def checksum(*arrays):
    return float(sum(np.float64(np.asarray(a, dtype=np.float64)).sum() for a in arrays))


def pose_case(seed, n, ratio, noise):
    return synth.make_correspondences(seed, n=n, inlier_ratio=ratio, noise_px=noise, h=GOLD_H, w=GOLD_W, K=GOLD_K)


def make_pose_golden():
    model = ref_import.load_model_module()
    base = dict(FEATURE_MATCHING="Precomputed", DEBUG=False, MATCHES_FILE_PATH="/tmp/_mfr_gold_corr.npz",
                EMAT_RANSAC=dict(PIX_THRESHOLD=2.0, SCALE_THRESHOLD=0.1, CONFIDENCE=0.9999),
                PNP=dict(RANSAC_ITER=1000, REPROJECTION_INLIER_THRESHOLD=3, CONFIDENCE=0.9999),
                DATASET=dict(PAIRS_TXT=dict(TEST=None)))
    out = {}
    for ci, (seed, n, ratio, noise) in enumerate(POSE_CASES):
        c = pose_case(seed, n, ratio, noise)
        corr = np.concatenate([c["kpts0"], c["kpts1"]], 1)[None].astype(np.float64)
        np.savez_compressed(base["MATCHES_FILE_PATH"], correspondences=corr)
        data0 = {"depth0": torch.from_numpy(c["depth0"])[None], "depth1": torch.from_numpy(c["depth1"])[None],
                 "K_color0": torch.from_numpy(c["K_color0"])[None], "K_color1": torch.from_numpy(c["K_color1"])[None],
                 "pair_id": torch.tensor([0])}
        out[f"c{ci}_checksum"] = checksum(c["kpts0"], c["kpts1"], c["depth0"], c["depth1"])
        for solver in ("EssentialMatrix", "EssentialMatrixMetric", "PNP"):
            cfg = ref_import.Cfg.wrap(dict(base, POSE_SOLVER=solver))
            m = model.FeatureMatchingModel(cfg)
            data = dict(data0)
            R, t = m(data)
            out[f"c{ci}_{solver}_R"] = R[0].numpy()
            out[f"c{ci}_{solver}_t"] = t[0, 0].numpy()
            out[f"c{ci}_{solver}_inliers"] = np.int64(data["inliers"])
            if solver == "EssentialMatrix":
                mask = getattr(m.pose_solver, "mask", None)
                out[f"c{ci}_emat_mask"] = (np.zeros(0, np.uint8) if mask is None else mask.ravel().astype(np.uint8))
    np.savez_compressed(os.path.join(HERE, "pose_solver_reference.npz"), **out)
    print("pose golden:", len(out), "arrays")


def make_loftr_golden():
    LoFTR, default_cfg = ref_import.load_loftr()
    sd = loftr_oracle.make_state_dict(0)
    m = LoFTR(config=default_cfg).eval()
    m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=False)
    out = {}
    for ci, (pair, thr, same) in enumerate([(0, 0.0, True), (1, 0.0, False)]):
        p = synth.make_pair(pair)
        g0 = synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0
        g1 = synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0
        H, W = 128, 96
        i0 = torch.from_numpy(g0[100:100 + H, 100:100 + W].copy())[None, None]
        i1 = torch.from_numpy((g0[108:108 + H, 116:116 + W] if same else g1[100:100 + H, 100:100 + W]).copy())[None, None]
        m.coarse_matching.thr = thr
        with torch.no_grad():
            b = {"image0": i0, "image1": i1}
            m(b)
        out[f"c{ci}_checksum"] = checksum(i0.numpy(), i1.numpy())
        out[f"c{ci}_conf_sum"] = np.float64(b["conf_matrix"].double().sum().item())
        out[f"c{ci}_conf_sample"] = b["conf_matrix"][0, ::7, ::5].numpy()
        for k in ("i_ids", "j_ids", "mconf", "mkpts0_f", "mkpts1_f", "expec_f"):
            out[f"c{ci}_{k}"] = b[k].numpy()
    np.savez_compressed(os.path.join(HERE, "loftr_reference.npz"), **out)
    print("loftr golden:", len(out), "arrays; M =", [len(out[f'c{i}_i_ids']) for i in range(2)])


FULLRES_CASES = [("dense", 0.0), ("functional", 0.2), ("functional_dense", 0.2)]   # weights, coarse threshold
FUNCTIONAL_DENSE_NOISE = 1e-3                            # bench.py's throughput weights (loftr.functional_state_dict(noise=...))
FULLRES_SEEDS = (1000, 1001)                             # the first two pairs of bench.py's pool


def fullres_inputs():
    """Two 720x540 synthetic pairs exactly as bench.py feeds them (gray float32 / 255), [2,1,720,540] each."""
    g0, g1 = [], []
    for sd_ in FULLRES_SEEDS:
        p = synth.make_pair(sd_)
        g0.append(synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0)
        g1.append(synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0)
    return torch.from_numpy(np.stack(g0))[:, None], torch.from_numpy(np.stack(g1))[:, None]


def fullres_state_dict(kind):
    from mfr_b200 import loftr
    if kind == "dense":
        return loftr_oracle.make_state_dict(0)
    return loftr.functional_state_dict(noise=FUNCTIONAL_DENSE_NOISE if kind == "functional_dense" else 0.0)


def make_loftr_fullres_golden():
    """BASELINE configuration (540x720 -> 720x544 after the reference's pad, L = 6120 coarse cells), the UNMODIFIED
    reference LoFTR on CPU fp32, one pair per forward (the reference's batch size). Two weight sets: dense seeded
    random weights (coarse threshold 0: every mutual nearest neighbour is a match) and the functional weights the
    benchmark's accuracy block uses (reference threshold 0.2), plain and with the dense perturbation of the throughput run."""
    from mfr_b200 import loftr
    LoFTR, default_cfg = ref_import.load_loftr()
    i0, i1 = fullres_inputs()
    out = {"checksum": checksum(i0.numpy(), i1.numpy())}
    for kind, thr in FULLRES_CASES:
        sd = fullres_state_dict(kind)
        m = LoFTR(config=default_cfg).eval()
        m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=False)
        m.coarse_matching.thr = thr
        cap = {}
        m.loftr_coarse.register_forward_hook(lambda mod, inp, outp: cap.__setitem__("c", outp))   # (feat_c0, feat_c1)
        for b in range(i0.shape[0]):
            d = {"image0": loftr.pad_to_8(i0[b:b + 1]), "image1": loftr.pad_to_8(i1[b:b + 1])}
            with torch.no_grad():
                m(d)
            pre = f"{kind}_p{b}_"
            out[pre + "i_ids"] = d["i_ids"].numpy().astype(np.int32)
            out[pre + "j_ids"] = d["j_ids"].numpy().astype(np.int32)
            out[pre + "mconf"] = d["mconf"].numpy()
            out[pre + "mkpts1_f"] = d["mkpts1_f"].numpy()
            out[pre + "conf_sample"] = d["conf_matrix"][0, ::97, ::89].numpy()
            out[pre + "feat_c0_sample"] = cap["c"][0][0, ::61, ::8].numpy()       # coarse tokens after the transformer
            out[pre + "feat_c1_sample"] = cap["c"][1][0, ::61, ::8].numpy()
            print(f"fullres golden {kind} pair {b}: M = {len(d['i_ids'])}, conf max {d['conf_matrix'].max().item():.4g}")
    np.savez_compressed(os.path.join(HERE, "loftr_fullres_reference.npz"), **out)


def spsg_case():
    p = synth.make_pair(5)
    g0 = synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0
    return (torch.from_numpy(g0[40:280, 30:350].copy())[None, None], torch.from_numpy(g0[48:288, 46:366].copy())[None, None])


def make_spsg_golden():
    """Reference SuperPoint/SuperGlue modules with the synthetic seeded weights loaded over the
    in-tree ones (same architecture), settings of matchers.py:65-71 except max_keypoints 256 and
    match_threshold 0 (so that the tiny synthetic case has matches)."""
    from mfr_b200 import spsg
    SuperPoint, SuperGlue, Matching = ref_import.load_superglue()
    sp_sd, sg_sd = spsg.synthetic_state_dicts(0)
    m = Matching({"superpoint": {"nms_radius": 4, "keypoint_threshold": 0.005, "max_keypoints": 256},
                  "superglue": {"weights": "indoor", "sinkhorn_iterations": 20, "match_threshold": 0.0}}).eval()
    m.superpoint.load_state_dict(sp_sd)
    m.superglue.load_state_dict(sg_sd)
    i0, i1 = spsg_case()
    with torch.no_grad():
        pred = m({"image0": i0, "image1": i1})
    out = {"checksum": checksum(i0.numpy(), i1.numpy())}
    for k in ("keypoints0", "keypoints1", "scores0", "scores1", "matches0", "matching_scores0"):
        out[k] = pred[k][0].numpy()
    out["descriptors0_sample"] = pred["descriptors0"][0][::8, ::4].numpy()
    np.savez_compressed(os.path.join(HERE, "spsg_reference.npz"), **out)
    print("spsg golden: kpts", out["keypoints0"].shape, out["keypoints1"].shape, "matches", int((out["matches0"] > -1).sum()))


def make_spsg_real_golden():
    """UNMODIFIED reference Matching (SuperPoint + SuperGlue) with the in-tree weights and the settings of
    etc/feature_matching_baselines/matchers.py:65-71."""
    from oracle import build_ref
    assert build_ref.build(verbose=False)
    SuperPoint, SuperGlue, Matching = ref_import.load_superglue()
    m = Matching({"superpoint": {"nms_radius": 4, "keypoint_threshold": 0.005, "max_keypoints": 1024},
                  "superglue": {"weights": "indoor", "sinkhorn_iterations": 20, "match_threshold": 0.2}}).eval()
    out = {}
    for name, i0, i1 in spsg_real_cases():
        with torch.no_grad():
            pred = m({"image0": i0, "image1": i1})
        out[name + "_checksum"] = checksum(i0.numpy(), i1.numpy())
        for k in ("keypoints0", "keypoints1", "scores0", "scores1", "matches0", "matching_scores0"):
            out[f"{name}_{k}"] = pred[k][0].numpy()
        out[f"{name}_descriptors0_sample"] = pred["descriptors0"][0][::8, ::4].numpy()
        print(f"spsg real-weights golden {name}: keypoints {len(out[name + '_keypoints0'])} / {len(out[name + '_keypoints1'])},"
              f" matches {int((out[name + '_matches0'] > -1).sum())}")
    np.savez_compressed(os.path.join(HERE, "spsg_real_reference.npz"), **out)


def make_loftr_module_golden():
    """The reference LoFTR module with seeded weights (make_state_dict(3)) at coarse threshold 0: the full
    confidence matrix and the matches."""
    LoFTR, default_cfg = ref_import.load_loftr()
    sd = loftr_oracle.make_state_dict(3)
    m = LoFTR(config=default_cfg).eval()
    m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=False)
    m.coarse_matching.thr = 0.0
    i0, i1 = loftr_module_case()
    with torch.no_grad():
        b = {"image0": i0, "image1": i1}
        m(b)
    out = {"checksum": checksum(i0.numpy(), i1.numpy()), "conf_matrix": b["conf_matrix"].numpy()}
    for k in ("i_ids", "j_ids", "mkpts1_f"):
        out[k] = b[k].numpy()
    np.savez_compressed(os.path.join(HERE, "loftr_module_reference.npz"), **out)
    print("loftr module golden: M =", len(out["i_ids"]))


def make_metrics_golden():
    """The reference's benchmark/metrics.py MetricManager and benchmark/utils.py precision_recall on
    metrics_cases(); transforms3d (not installed) is stood in for by the oracle's restatement of the four
    quaternion helpers it provides."""
    import types
    from oracle import metrics_oracle as mo
    t3d = types.ModuleType("transforms3d"); tq = types.ModuleType("transforms3d.quaternions"); te = types.ModuleType("transforms3d.euler")
    for n in ("quat2mat", "qmult", "qinverse", "rotate_vector", "axangle2quat"):
        setattr(tq, n, getattr(mo, n))
    te.euler2quat = mo.euler2quat
    t3d.quaternions, t3d.euler = tq, te
    sys.modules.update({"transforms3d": t3d, "transforms3d.quaternions": tq, "transforms3d.euler": te})
    sys.path.insert(0, ref_import.REF)
    from benchmark.metrics import Inputs, MetricManager
    from benchmark.utils import precision_recall
    cases = metrics_cases()
    res = {"trans_err": [], "rot_err": [], "reproj_err": [], "confidence": []}
    mm = MetricManager()
    for qg, tg, qe, te_, conf in cases:
        mm(Inputs(q_gt=qg, t_gt=tg, q_est=qe, t_est=te_, confidence=conf, K=METRICS_K, W=540, H=720), res)
    out = {k: np.asarray(v, np.float64) for k, v in res.items()}
    out["checksum"] = metrics_checksum(cases)
    tp = (out["trans_err"] < 0.25) * (out["rot_err"] < 5)
    out["precision"], out["recall"], out["ap"] = [np.asarray(x, np.float64) for x in precision_recall(out["confidence"].tolist(), tp, 3)]
    np.savez_compressed(os.path.join(HERE, "metrics_reference.npz"), **out)
    print("metrics golden:", len(cases), "poses, AP", float(out["ap"]))


README_PAIR = ("scene0711_00_frame-001680.jpg", "scene0711_00_frame-001995.jpg")


def make_readme_pair_fixtures():
    """The SuperGlue README's ScanNet sample pair (1296x968 camera JPEGs), re-encoded at quality 75 to keep the
    repository small; they exercise the GPU JPEG loader on real photographs."""
    import cv2
    src = os.path.join(ref_import.FMB, "SuperGlue", "assets", "scannet_sample_images")
    for n in README_PAIR:
        im = cv2.imread(os.path.join(src, n), cv2.IMREAD_COLOR)
        assert cv2.imwrite(os.path.join(HERE, n), im, [cv2.IMWRITE_JPEG_QUALITY, 75])
    print("readme pair fixtures:", ", ".join(README_PAIR))


if __name__ == "__main__":
    assert ref_import.available(), "needs the reference tree (MFR_REFERENCE)"
    which = sys.argv[1:] or ["pose", "loftr", "fullres", "spsg", "spsg_real", "loftr_module", "metrics", "images"]
    if "pose" in which:
        make_pose_golden()
    if "loftr" in which:
        make_loftr_golden()
    if "fullres" in which:
        make_loftr_fullres_golden()
    if "spsg" in which:
        make_spsg_golden()
    if "spsg_real" in which:
        make_spsg_real_golden()
    if "loftr_module" in which:
        make_loftr_module_golden()
    if "metrics" in which:
        make_metrics_golden()
    if "images" in which:
        make_readme_pair_fixtures()
