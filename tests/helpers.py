import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

import mfr_b200  # noqa: E402,F401
from mfr_b200 import synth  # noqa: E402

POSE_CASES = [(11, 400, 0.6, 0.3), (12, 800, 0.5, 0.5), (13, 300, 0.8, 0.0), (14, 1000, 0.4, 1.0),
              (15, 4, 1.0, 0.0), (16, 600, 0.7, 0.2)]
GOLD_H, GOLD_W = 720, 540
GOLD_K = np.array([[600.0, 0, 269.5], [0, 600.0, 359.5], [0, 0, 1]])


def pose_case(ci):
    seed, n, ratio, noise = POSE_CASES[ci]
    return synth.make_correspondences(seed, n=n, inlier_ratio=ratio, noise_px=noise, h=GOLD_H, w=GOLD_W, K=GOLD_K)


def checksum(*arrays):
    return float(sum(np.float64(np.asarray(a, dtype=np.float64)).sum() for a in arrays))


def loftr_case(ci):
    import torch
    pair, thr, same = [(0, 0.0, True), (1, 0.0, False)][ci]
    p = synth.make_pair(pair)
    g0 = synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0
    g1 = synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0
    H, W = 128, 96
    i0 = torch.from_numpy(g0[100:100 + H, 100:100 + W].copy())[None, None]
    i1 = torch.from_numpy((g0[108:108 + H, 116:116 + W] if same else g1[100:100 + H, 100:100 + W]).copy())[None, None]
    return i0, i1, thr


def rot_angle(Ra, Rb):
    c = (np.trace(np.asarray(Ra, dtype=np.float64) @ np.asarray(Rb, dtype=np.float64).T) - 1.0) / 2.0
    return float(np.arccos(np.clip(c, -1.0, 1.0)))


def vec_angle(a, b):
    a = np.asarray(a, dtype=np.float64).ravel(); b = np.asarray(b, dtype=np.float64).ravel()
    return float(np.arccos(np.clip(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)), -1.0, 1.0)))


def loftr_module_case():
    """Seeded 96x64 input and its shifted copy (tests/golden/make_golden.py: make_loftr_module_golden)."""
    import torch
    g = torch.Generator().manual_seed(5)
    i0 = torch.rand(1, 1, 96, 64, generator=g)
    return i0, torch.roll(i0, (8, 8), (2, 3))


METRICS_K = np.array([[590.0, 0, 270.0], [0, 590.0, 360.0], [0, 0, 1]])


def metrics_cases():
    """40 seeded (q_gt, t_gt, q_est, t_est, confidence) pose estimates around ground truth, drawn with the oracle's
    restatement of the transforms3d helpers (tests/golden/make_golden.py: make_metrics_golden)."""
    from oracle import metrics_oracle as mo
    rng = np.random.default_rng(1)
    cases = []
    for _ in range(40):
        qg = mo.euler2quat(*rng.uniform(0, 2 * np.pi, 3))
        qe = mo.qmult(qg, mo.axangle2quat(rng.uniform(-1, 1, 3), rng.uniform(0, 0.3)))
        tg = rng.normal(0, 1, 3)
        te = tg + rng.normal(0, 0.2, 3)
        cases.append((qg, tg, qe, te, float(rng.integers(0, 50))))
    return cases


def metrics_checksum(cases):
    return checksum(*[np.concatenate([qg, tg, qe, te, [conf]]) for qg, tg, qe, te, conf in cases])


# ---- BASELINE-configuration LoFTR case (tests/golden/make_golden.py: make_loftr_fullres_golden) ----
FULLRES_CASES = [("dense", 0.0), ("functional", 0.2), ("functional_dense", 0.2)]
FULLRES_SEEDS = (1000, 1001)
FUNCTIONAL_DENSE_NOISE = 1e-3


def fullres_inputs():
    import torch
    g0, g1 = [], []
    for sd_ in FULLRES_SEEDS:
        p = synth.make_pair(sd_)
        g0.append(synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0)
        g1.append(synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0)
    return torch.from_numpy(np.stack(g0))[:, None], torch.from_numpy(np.stack(g1))[:, None]


def fullres_state_dict(kind):
    from mfr_b200 import loftr
    if kind == "dense":
        from oracle import loftr_oracle
        return loftr_oracle.make_state_dict(0)
    return loftr.functional_state_dict(noise=FUNCTIONAL_DENSE_NOISE if kind == "functional_dense" else 0.0)


def fullres_compare(kind, thr, precision, graph=False):
    """Runs the CUDA engine (B = 2, 720x544 frame) on the golden inputs and compares with the vectors of the
    unmodified reference. Returns one dict per pair: M_ref, M_gpu, iou (match set), mkpts1_max_px (on the common
    matches), mconf_max_abs, conf_max_abs (subsampled confidence matrix), tok_rel (coarse tokens after the transformer)."""
    import torch
    from mfr_b200 import loftr
    G = np.load(os.path.join(GOLDEN, "loftr_fullres_reference.npz"))
    i0, i1 = fullres_inputs()
    assert abs(checksum(i0.numpy(), i1.numpy()) - float(G["checksum"])) < 1e-6 * abs(float(G["checksum"])), "synthetic inputs drifted"
    B = i0.shape[0]
    eng = loftr.LoFTR(fullres_state_dict(kind), batch=B, height=720, width=544, cfg={"thr": thr}, graph=graph, precision=precision)
    out = eng.forward(i0.cuda(), i1.cuda())
    L = 90 * 68
    sim = eng.debug_tensor("sim", (B, L, L))
    tok = eng.debug_tensor("tok", (2 * B, L, 512))
    res = []
    for b in range(B):
        pre = f"{kind}_p{b}_"
        sel = (out["b_ids"] == b).nonzero().flatten().cpu()
        gi, gj = out["i_ids"].cpu()[sel].tolist(), out["j_ids"].cpu()[sel].tolist()
        ref = {k: n for n, k in enumerate(zip(G[pre + "i_ids"].tolist(), G[pre + "j_ids"].tolist()))}
        got = {k: int(sel[n]) for n, k in enumerate(zip(gi, gj))}
        common = sorted(set(ref) & set(got))
        r = {"M_ref": len(ref), "M_gpu": len(got), "iou": len(common) / max(1, len(set(ref) | set(got)))}
        if common:
            ig = torch.tensor([got[k] for k in common]); ir = np.array([ref[k] for k in common])
            r["mkpts1_max_px"] = float(np.abs(out["mkpts1_f"].cpu().numpy()[ig] - G[pre + "mkpts1_f"][ir]).max())
            r["mconf_max_abs"] = float(np.abs(out["mconf"].cpu().numpy()[ig] - G[pre + "mconf"][ir]).max())
        s = sim[b]
        conf = (torch.softmax(s, 0) * torch.softmax(s, 1))[::97, ::89].cpu().numpy()
        r["conf_max_abs"] = float(np.abs(conf - G[pre + "conf_sample"]).max())
        t0 = tok[b, ::61, :256:8].cpu().numpy(); t1 = tok[B + b, ::61, :256:8].cpu().numpy()
        r["tok_rel"] = float(max(np.abs(t0 - G[pre + "feat_c0_sample"]).max() / np.abs(G[pre + "feat_c0_sample"]).max(),
                                 np.abs(t1 - G[pre + "feat_c1_sample"]).max() / np.abs(G[pre + "feat_c1_sample"]).max()))
        res.append(r)
    eng.close()
    del sim, tok
    torch.cuda.empty_cache()
    return res


# ---- real-weights SuperPoint + SuperGlue cases (tests/golden/make_golden.py: make_spsg_real_golden) ----
def spsg_real_cases():
    """(name, image0, image1 [1,1,H,W] float32) for the real-weights SuperPoint+SuperGlue golden: the SuperGlue README's
    known-answer ScanNet pair at 640x480 (README.md:121-127) and the first synthetic pair of the bench pool at the
    BASELINE resolution 540x720 (config C3: resize (540, 720), 1024 keypoints)."""
    import cv2
    import torch
    from oracle import build_ref
    cases = []
    ims = []
    for n in ("scene0711_00_frame-001680.jpg", "scene0711_00_frame-001995.jpg"):
        im = cv2.resize(cv2.imread(os.path.join(build_ref.data_dir(), n), cv2.IMREAD_GRAYSCALE).astype("float32"), (640, 480))
        ims.append(torch.from_numpy(im / 255.0).float()[None, None])
    cases.append(("readme", ims[0], ims[1]))          # float resize: what the FMB matcher plugin feeds (matchers.py:100-103)
    ims = []
    for n in ("scene0711_00_frame-001680.jpg", "scene0711_00_frame-001995.jpg"):   # uint8 resize: match_pairs.py's default,
        im = cv2.resize(cv2.imread(os.path.join(build_ref.data_dir(), n), cv2.IMREAD_GRAYSCALE), (640, 480)).astype("float32")
        ims.append(torch.from_numpy(im / 255.0).float()[None, None])               # the README's 382 / 391 keypoints
    cases.append(("readme_u8", ims[0], ims[1]))
    p = synth.make_pair(1000)
    g0 = synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0
    g1 = synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0
    cases.append(("synth1000", torch.from_numpy(g0)[None, None], torch.from_numpy(g1)[None, None]))
    return cases
