#!/usr/bin/env python
"""Benchmark of the feature-matching + scale-from-depth hot path (BASELINE.json metric:
image-pairs/sec @ 540x720).

Headline workload (BASELINE.json configs[1], "C2"): LoFTR coarse-to-fine matching + 5-point essential matrix with the
scale recovered from depth (the reference's config/matching/mapfree/loftr_emat_dptkitti.yaml: EssentialMatrixMetric,
2 px / 0.1 / 0.9999), synthetic 540x720 gray + depth pairs. The reference does not ship the LoFTR checkpoints; the
weights are `loftr.functional_state_dict(noise=1e-3)`: full-shape layers that implement a working patch matcher, with
a dense Gaussian perturbation on every conv / linear weight so that no tensor-core operand is structurally zero (a
chip multiplying zeros draws less power and clocks higher than one running a trained checkpoint).

A "step" = `--micro` engine batches of `--batch` pairs (default 5 x 32 = 160 pairs) through matcher + solver on one
GPU, so that the driver's 20 steps time >= 5 s of steady state. With N GPUs every rank runs its own pairs (weak
scaling); one NCCL gather of the pose records at the end of the stream.

  python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU, torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   # reference arm: CPU path on the host cores
  python bench.py --steps K --warmup W --dump-outputs DIR  # also write the poses of the last timed step as DIR/*.npy

Prints ONE JSON line (rank 0). `value`: inputs resident in HBM. `e2e`: host (pinned) buffers in, pose records out,
copies inside the timed region, through the public Python API. `precisions`: the same workload in the TF32 and the
fp32-faithful (3xTF32) engine modes. `configs`: the other BASELINE.json configurations measured in the same run —
C1 (SIFT + exact NN + 5-pt, 16 pairs), C3 (SuperPoint + SuperGlue + PnP), C4 (10 k-pair stream sharded over the
ranks, strong scaling), C5 (RANSAC hypothesis sweep).
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H0, W0 = 720, 540            # dataset frame (config/mapfree.yaml HEIGHT/WIDTH)
PIX_THR, SCALE_THR = 2.0, 0.1
WEIGHT_NOISE = 1e-3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=int(os.environ.get("MFR_BENCH_BATCH", 32)), help="pairs per engine batch")
    ap.add_argument("--micro", type=int, default=int(os.environ.get("MFR_BENCH_MICRO", 5)), help="engine batches per step")
    ap.add_argument("--hyp", type=int, default=1024, help="5-point hypotheses per pair")
    ap.add_argument("--match-thr", type=float, default=0.2, help="LoFTR coarse confidence threshold (reference: 0.2)")
    ap.add_argument("--precision", default=os.environ.get("MFR_BENCH_PRECISION", "bf16"), choices=["tf32", "bf16", "fp32x3"],
                    help="engine mode of the headline run (include/mfr_b200.h: MFR_PRECISION_*)")
    ap.add_argument("--weights", default="functional_dense", choices=["functional_dense", "functional"],
                    help="functional_dense: working matcher + dense perturbation (default); functional: the 99.8 %% zero version")
    ap.add_argument("--pool", type=int, default=32, help="distinct synthetic pairs cycled through")
    ap.add_argument("--cpu-sample", type=int, default=4, help="pairs timed for the cpu_baseline leg")
    ap.add_argument("--configs", default=os.environ.get("MFR_BENCH_CONFIGS", "C1,C3,C4,C5"), help="extra BASELINE configs to measure ('' = none)")
    ap.add_argument("--stream-pairs", type=int, default=10000, help="length of the C4 pair stream")
    ap.add_argument("--no-siblings", action="store_true", help="skip the tf32 / fp32x3 runs of the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the poses of the last timed step of the headline run as DIR/<name>.npy")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------
# synthetic inputs
# ------------------------------------------------------------------------------------------------
def make_pool(n, seed0):
    from mfr_b200 import synth
    g0, g1, d0, d1, K, gt, rgb = [], [], [], [], [], [], []
    for i in range(n):
        p = synth.make_pair(seed0 + i)
        g0.append(synth.rgb_to_gray_u8(p["image0"]).astype(np.float32) / 255.0)
        g1.append(synth.rgb_to_gray_u8(p["image1"]).astype(np.float32) / 255.0)
        d0.append(p["depth0"]); d1.append(p["depth1"]); K.append(p["K_color0"])
        gt.append((p["R_gt"], p["t_gt"]))
    return (np.stack(g0), np.stack(g1), np.stack(d0), np.stack(d1), np.stack(K).astype(np.float32), gt)


def loftr_weights(kind):
    from mfr_b200 import loftr
    return loftr.functional_state_dict(noise=WEIGHT_NOISE if kind == "functional_dense" else 0.0)


def rot_err(Ra, Rb):
    c = np.clip((np.trace(np.asarray(Ra, np.float64).T @ np.asarray(Rb, np.float64)) - 1.0) / 2.0, -1.0, 1.0)
    return float(np.arccos(c))


def pose_errors(R, t, gt):
    """Rotation error (deg) and translation error (m) of one estimate against ground truth; NaN -> inf."""
    Rg, tg = gt
    if not (np.all(np.isfinite(R)) and np.all(np.isfinite(t))):
        return float("inf"), float("inf")
    return float(np.degrees(rot_err(R, Rg))), float(np.linalg.norm(np.ravel(t).astype(np.float64) - np.ravel(tg)))


fin = lambda v: [x for x in v if np.isfinite(x)]
med = lambda v, nd=4: (round(float(np.median(v)), nd) if len(v) else None)


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self._stop, self._t = gpu_index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=6)

    def __enter__(self):
        self.start()
        return self

    def __exit__(self, *a):
        self.stop()

    def summary(self):
        sm, mx, pw, reasons, capped = [], [], [], set(), 0
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
                    capped += name == "sw_power_cap"
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_mhz_min": float(min(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_median": float(np.median(pw)), "power_w_max": float(max(pw)), "sw_power_cap_samples": capped}


WEIGHTS_NOTE = {
    "functional_dense": ("loftr.functional_state_dict(noise=1e-3): hand-constructed full-shape LoFTR weights that implement a patch descriptor + "
                         "normalised cross-correlation (a working matcher: ~1-3.6 k matches per pair), plus seeded Gaussian noise on every conv / "
                         "linear weight so that all tensor-core operands are dense; the reference does not ship its checkpoints"),
    "functional": "loftr.functional_state_dict(): the same without the perturbation (99.8 % of the weights are zero)"}
WORKLOAD = "LoFTR coarse-to-fine + 5-pt essential (EssentialMatrixMetric, scale from depth), 540x720 (720x544 padded), 1xB200 per rank"
DTYPE = {"bf16": ("bf16 (ResNet-FPN maps, token-GEMM / correlation / linear-attention operands: bf16 storage, kind::f16 MMA, fp32 accumulate; "
                  "token residual stream, LayerNorm, similarity matrix, dual softmax, fine matching fp32; pose solve fp64/fp32)"),
         "tf32": "tf32 (fp32 storage, kind::tf32 MMA inputs in every GEMM, fp32 accumulate; attention / LayerNorm / softmax fp32; pose solve fp64/fp32)",
         "fp32x3": "fp32 via 3xTF32 split GEMMs (fp32 storage, hi/lo operand split, fp32 accumulate; everything else fp32; pose solve fp64/fp32)"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured", d.get("bf16_tflops_sustained")
    return 6650.0, 1590.0, "fallback", 1400.0


def load_traffic(precision, batch):
    """DRAM bytes of the ResNet-FPN conv launches of one engine batch, from the committed ncu capture of this
    workload (profiles/README.md); None when no capture exists for the configuration."""
    for rnd in ("r02", "r01"):
        p = os.path.join(ROOT, "profiles", f"{rnd}_conv_gemm_metrics_{precision}_B{batch}.json")
        if os.path.exists(p):
            d = json.load(open(p))["backbone"]
            return int(d["dram_read"] + d["dram_write"]), os.path.relpath(p, ROOT)
    return None, None


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Harness:
    """Device context of one rank: pool of synthetic pairs (pinned host + device resident), timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.local_rank, self.world = dist_env()
        assert torch.cuda.is_available(), "bench.py needs CUDA devices (no CPU fallback in the product path)"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.B = args.batch
        self.HP, self.WP = H0 + H0 % 8, W0 + W0 % 8                       # matchers.py:41-46 -> 720 x 544
        self.L = (self.HP // 8) * (self.WP // 8)
        # every rank holds the same pool: pair i of the C4 stream is the same pair whatever the number of ranks
        self.g0, self.g1, self.d0, self.d1, self.Kc, self.gt = make_pool(args.pool, 1000)
        self.n_pool = args.pool
        self.h = {k: torch.from_numpy(v).pin_memory() for k, v in (("g0", self.g0), ("g1", self.g1), ("d0", self.d0), ("d1", self.d1), ("K", self.Kc))}
        self.dres = {k: v.to(self.dev) for k, v in self.h.items()}
        self.idx_cache = [torch.tensor(self.batch_idx(s), device=self.dev) for s in range(self.n_pool)]   # period divides n_pool

    def batch_idx(self, b):
        return [(b * self.B + j) % self.n_pool for j in range(self.B)]

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def engine(self, precision, weights, thr):
        from mfr_b200 import loftr
        return loftr.LoFTR(loftr_weights(weights), batch=self.B, height=self.HP, width=self.WP, cfg={"thr": thr},
                           device=self.local_rank, graph=True, precision=precision, pipelined=True)

    def pipeline(self, eng, be):
        from mfr_b200.pipeline import RelocPipeline
        return RelocPipeline([eng], be, PIX_THR, SCALE_THR, self.args.hyp, depth_hw=(H0, W0))

    def submit_resident(self, pipe, eng, b):
        """inputs already in HBM; returns the poses of the previous batch (one-deep pipeline)"""
        idx = self.idx_cache[b % self.n_pool]
        d = self.dres
        with self.torch.cuda.stream(eng.stream):
            a, b_, p0, p1, Kb = (d["g0"][idx], d["g1"][idx], d["d0"][idx], d["d1"][idx], d["K"][idx].contiguous())
        return pipe.submit_device(a, b_, p0, p1, Kb, Kb)

    def submit_host(self, pipe, b):
        """host (pinned) inputs -> device copies inside the step; the previous batch's poses are read back"""
        idx = self.batch_idx(b)
        h = self.h
        return pipe.submit_host(*[[h[k][i] for i in idx] for k in ("g0", "g1", "d0", "d1", "K", "K")])

    def timed(self, pipe, eng, submit, n_batches, warm_batches, gather_at_end=False, sampler=None, keep=1):
        """CUDA-event time (ms, max over ranks) of `n_batches` engine batches through `pipe`, after `warm_batches`, and
        the results of the last `keep` of them, oldest first. `sampler` (ClockSampler) runs during the timed region only
        (not during the warm-up)."""
        torch, dist = self.torch, self.dist
        for b in range(warm_batches):
            submit(b)
        pipe.drain()
        self.barrier()
        if sampler is not None:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(eng.stream):
            e0.record()
        tail = collections.deque(maxlen=keep)
        for b in range(n_batches):
            r = submit(warm_batches + b)             # the result of the batch submitted before this one
            if r is not None:
                tail.append(r)
        last = pipe.drain()                          # the timed region ends when the last batch's poses are on the host
        tail.append(last)
        if gather_at_end and self.world > 1:
            R, t, n = last
            with torch.cuda.stream(eng.stream):
                rec = torch.cat([R.reshape(self.B, 9), t.reshape(self.B, 3), n.reshape(self.B, 1).float()], 1).to(self.dev).contiguous()
                allr = [torch.empty_like(rec) for _ in range(self.world)]
                dist.all_gather(allr, rec)           # the path's only collective: 52-byte records per pair
        with torch.cuda.stream(eng.stream):
            eng.stream.wait_stream(pipe.s_solve)
            e1.record()
        self.barrier()
        if sampler is not None:
            sampler.stop()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), list(tail)


def matches_of(eng, i0, i1):
    """Per-pair match lists of one synchronous forward: [(i_ids, j_ids, mkpts0, mkpts1)] as numpy."""
    out = eng.forward(i0, i1)
    off = out["m_offsets"].tolist()
    res = []
    for b in range(eng.B):
        s, e = off[b], off[b + 1]
        res.append((out["i_ids"][s:e].cpu().numpy(), out["j_ids"][s:e].cpu().numpy(),
                    out["mkpts0_f"][s:e].cpu().numpy(), out["mkpts1_f"][s:e].cpu().numpy()))
    return res


def decomposition(hs, be, eng_matches, label):
    """Pose deltas vs the CPU port on the pairs it solved, decomposed (VERDICT r1 #1c):
       matcher  = GPU matches -> OpenCV solver   vs  CPU matches -> OpenCV solver
       solver   = CPU matches -> GPU solver      vs  CPU matches -> OpenCV solver
       total    = GPU matches -> GPU solver      vs  CPU matches -> OpenCV solver
    plus the full-resolution match-set IoU between the engine and the fp32 CPU port."""
    import torch
    from oracle import pose_solver_oracle as po
    n = min(len(CPU_MATCHES), hs.B)
    ious, rows = [], {"matcher": [], "solver": [], "total": []}
    for i in range(n):
        ci, cj, ck0, ck1 = CPU_MATCHES[i]
        gi, gj, gk0, gk1 = eng_matches[i]
        a, b = set(zip(ci.tolist(), cj.tolist())), set(zip(gi.tolist(), gj.tolist()))
        ious.append(len(a & b) / max(1, len(a | b)))
        Rc, tc = CPU_POSES[i]
        # GPU matches -> OpenCV solver
        Rm, tm = po.essential_matrix_metric_solver(gk0, gk1, hs.d0[i], hs.d1[i], hs.Kc[i], hs.Kc[i], PIX_THR, 0.9999, SCALE_THR)[:2]
        # CPU matches -> GPU solver, GPU matches -> GPU solver
        poses = []
        for k0, k1 in ((ck0, ck1), (gk0, gk1)):
            dev = be.device
            tk0 = torch.from_numpy(np.ascontiguousarray(k0, np.float32)).to(dev); tk1 = torch.from_numpy(np.ascontiguousarray(k1, np.float32)).to(dev)
            off = torch.tensor([0, len(k0)], dtype=torch.int32, device=dev)
            Kd = torch.from_numpy(hs.Kc[i:i + 1]).to(dev).contiguous()
            R, t, nn = be.emat_metric(tk0, tk1, off, Kd, Kd, torch.from_numpy(hs.d0[i:i + 1]).to(dev), torch.from_numpy(hs.d1[i:i + 1]).to(dev),
                                      PIX_THR, SCALE_THR, hs.args.hyp)
            poses.append((R[0].cpu().numpy(), t[0].cpu().numpy()))
        for key, (R, t) in (("matcher", (Rm, np.ravel(tm))), ("solver", poses[0]), ("total", poses[1])):
            ok = np.all(np.isfinite(R)) and np.all(np.isfinite(Rc))
            rows[key].append((rot_err(R, Rc), float(np.linalg.norm(np.ravel(t) - np.ravel(tc)))) if ok else (float("inf"), float("inf")))
    out = {"precision": label, "pairs": n, "match_set_iou_vs_cpu_port_median": med(ious), "match_set_iou_vs_cpu_port_min": round(min(ious), 4) if ious else None}
    for key, v in rows.items():
        out[key + "_delta_rot_rad_median"] = med(fin([x[0] for x in v]), 5)
        out[key + "_delta_t_m_median"] = med(fin([x[1] for x in v]), 5)
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    import mfr_b200  # noqa: F401
    from mfr_b200 import pose_solver

    hs = Harness(args)
    rank, world, dev, B, K = hs.rank, hs.world, hs.dev, hs.B, args.steps
    Wm, micro = max(args.warmup, 3), max(1, args.micro)
    be = pose_solver.PoseBackend(max_pairs=B, max_pts=hs.L, max_hyp=max(args.hyp, 128), device=hs.local_rank)

    # ---------------------------------------------------------------- headline run (C2)
    eng = hs.engine(args.precision, args.weights, args.match_thr)
    pipe = hs.pipeline(eng, be)
    outs = eng.device_outputs()
    in_bytes = sum(int(np.prod(hs.h[k].shape[1:])) * hs.h[k].element_size() * B for k in ("g0", "g1", "d0", "d1", "K", "K")) * micro
    out_bytes = int(pipe.slots[0]["rec_host"].numel() * 4) * micro
    clk, clk2 = ClockSampler(hs.local_rank), ClockSampler(hs.local_rank)
    ms_res, last_step = hs.timed(pipe, eng, lambda b: hs.submit_resident(pipe, eng, b), K * micro, Wm * micro, gather_at_end=True,
                                 sampler=clk, keep=micro)
    clocks = clk.summary()
    ms_e2e, _ = hs.timed(pipe, eng, lambda b: hs.submit_host(pipe, b), K * micro, Wm * micro, sampler=clk2)
    clocks_e2e = clk2.summary()
    pairs = K * micro * B * world
    value, e2e_value = pairs / (ms_res / 1e3), pairs / (ms_e2e / 1e3)
    with torch.cuda.stream(eng.stream):
        m_last = int(outs["m_total"][0].item())

    # ---- accuracy pass (untimed): every pair of the pool once through the host-buffer path
    acc_rows = {}
    n_acc = (hs.n_pool + B - 1) // B
    res_list = [hs.submit_host(pipe, s_) for s_ in range(n_acc)][1:] + [pipe.drain()]     # results arrive one call late
    for s_, (Rb, tb, nb) in enumerate(res_list):
        for j, i in enumerate(hs.batch_idx(s_)):
            if i not in acc_rows:
                acc_rows[i] = (Rb[j].numpy(), tb[j].numpy(), int(nb[j]))
    gpu_errs = [pose_errors(acc_rows[i][0], acc_rows[i][1], hs.gt[i]) for i in sorted(acc_rows)]

    result = None
    if rank == 0:
        hbm, bf16, how, bf16_sus = load_peaks()
        # ---- roofline of the dominant kernel (tcgen05 conv/GEMM), per-launch device times by CUDA events
        prof = eng.profile(hs.dres["g0"][hs.idx_cache[0]], hs.dres["g1"][hs.idx_cache[0]])
        tot_ms = sum(p[2] for p in prof)
        traffic, traffic_src = load_traffic(args.precision, B)
        is_bb = lambda p: p[1] == 1 and p[0].startswith("layer")          # ResNet-FPN implicit-GEMM convs
        bb = [p for p in prof if is_bb(p)]
        og = [p for p in prof if p[1] == 1 and not is_bb(p)]             # transformer / correlation / fine-level GEMMs
        bb_ms, bb_fl = sum(p[2] for p in bb), sum(p[3] for p in bb)
        og_ms, og_fl = sum(p[2] for p in og), sum(p[3] for p in og)
        kind = {"bf16": "f16/bf16", "tf32": "tf32", "fp32x3": "tf32 (3 MMAs per product)"}[args.precision]
        peak = bf16 if args.precision == "bf16" else bf16 / 2.0
        peak_sus = (bf16_sus if args.precision == "bf16" else bf16_sus / 2.0) if bf16_sus else None
        achieved = bb_fl / (bb_ms * 1e-3) / 1e12
        roofline = {"kernel": f"conv_gemm_tf32_kernel, ResNet-FPN convs (tcgen05 kind::{kind}, {len(bb)} launches per engine batch)",
                    "bound": "tensor", "achieved": round(achieved, 1), "peak": round(peak, 1), "unit": "TFLOP/s",
                    "frac": round(achieved / peak, 4),
                    "peak_note": f"{how} cuBLAS bf16 burst {bf16} TFLOP/s" + ("" if args.precision == "bf16" else " / 2 (kind::tf32 issues at half the bf16 rate)") +
                                 "; the per-launch times behind `achieved` come from an eager pass with an event pair per launch (a kernel timed alone: burst peak)",
                    "frac_of_sustained_peak": round(achieved / peak_sus, 4) if peak_sus else None,
                    "sustained_peak_note": f"cuBLAS bf16 sustained {bf16_sus} TFLOP/s (back to back for 4 s, power-capped clocks): the denominator that matches the multi-second timed region",
                    "algorithmic_flops_per_launch_avg": bb_fl / max(1, len(bb)), "avg_launch_ms": round(bb_ms / max(1, len(bb)), 4),
                    "share_of_step": round(bb_ms / tot_ms, 3), "flops_per_engine_batch": bb_fl, "traffic": traffic,
                    "traffic_note": (f"dram__bytes_read.sum + dram__bytes_write.sum summed over the {len(bb)} launches of one engine batch, {traffic_src}"
                                     if traffic else "no ncu capture committed for this precision / batch"),
                    "other_gemms": {"what": "token (q|k|v, merge, MLP), correlation and fine-level GEMMs of the same kernel", "launches": len(og),
                                    "achieved": round(og_fl / (og_ms * 1e-3) / 1e12, 1), "peak": round(peak, 1),
                                    "frac": round(og_fl / (og_ms * 1e-3) / 1e12 / peak, 4), "share_of_step": round(og_ms / tot_ms, 3)},
                    "whole_step_tflops": round((bb_fl + og_fl) * K * micro / (ms_res * 1e-3) / 1e12, 1)}
        cpu = cpu_baseline(args, hs, sample=args.cpu_sample)
        decomp = [decomposition(hs, be, matches_of(eng, hs.dres["g0"][hs.idx_cache[0]], hs.dres["g1"][hs.idx_cache[0]]), args.precision)]
        accuracy = {"against": "synthetic ground-truth poses of the pool pairs (EssentialMatrixMetric: R, metric t)",
                    "pairs": len(gpu_errs), "solved": len(fin([e[0] for e in gpu_errs])),
                    "median_rot_err_deg": med(fin([e[0] for e in gpu_errs])),
                    "median_trans_err_m": med(fin([e[1] for e in gpu_errs])),
                    "median_inliers": med([acc_rows[i][2] for i in sorted(acc_rows)]),
                    "reference_cpu_port": {"pairs": len(CPU_ERRS), "median_rot_err_deg": med(fin([e[0] for e in CPU_ERRS])),
                                           "median_trans_err_m": med(fin([e[1] for e in CPU_ERRS])),
                                           "median_matches": med([e[2] for e in CPU_ERRS]),
                                           "note": "same first pairs of the pool, oracle LoFTR fp32 + OpenCV USAC_MAGSAC"},
                    "vs_reference_cpu_port": decomp,
                    "vs_reference_note": ("angle(R_a R_b^T) [rad] and |t_a - t_b| [m] against the CPU port's pose on the same pairs. `matcher`: only the matcher differs "
                                          "(engine matches fed to OpenCV); `solver`: only the solver differs (CPU matches fed to the GPU RANSAC); `total`: both. OpenCV's "
                                          "USAC_MAGSAC output is itself 5e-3..2e-2 rad from the least-squares optimum of its own inlier set (scripts/emat_protocol.py), "
                                          "which is what the solver column measures; tests/test_geometry_gpu.py holds the E-mat protocol of SURVEY §7")}
    eng_main_launches = eng.num_launches()

    # ---------------------------------------------------------------- the same workload in the other engine modes
    precisions = {}
    if not args.no_siblings:
        for prec, nb in (("tf32", 24), ("fp32x3", 8)):
            if prec == args.precision:
                continue
            eng.close(); del pipe, eng
            torch.cuda.empty_cache()
            eng = hs.engine(prec, args.weights, args.match_thr)
            pipe = hs.pipeline(eng, be)
            ms_p, _ = hs.timed(pipe, eng, lambda b: hs.submit_resident(pipe, eng, b), nb, 3)
            precisions[prec] = {"value": round(nb * B * world / (ms_p / 1e3), 2), "unit": "pairs/s", "ms_per_engine_batch": round(ms_p / nb, 3),
                                "engine_batches_timed": nb, "dtype": DTYPE[prec]}
            if rank == 0:
                accuracy["vs_reference_cpu_port"].append(
                    decomposition(hs, be, matches_of(eng, hs.dres["g0"][hs.idx_cache[0]], hs.dres["g1"][hs.idx_cache[0]]), prec))
    eng.close(); del pipe, eng
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- other BASELINE configs
    configs = {}
    want = [c for c in args.configs.split(",") if c]
    if "C4" in want:
        configs["C4"] = config_c4(hs, be, args)
    be.close()
    if rank == 0 and world == 1:
        for name, fn in (("C3", config_c3), ("C5", config_c5), ("C1", config_c1)):
            if name in want:
                try:
                    configs[name] = fn(hs, args)
                except Exception as e:  # a broken side config must not take the headline line with it
                    configs[name] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        precisions[args.precision] = {"value": round(value, 2), "unit": "pairs/s", "ms_per_engine_batch": round(ms_res / (K * micro), 3),
                                      "engine_batches_timed": K * micro, "dtype": DTYPE[args.precision]}
        result = {
            "metric": "image-pairs/sec @ 540x720", "value": round(value, 2), "unit": "pairs/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": round(ms_res / K, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_step_per_gpu": B * micro, "engine_batch": B, "engine_batches_per_step": micro,
                       "precision": args.precision, "hypotheses_per_pair": args.hyp, "match_thr": args.match_thr,
                       "matches_last_batch": m_last, "weights": WEIGHTS_NOTE[args.weights], "timed_region_s": round(ms_res / 1e3, 2),
                       "l2": "per-batch working set (activations + 150 MB similarity matrix per pair) far exceeds the 126 MB L2; inputs rotate over %d distinct pairs" % hs.n_pool},
            "e2e": {"value": round(e2e_value, 2), "unit": "pairs/s", "h2d_bytes_per_step": in_bytes,
                    "d2h_bytes_per_step": out_bytes, "ms_per_step": round(ms_e2e / K, 3), "clocks": clocks_e2e,
                    "api": "mfr_b200.pipeline.RelocPipeline.submit_host (copy / matcher / RANSAC stages of consecutive batches overlap)"},
            "gpu_launches": int((eng_main_launches + 5) * K * micro),   # + emat_normalise, emat_hyp, emat_lo, emat_final, scale_consensus
            "kernels_per_engine_batch": eng_main_launches + 5,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "precisions": precisions, "accuracy": accuracy, "configs": configs,
        }
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
        print(json.dumps(result))


def dump_outputs(out_dir, results):
    """Writes the poses the pipeline handed out for the engine batches of one step, one row per pair in submission
    order (row j of the b-th batch since the first warm-up batch is pool pair (b * batch + j) mod pool): R.npy [P,3,3],
    t.npy [P,3] float32 and inliers.npy [P] (counts, as float32)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    R, t, n = (torch.cat([r[k] for r in results]) for k in range(3))
    for name, a in (("R", R), ("t", t), ("inliers", n)):
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------
# C4: a fixed pair stream sharded over the ranks in contiguous blocks (strong scaling), SURVEY §8(d)/(e)
# ------------------------------------------------------------------------------------------------
def config_c4(hs, be, args):
    import torch
    from mfr_b200 import parallel
    B, n_pairs = hs.B, args.stream_pairs
    eng = hs.engine(args.precision, args.weights, args.match_thr)
    pipe = hs.pipeline(eng, be)

    def submit(ids):            # pair i of the stream = pool pair i mod n_pool; host (pinned) buffers in
        idx = [i % hs.n_pool for i in ids]
        return pipe.submit_host(*[[hs.h[k][i] for i in idx] for k in ("g0", "g1", "d0", "d1", "K", "K")])

    for _ in range(3):
        submit(list(range(B)))
    pipe.reset()                # the stream starts with an empty pipeline: its first submit returns None
    hs.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(eng.stream):
        e0.record()
    table = parallel.run_stream(n_pairs, B, submit, pipe.drain, hs.rank, hs.world, hs.dev)   # ends with the NCCL gather of the records
    e1.record()
    hs.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=hs.dev)
    if hs.world > 1:
        hs.dist.all_reduce(ms, op=hs.dist.ReduceOp.MAX)
    eng.close()
    if hs.rank != 0:
        return None
    ms = float(ms.item())
    R_ref = np.stack([hs.gt[i % hs.n_pool][0] for i in range(n_pairs)]); t_ref = np.stack([hs.gt[i % hs.n_pool][1] for i in range(n_pairs)])
    ang, dt, solved = parallel.median_pose_errors(table.cpu(), R_ref, t_ref)
    a, b = parallel.shard_range(n_pairs, 0, hs.world)
    r = {"value": round(n_pairs / (ms * 1e-3), 2), "unit": "pairs/s", "pairs": n_pairs, "seconds": round(ms * 1e-3, 3), "n_gpus": hs.world,
         "pairs_of_rank0": b - a, "records_gathered": int(table.shape[0]), "ordered": bool(torch.equal(table[:, 0].cpu(), torch.arange(n_pairs, dtype=torch.float64))),
         "solved": solved, "median_rot_err_rad_vs_gt": round(ang, 5), "median_trans_err_m_vs_gt": round(dt, 5),
         "e2e": "host (pinned) inputs per batch, records back to the host per batch: this IS the end-to-end path (RelocPipeline.submit_host)"}
    r.update({"workload": f"LoFTR + batched 5-pt RANSAC + scale from depth, a stream of {args.stream_pairs} pairs (pair i = pool pair i mod {hs.n_pool} of its rank's "
                          f"pool; ground truth known per pair), contiguous blocks per rank, one gather of the 112-byte records at the end",
              "scaling": "strong", "precision": args.precision})
    return r


# ------------------------------------------------------------------------------------------------
# C3: SuperPoint + SuperGlue + PnP from depth (sg_pnp_dptkitti.yaml), 540x720, 1024 keypoints
# ------------------------------------------------------------------------------------------------
def spsg_weights():
    """The reference's in-tree weights when they were staged next to the repo (data files, oracle/_ref/weights or
    $MFR_SPSG_WEIGHTS), else seeded synthetic ones."""
    import torch
    from mfr_b200 import spsg
    wd = os.environ.get("MFR_SPSG_WEIGHTS", os.path.join(ROOT, "oracle", "_ref", "weights"))
    sp, sg = os.path.join(wd, "superpoint_v1.pth"), os.path.join(wd, "superglue_indoor.pth")
    if os.path.exists(sp) and os.path.exists(sg):
        return torch.load(sp, map_location="cpu"), torch.load(sg, map_location="cpu"), "reference in-tree superpoint_v1 + superglue_indoor"
    a, b = spsg.synthetic_state_dicts(0)
    return a, b, "seeded synthetic (mfr_b200.spsg.synthetic_state_dicts)"


def config_c3(hs, args):
    import torch
    from mfr_b200 import pose_solver, spsg
    B = 8
    sp, sg, wnote = spsg_weights()
    eng = spsg.SuperPointSuperGlue(sp, sg, batch=B, height=H0, width=W0, graph=True, device=hs.local_rank)
    be = pose_solver.PoseBackend(max_pairs=B, max_pts=1024, max_hyp=1024, device=hs.local_rank)
    outs = eng.device_outputs()
    stage = {k: torch.empty(B, *hs.h[k].shape[1:], device=hs.dev) for k in ("g0", "g1", "d0", "K")}
    rec_host = torch.zeros(B, 13).pin_memory()
    idx = lambda b: [(b * B + j) % hs.n_pool for j in range(B)]

    def solve(d0, K):
        with torch.cuda.stream(eng.stream):
            R, t, n, _ = be.pnp(outs["mkpts0"], outs["mkpts1"], outs["m_offsets"], K, K, d0, 3.0, 1024)
        return R, t, n

    def step_res(b):
        ix = torch.tensor(idx(b), device=hs.dev)
        eng.forward_async(hs.dres["g0"][ix], hs.dres["g1"][ix])
        return solve(hs.dres["d0"][ix], hs.dres["K"][ix].contiguous())

    def step_e2e(b):
        with torch.cuda.stream(eng.stream):
            for k in stage:
                for j, i in enumerate(idx(b)):
                    stage[k][j].copy_(hs.h[k][i], non_blocking=True)
        eng.forward_async(stage["g0"], stage["g1"])
        R, t, n = solve(stage["d0"], stage["K"])
        with torch.cuda.stream(eng.stream):
            rec = torch.cat([R.reshape(B, 9), t.reshape(B, 3), n.reshape(B, 1).float()], 1)
            rec_host.copy_(rec, non_blocking=True)
        eng.stream.synchronize()
        return R, t, n

    def timed(fn, n):
        for b in range(3):
            fn(b)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(eng.stream):
            e0.record()
        for b in range(n):
            r = fn(3 + b)
        with torch.cuda.stream(eng.stream):
            e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    nb = 40
    ms_res, _ = timed(step_res, nb)
    ms_e2e, _ = timed(step_e2e, nb)
    # accuracy over the pool + keypoint / match statistics
    errs, kp, mt = [], [], []
    for b in range((hs.n_pool + B - 1) // B):
        R, t, n = step_res(b)
        torch.cuda.synchronize()
        kp.append(outs["counts"].float().mean().item())
        mt.append((outs["m_offsets"][1:] - outs["m_offsets"][:-1]).float().mean().item())
        for j, i in enumerate(idx(b)):
            errs.append(pose_errors(R[j].cpu().numpy(), t[j].cpu().numpy(), hs.gt[i]))
    flops_pair = 219.9e9                       # SURVEY §8(d): 131.7 (SuperPoint x2) + 88.2 (SuperGlue at n = m = 1024) GFLOP
    hbm, bf16, how, bf16_sus = load_peaks()
    achieved = flops_pair * B * nb / (ms_res * 1e-3) / 1e12
    # CPU baseline: oracle SuperPoint + SuperGlue (torch CPU fp32) + OpenCV solvePnPRansac, bounded sample
    from oracle import pose_solver_oracle as po, spsg_oracle as so
    cores = use_all_host_threads()
    t_net = t_solve = 0.0
    n_cpu = 2
    for i in range(n_cpu):
        i0 = torch.from_numpy(hs.g0[i])[None, None]; i1 = torch.from_numpy(hs.g1[i])[None, None]
        t0 = time.perf_counter()
        with torch.no_grad():
            k0, s0, d0 = so.superpoint(i0, sp); k1, s1, d1 = so.superpoint(i1, sp)
            m0, _ = so.superglue(k0, s0, d0, k1, s1, d1, H0, W0, sg)
        t1 = time.perf_counter()
        v = m0 > -1
        po.pnp_solver(k0[v].numpy(), k1[m0[v]].numpy(), hs.d0[i], hs.Kc[i], hs.Kc[i], 1000, 3, 0.9999)
        t_net += t1 - t0; t_solve += time.perf_counter() - t1
    n_launch = eng.num_launches() + 5
    eng.close(); be.close()
    return {"workload": "SuperPoint + SuperGlue (1024 keypoints, matchers.py:65-71) + PnPSolver (P3P RANSAC 3 px + LM refine), 540x720",
            "weights": wnote, "value": round(B * nb / (ms_res * 1e-3), 2), "unit": "pairs/s", "pairs_per_batch": B, "ms_per_batch": round(ms_res / nb, 3),
            "dtype": "tf32 (fp32 storage, kind::tf32 MMA inputs; softmax / Sinkhorn / NMS fp32; pose solve fp64/fp32)",
            "e2e": {"value": round(B * nb / (ms_e2e * 1e-3), 2), "unit": "pairs/s",
                    "h2d_bytes_per_batch": int(sum(np.prod(hs.h[k].shape[1:]) * 4 for k in stage) * B), "d2h_bytes_per_batch": B * 13 * 4},
            "keypoints_per_image": round(float(np.mean(kp)), 1), "matches_per_pair": round(float(np.mean(mt)), 1),
            "gpu_launches_per_batch": n_launch,
            "roofline": {"kernel": "conv_gemm_tf32_kernel (SuperPoint convs, SuperGlue linears + attention GEMMs); whole-step figure", "bound": "tensor",
                         "achieved": round(achieved, 1), "peak": round(bf16 / 2, 1), "unit": "TFLOP/s", "frac": round(achieved / (bf16 / 2), 4),
                         "algorithmic_flops_per_pair": flops_pair, "traffic": None},
            "accuracy": {"pairs": len(errs), "solved": len(fin([e[0] for e in errs])), "median_rot_err_deg": med(fin([e[0] for e in errs])),
                         "median_trans_err_m": med(fin([e[1] for e in errs]))},
            "cpu_baseline": {"value": round(n_cpu / (t_net + t_solve), 4), "unit": "pairs/s", "cores": cores, "kind": "port",
                             "stage_b_only_pairs_per_s": round(n_cpu / t_solve, 2),
                             "sample": f"{n_cpu} pairs: oracle SuperPoint+SuperGlue (torch CPU fp32) {t_net / n_cpu:.2f} s/pair + OpenCV solvePnPRansac(P3P) + LM {t_solve / n_cpu * 1e3:.1f} ms/pair"}}


# ------------------------------------------------------------------------------------------------
# C5: RANSAC hypothesis sweep (warp-per-hypothesis E-matrix kernel + LO), SURVEY §8(d)
# ------------------------------------------------------------------------------------------------
def config_c5(hs, args):
    import torch
    from mfr_b200 import pose_solver, synth
    P, N, cells_pairs = 64, 2000, 256
    be = pose_solver.PoseBackend(max_pairs=P, max_pts=N, max_hyp=65536, device=hs.local_rank)
    cells = []
    best_rate = 0.0
    for ratio in (0.05, 0.1, 0.2, 0.3, 0.5):
        cs = [synth.make_correspondence_points(5000 + i, n=N, inlier_ratio=ratio, noise_px=0.5) for i in range(cells_pairs)]
        chunks = []
        for c0 in range(0, cells_pairs, P):
            cc = cs[c0:c0 + P]
            chunks.append((torch.from_numpy(np.concatenate([c["kpts0"] for c in cc])).to(hs.dev), torch.from_numpy(np.concatenate([c["kpts1"] for c in cc])).to(hs.dev),
                           torch.from_numpy(np.stack([c["K_color0"] for c in cc])).to(hs.dev).contiguous()))
        off = torch.arange(P + 1, dtype=torch.int32, device=hs.dev) * N
        for hyp in (256, 1024, 4096, 16384, 65536):
            for k0, k1, Kd in chunks[:1]:
                be.emat(k0, k1, off, Kd, Kd, PIX_THR, hyp)          # warm
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            outs = []
            e0.record()
            for k0, k1, Kd in chunks:
                outs.append(be.emat(k0, k1, off, Kd, Kd, PIX_THR, hyp)[:2])
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            Rn = torch.cat([o[0] for o in outs]).cpu().numpy().astype(np.float64); tn = torch.cat([o[1] for o in outs]).cpu().numpy().astype(np.float64)
            ok = 0
            for i, c in enumerate(cs):
                if np.all(np.isfinite(Rn[i])):
                    ta = np.arccos(np.clip(tn[i] @ c["t_gt"] / np.linalg.norm(c["t_gt"]), -1, 1))
                    ok += (np.degrees(rot_err(Rn[i], c["R_gt"])) < 1.0) and (np.degrees(ta) < 5.0)
            rate = cells_pairs * hyp / (ms * 1e-3)
            best_rate = max(best_rate, rate)
            cells.append({"inlier_ratio": ratio, "hypotheses": hyp, "ms_per_pair": round(ms / cells_pairs, 4), "hyp_per_s": round(rate),
                          "solved_fraction": round(ok / cells_pairs, 3)})
    # OpenCV reference point on one cell (bounded sample)
    from oracle import pose_solver_oracle as po
    cores = use_all_host_threads()
    cs = [synth.make_correspondence_points(5000 + i, n=N, inlier_ratio=0.3, noise_px=0.5) for i in range(8)]
    t0 = time.perf_counter()
    okc = 0
    for c in cs:
        R, t = po.essential_matrix_solver(c["kpts0"], c["kpts1"], c["K_color0"], c["K_color1"], PIX_THR, 0.9999)[:2]
        if np.all(np.isfinite(R)):
            ta = np.arccos(np.clip(np.ravel(t) @ c["t_gt"] / np.linalg.norm(c["t_gt"]), -1, 1))
            okc += (np.degrees(rot_err(R, c["R_gt"])) < 1.0) and (np.degrees(ta) < 5.0)
    dt = time.perf_counter() - t0
    be.close()
    # algorithmic work of a hypothesis: ~1e4 flop solve + ~4 real models x N x 35 flop of Sampson scoring (SURVEY §8(d))
    flop_h = 1e4 + 4 * N * 35
    return {"workload": f"5-pt essential RANSAC + LO, {N} correspondences per pair (0.5 px inlier noise, uniform outliers), {cells_pairs} pairs per cell in calls of {P}",
            "value": round(best_rate), "unit": "hypotheses/s (best cell)", "cells": cells,
            "solved_definition": "rotation error < 1 deg and translation-direction error < 5 deg vs ground truth",
            "roofline": {"kernel": "emat_hyp_kernel", "bound": "fp32/fp64 ALU + latency (not HBM: the working set is 32 KB per pair)",
                         "achieved": round(best_rate * flop_h / 1e12, 2), "peak": 80.0, "unit": "TFLOP/s (fp32 SIMT nominal)",
                         "frac": round(best_rate * flop_h / 1e12 / 80.0, 4), "traffic": None,
                         "note": "algorithmic flop per hypothesis = 1e4 (solve) + 4 x N x 35 (scoring); early exit makes the executed work smaller"},
            "cpu_baseline": {"value": round(len(cs) / dt, 2), "unit": "pairs/s", "cores": cores, "kind": "port",
                             "sample": f"OpenCV findEssentialMat(USAC_MAGSAC) + recoverPose on 8 sets of the 30 % cell: {dt / len(cs) * 1e3:.1f} ms/pair, solved {okc}/8 "
                                       f"(OpenCV caps RANSAC at 1000 iterations)"}}


# ------------------------------------------------------------------------------------------------
# C1: 16 pairs, SIFT(2048) + RootSIFT + exact NN + 5-pt essential + scale (sift_emat_dptkitti.yaml) — the plumbing line
# ------------------------------------------------------------------------------------------------
def config_c1(hs, args):
    import cv2
    import torch
    from mfr_b200 import model as mmodel, pose_solver
    n = 16
    sift = cv2.SIFT_create(2048)
    be = pose_solver.PoseBackend(max_pairs=1, max_pts=4096, max_hyp=2048, device=hs.local_rank)
    u8 = lambda g: np.clip(np.round(g * 255.0), 0, 255).astype(np.uint8)

    def ours(i):
        t0 = time.perf_counter()
        kp0, de0 = sift.detectAndCompute(u8(hs.g0[i]), None); kp1, de1 = sift.detectAndCompute(u8(hs.g1[i]), None)
        t1 = time.perf_counter()
        i1, d1, _, d2 = mmodel.knn2_gpu(mmodel.root_sift(de0), mmodel.root_sift(de1))
        good = d1 < 0.8 * d2
        p0 = np.float32([kp0[a].pt for a in np.where(good)[0]]).reshape(-1, 2); p1 = np.float32([kp1[b].pt for b in i1[good]]).reshape(-1, 2)
        dev = hs.dev
        off = torch.tensor([0, len(p0)], dtype=torch.int32, device=dev)
        Kd = torch.from_numpy(hs.Kc[i:i + 1]).to(dev).contiguous()
        R, t, nn = be.emat_metric(torch.from_numpy(p0).to(dev), torch.from_numpy(p1).to(dev), off, Kd, Kd, torch.from_numpy(hs.d0[i:i + 1]).to(dev),
                                  torch.from_numpy(hs.d1[i:i + 1]).to(dev), 3.0, SCALE_THR, 2048)
        R, t = R[0].cpu().numpy(), t[0].cpu().numpy()
        return (t1 - t0, time.perf_counter() - t1, R, t, len(p0), (kp0, de0, kp1, de1))

    ours(0)
    rows = [ours(i) for i in range(n)]
    t_sift, t_gpu = sum(r[0] for r in rows), sum(r[1] for r in rows)
    errs = [pose_errors(r[2], r[3], hs.gt[i]) for i, r in enumerate(rows)]
    # CPU reference: same SIFT features, exact mutual... the reference's ratio test on an exact 2-NN (cv2.BFMatcher), OpenCV solver
    from oracle import pose_solver_oracle as po
    cores = use_all_host_threads()
    bf = cv2.BFMatcher(cv2.NORM_L2)
    t_cpu = 0.0
    cerrs = []
    for i, r in enumerate(rows):
        kp0, de0, kp1, de1 = r[5]
        t0 = time.perf_counter()
        mm = bf.knnMatch(mmodel.root_sift(de0), mmodel.root_sift(de1), k=2)
        good = [a for a, b in mm if a.distance < 0.8 * b.distance]
        p0 = np.float32([kp0[a.queryIdx].pt for a in good]).reshape(-1, 2); p1 = np.float32([kp1[a.trainIdx].pt for a in good]).reshape(-1, 2)
        R, t = po.essential_matrix_metric_solver(p0, p1, hs.d0[i], hs.d1[i], hs.Kc[i], hs.Kc[i], 3.0, 0.9999, SCALE_THR)[:2]
        t_cpu += time.perf_counter() - t0
        cerrs.append(pose_errors(R, t, hs.gt[i]))
    be.close()
    return {"workload": "16 synthetic 540x720 pairs: SIFT(2048) + RootSIFT (OpenCV, host) -> exact 2-NN + ratio 0.8 (GPU) -> 5-pt essential RANSAC + scale from depth (GPU), "
                        "EMAT_RANSAC 3 px / 0.1 / 0.9999 (sift_emat_dptkitti.yaml); one pair per call, host arrays in and out",
            "value": round(n / (t_sift + t_gpu), 3), "unit": "pairs/s", "pairs": n,
            "ms_per_pair": {"sift_detect_cpu": round(t_sift / n * 1e3, 1), "nn_plus_pose_gpu_incl_copies": round(t_gpu / n * 1e3, 2)},
            "value_after_detection": round(n / t_gpu, 2), "median_matches": med([r[4] for r in rows]),
            "accuracy": {"median_rot_err_deg": med(fin([e[0] for e in errs])), "median_trans_err_m": med(fin([e[1] for e in errs])), "solved": len(fin([e[0] for e in errs]))},
            "cpu_baseline": {"value": round(n / (t_sift + t_cpu), 3), "unit": "pairs/s", "cores": cores, "kind": "port",
                             "after_detection_pairs_per_s": round(n / t_cpu, 2),
                             "accuracy": {"median_rot_err_deg": med(fin([e[0] for e in cerrs])), "median_trans_err_m": med(fin([e[1] for e in cerrs]))},
                             "sample": f"the same {n} pairs and SIFT features: cv2.BFMatcher exact 2-NN + ratio test + OpenCV USAC_MAGSAC + scale consensus, {t_cpu / n * 1e3:.1f} ms/pair after detection"}}


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's algorithm restated in oracle/ (torch CPU LoFTR +
# OpenCV USAC_MAGSAC + scale consensus), all host threads
# ------------------------------------------------------------------------------------------------
CPU_ERRS = []     # (rot err deg, trans err m, matches) of every pair the CPU leg solved
CPU_POSES = []    # its (R, t) per pair, same order as the pool
CPU_MATCHES = []  # its (i_ids, j_ids, mkpts0, mkpts1) per pair


def cpu_pairs(n_pairs, match_thr, weights, seed0=1000, pool=None, device="cpu"):
    """Oracle LoFTR (torch fp32 on `device`) + OpenCV solver for the first n_pairs of the pool. Returns (net s, solver s)."""
    import torch
    from mfr_b200 import loftr
    from oracle import loftr_oracle as lo, pose_solver_oracle as po
    sd = loftr_weights(weights)
    if device != "cpu":
        sd = {k: v.to(device) for k, v in sd.items()}
    g0, g1, d0, d1, Kc, gt = pool if pool is not None else make_pool(n_pairs, seed0)
    t_net = t_solve = 0.0
    for i in range(n_pairs):
        i0 = loftr.pad_to_8(torch.from_numpy(g0[i])[None, None]); i1 = loftr.pad_to_8(torch.from_numpy(g1[i])[None, None])
        t0 = time.perf_counter()
        with torch.no_grad():
            o = lo.loftr_forward(i0.to(device), i1.to(device), sd, {"thr": match_thr})
            k0, k1 = o["mkpts0_f"].cpu().numpy(), o["mkpts1_f"].cpu().numpy()
        t1 = time.perf_counter()
        Rc, tc = po.essential_matrix_metric_solver(k0, k1, d0[i], d1[i], Kc[i], Kc[i], PIX_THR, 0.9999, SCALE_THR)[:2]
        t2 = time.perf_counter()
        t_net += t1 - t0; t_solve += t2 - t1
        if device == "cpu":
            CPU_ERRS.append(pose_errors(Rc, tc, gt[i]) + (len(k0),))
            CPU_POSES.append((np.asarray(Rc, np.float64), np.ravel(tc).astype(np.float64)))
            CPU_MATCHES.append((o["i_ids"].numpy(), o["j_ids"].numpy(), k0, k1))
    return t_net, t_solve


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs are meant to use every core the process may run on."""
    import torch
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:                                   # one thread per physical core (SMT siblings only slow the GEMMs down)
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = max(1, min(n, phys))
    except Exception:
        pass
    torch.set_num_threads(n)
    try:
        import cv2
        cv2.setNumThreads(n)
    except Exception:
        pass
    return torch.get_num_threads()


def cpu_baseline(args, hs, sample):
    cores = use_all_host_threads()
    pool = (hs.g0, hs.g1, hs.d0, hs.d1, hs.Kc, hs.gt)
    t_net, t_solve = cpu_pairs(sample, args.match_thr, args.weights, pool=pool)
    out = {"value": round(sample / (t_net + t_solve), 4), "unit": "pairs/s", "cores": cores, "kind": "port",
           "sample": f"{sample} pairs of the same workload: oracle LoFTR (torch CPU fp32, {cores} threads) {t_net / sample:.2f} s/pair + OpenCV USAC_MAGSAC 5-pt + scale consensus {t_solve / sample * 1e3:.1f} ms/pair",
           "stage_b_only_pairs_per_s": round(sample / t_solve, 2), "stage_b_ms_per_pair": round(t_solve / sample * 1e3, 1),
           "net_on_cpu_s_per_pair": round(t_net / sample, 2),
           "stage_b_note": "what the reference runs ONLINE on the CPU (submission.py: precomputed correspondences -> OpenCV solver); the matcher is an offline GPU job there"}
    try:     # the reference's real Stage A: the same torch-eager network on THIS GPU (cuDNN / cuBLAS, TF32 off like torch 2.0.1), OpenCV solver on the host
        import torch
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        cpu_pairs(1, args.match_thr, args.weights, pool=pool, device="cuda")          # warm-up (cuDNN autotune, allocator)
        torch.cuda.synchronize()
        tn, ts = cpu_pairs(sample, args.match_thr, args.weights, pool=pool, device="cuda")
        out["torch_eager_on_this_gpu"] = {"loftr_ms_per_pair": round(tn / sample * 1e3, 1), "opencv_solver_ms_per_pair": round(ts / sample * 1e3, 1),
                                          "pairs_per_s": round(sample / (tn + ts), 2),
                                          "note": "oracle LoFTR as torch eager fp32 on the B200 (one pair per forward, the reference's batch size) + OpenCV solver on the host: "
                                                  "the deployment the reference documents (offline GPU matcher + online CPU solver), serialised"}
    except Exception as e:
        out["torch_eager_on_this_gpu"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    K, Wm = args.steps, args.warmup
    cores = use_all_host_threads()
    if Wm > 0:
        cpu_pairs(1, args.match_thr, args.weights)             # warm-up (thread pools, allocator)
        CPU_ERRS.clear(); CPU_POSES.clear(); CPU_MATCHES.clear()
    t0 = time.perf_counter()
    t_net, t_solve = cpu_pairs(K, args.match_thr, args.weights)   # one pair per step (bounded sample of a step)
    wall = time.perf_counter() - t0
    v = K / wall
    print(json.dumps({
        "impl": "reference", "metric": "image-pairs/sec @ 540x720", "value": round(v, 4), "unit": "pairs/s",
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(wall / K * 1e3, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 (OpenCV solve f64)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "match_thr": args.match_thr, "weights": WEIGHTS_NOTE[args.weights],
                   "reference_sample": "reference CPU path (oracle port: torch CPU fp32 LoFTR + OpenCV USAC_MAGSAC + scale consensus), 1 pair per step on rank 0"},
        "cpu_baseline": {"value": round(v, 4), "unit": "pairs/s", "cores": cores, "kind": "port",
                         "sample": f"{K} pairs, LoFTR {t_net / K:.2f} s/pair + solver {t_solve / K * 1e3:.1f} ms/pair",
                         "stage_b_only_pairs_per_s": round(K / t_solve, 2), "net_on_cpu_s_per_pair": round(t_net / K, 2)},
        "e2e": {"value": round(v, 4), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "accuracy": {"against": "synthetic ground-truth poses", "pairs": len(CPU_ERRS),
                     "median_rot_err_deg": round(float(np.median([e[0] for e in CPU_ERRS])), 4),
                     "median_trans_err_m": round(float(np.median([e[1] for e in CPU_ERRS])), 4),
                     "median_matches": float(np.median([e[2] for e in CPU_ERRS]))}}))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
