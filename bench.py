#!/usr/bin/env python
"""bench.py - headline benchmark of the multi-view reconstruction hot path (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

One "step" = one pass of the fused triangulate+reproject kernel over one clip of synthetic
observations (BASELINE config 2: 2-view front/side rig, 1M frames x 17 COCO joints, K / distortion
from camera_calibration/calibration_parameters.npz).  With N>1 (torchrun, one rank per GPU) every
rank processes its own 1M-frame clip - frames shard with no data-path collective - so scaling is
"weak" and `value` is the whole-job joints/s = N*T*J / max-over-ranks time.

Prints ONE JSON line (see the task contract): value = kernel throughput with inputs resident in
HBM, e2e = the same metric through the host-buffer API (pinned H2D + kernel + D2H every step),
roofline = algorithmic bytes / CUDA-event time against the measured HBM peak, cpu_baseline = the
reference's per-frame CPU path (oracle port: cv2.triangulatePoints + cv2.projectPoints loop) timed
on this box's host cores on a bounded sample.  `--impl reference` times that CPU path alone with
all host cores.  `--dump-outputs DIR` writes the arrays the timed step computed (X, err; rank 0) as .npy files: the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "triangulated_joints_per_sec"
UNIT = "joints/s"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of the headline kernel loop (`value`, `ms_per_step`); the "
                    "host-buffer arms time min(steps, 10) but at least 3 (their `steps`), the extra objects their own fixed counts")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=1_000_000)
    ap.add_argument("--joints", type=int, default=17)
    ap.add_argument("--rig", default="2b")
    ap.add_argument("--conf", action="store_true", help="confidence-weighted DLT (default: unit weights, the reference's behaviour)")
    ap.add_argument("--pinhole", action="store_true", help="score without the distortion model")
    ap.add_argument("--solver", default="secular")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ba", action="store_true")
    ap.add_argument("--cpu-sample-frames", type=int, default=20000)
    ap.add_argument("--ba-iters", type=int, default=20)
    ap.add_argument("--no-ba-graph", action="store_true", help="enqueue the LM trials one by one instead of replaying a captured CUDA graph")
    ap.add_argument("--record-ba-parity", action="store_true", help="1 GPU: write the BA cost trajectories to gpurun_out/ba_parity_n1.json (commit as profiles/ba_parity_n1.json)")
    ap.add_argument("--no-extra", action="store_true", help="skip the 8-view north-star shape (extra object `tri_8view`)")
    ap.add_argument("--e2e-chunk", type=int, default=131072, help="frames per H2D -> kernel -> D2H chunk of the host pipeline")
    ap.add_argument("--e2e-streams", type=int, default=3)
    ap.add_argument("--e2e-graph", action="store_true", help="replay the host pipeline's copies and kernels as one CUDA graph instead of enqueueing them call by call (same speed: the copies bound it)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write X.npy (T,J,3) and err.npy (V,T,J) of the last step "
                    "(float32, rank 0) to DIR; above 32 MiB a fixed seeded sample of frames is written")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def workload_config(a, V):
    return {
        "workload": f"config2: {V}-view rig '{a.rig}' DLT triangulation + fused reprojection scoring, "
        f"T={a.frames} frames x J={a.joints} joints per GPU",
        "frames_per_gpu": a.frames,
        "joints": a.joints,
        "views": V,
        "confidence_weighted": bool(a.conf),
        "distortion_scoring": (not a.pinhole),
        "layout": "view-major (V,T,J,2)",
        "solver": a.solver,
        "parallelism": f"frame-sharded x{a.gpus}, no data-path collective",
        "l2_policy": "inputs+outputs per step exceed the 126 MB L2 (no flush needed)",
    }


# ------------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    kL, kR, K, R, t, dist = args
    from oracle import reference_path as RP

    n = len(kL)
    RP.clip_two_view(kL, kR, K, [R] * n, [t] * n, dist=dist)
    return n


def cpu_reference_rate(clip, dist, frames, procs):
    """joints/s of the reference's per-frame CPU path (oracle port) on `frames` frames with `procs`
    worker processes (1 = how the reference itself runs: a single Python loop)."""
    kL, kR = clip.x_vm[0][:frames], clip.x_vm[1][:frames]
    K, R, t = clip.K[0], clip.R[1], clip.t[1]
    J = kL.shape[1]
    if procs <= 1:
        t0 = time.perf_counter()
        _cpu_worker((kL, kR, K, R, t, dist))
        dt = time.perf_counter() - t0
    else:
        import multiprocessing as mp

        chunks = np.array_split(np.arange(frames), procs)
        jobs = [(kL[c], kR[c], K, R, t, dist) for c in chunks if len(c)]
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_cpu_worker, [(kL[:8], kR[:8], K, R, t, dist)] * procs)  # spin the workers up
            t0 = time.perf_counter()
            pool.map(_cpu_worker, jobs)
            dt = time.perf_counter() - t0
    return frames * J / dt, dt


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from skiing_analysis_pytorch_b200 import synth

    if a.rig not in ("2a", "2b", "2"):
        print(json.dumps({"impl": "reference", "unavailable": "the reference's CPU path is two-view only (triangulate.py:65-67)"}))
        return 0
    cores = os.cpu_count() or 1
    per_step = max(cores * 500, min(a.cpu_sample_frames, 4000 * cores))
    clip = synth.make_clip(a.rig, per_step, a.joints, seed=0)
    dist = None if a.pinhole else synth.DIST_CALIB
    for _ in range(a.warmup):
        cpu_reference_rate(clip, dist, min(per_step, cores * 64), cores)
    times = []
    for _ in range(a.steps):
        _, dt = cpu_reference_rate(clip, dist, per_step, cores)
        times.append(dt)
    total = float(np.sum(times))
    value = a.steps * per_step * a.joints / total
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": a.gpus,
        "steps": a.steps,
        "warmup": a.warmup,
        "ms_per_step": 1e3 * total / a.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": dict(workload_config(a, 2), reference_sample_frames_per_step=per_step,
                       note="the CPU arm times a bounded sample of the workload per step (a rate: joints/s does not depend on the clip length)"),
        "cpu_baseline": {
            "value": value,
            "unit": UNIT,
            "cores": cores,
            "kind": "port",
            "sample": f"{per_step} frames x {a.joints} joints per step, per-frame cv2.triangulatePoints + cv2.projectPoints "
            f"loop (oracle/reference_path.py) split over {cores} processes",
        },
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    REASONS = {
        0x8: "hw_slowdown",
        0x40: "hw_thermal_slowdown",
        0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap",
        0x80: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None

    def __enter__(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        except Exception:
            self._nvml = None
        return self

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                for b, name in self.REASONS.items():
                    if bits & b:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {
            "sm_mhz": float(np.median(self.samples)),
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(self.samples),
        }


# ------------------------------------------------------------------------------------------ GPU arm
def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def recorded_traffic(key: str):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    p = ROOT / "profiles" / "traffic.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get(key)
        except Exception:
            return None
    return None


BA_CONFIGS = {
    # name: (rig, total frames, joints) - BASELINE.json configs[2] and configs[4]
    "config3": ("2b", 100_000, 17),
    "config3_calib": ("2b", 100_000, 17),  # config 3 with every camera's intrinsics + distortion free (15 parameters per camera)
    "config5": ("8", 1_000_000, 70),
}


def ba_cpu_iteration_rate(frames=1500, joints=17, rig="2b", iters=3):
    """LM iterations/s of the fp64 numpy Schur-LM oracle (oracle/lm.py) on `frames` frames; the
    reference has no LM of its own (run_local_ba is undefined), so this port is the CPU arm."""
    from oracle import lm

    clip, R0, t0, X0 = lm.make_problem(rig, frames, joints)
    t0_ = time.perf_counter()
    lm.run_lm(X0, R0, t0, clip.K, clip.x_fm, clip.conf_fm, num_iters=iters)
    return iters / (time.perf_counter() - t0_)


def run_first_order(a, dev, rank, n_gpus, dist=None):
    """Row N1 (first-order form): Adam iterations/s on the reference's full configured objective (configs/vggt.yaml:43-52)
    with per-frame cameras at config-3 size, one iteration replayed from a CUDA graph; N GPUs: the clip's frames sharded by
    range (strong scaling; one-frame halos + all-reduced sums inside the graph).  Beside it, at N = 1, the same iteration
    (forward + backward of the five loss terms, all host threads) of the torch restatement on the CPU."""
    import torch

    from skiing_analysis_pytorch_b200 import api, ba, synth

    T_total, J = 100_000, 17
    T = T_total // n_gpus
    d = synth.make_clip_device("2b", T, J, dev, seed=100, shardable=True, frame_offset=rank * T)  # the same clip at every N
    R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
    R = torch.tensor(R0, device=dev, dtype=torch.float32)[None].expand(T, 2, 3, 3).contiguous()
    t = torch.tensor(t0, device=dev, dtype=torch.float32)[None].expand(T, 2, 3).contiguous()
    X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), d["K"], R0, t0, want=("X",)).X  # DLT under the perturbed rig
    args = (torch.tensor(d["K"], dtype=torch.float32), R, t, X0, d["x2d"], d["conf"])
    kw = dict(lr=1e-2, device=dev, mode="full", group=dist.group.WORLD if n_gpus > 1 else None)
    ba.run_local_ba_first_order(*args, num_iters=8, **kw)  # warm-up
    torch.cuda.synchronize()

    def wall(n):
        torch.cuda.synchronize()
        if n_gpus > 1:
            dist.barrier()
        t0_ = time.perf_counter()
        out_ = ba.run_local_ba_first_order(*args, num_iters=n, **kw)
        torch.cuda.synchronize()
        return time.perf_counter() - t0_, out_[3]

    (t_short, _), (t_long, h) = wall(100), wall(500)   # set-up + graph capture cancel in the difference
    ms = 1e3 * (t_long - t_short) / 400
    if n_gpus > 1:
        m = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(m, op=dist.ReduceOp.MAX)
        ms = float(m.item())
    losses_rec = [h[k]["loss"] for k in (0, 99, 499)]
    parity = {"reference": "unrecorded", "ok": None}
    try:
        ref = json.loads((ROOT / "profiles" / "ba_parity_n1.json").read_text()).get("first_order")
    except Exception:
        ref = None
    if ref is not None:
        rel = max(abs(x - y) / abs(y) for x, y in zip(losses_rec, ref["losses"]))
        parity = {"reference": f"profiles/ba_parity_n1.json ({ref.get('recorded', '?')})", "max_rel_loss_dev": rel, "tolerance": 1e-4, "ok": bool(rel <= 1e-4)}
    if a.record_ba_parity and n_gpus == 1:
        f = ROOT / "gpurun_out" / "ba_parity_n1.json"
        try:
            rec = json.loads(f.read_text())
        except Exception:
            rec = {}
        rec["first_order"] = {"losses": losses_rec, "recorded": f"loss at iterations 0 / 99 / 499, {T_total} frames x {J} joints x 2 per-frame cameras, float32, mode full"}
        f.parent.mkdir(exist_ok=True)
        f.write_text(json.dumps(rec, indent=1))
    out = {"metric": "ba_first_order_iterations_per_sec", "value": 1e3 / ms, "unit": "iters/s", "ms_per_iter": ms, "scaling": "strong",
           "frames_total": T * n_gpus, "frames_per_gpu": T, "joints": J,
           "cameras": 2, "mode": "full", "objective": "reproj + camera_smooth + baseline_reg + bone_length + pose_temporal (configs/vggt.yaml weights)",
           "timing": "(wall clock of 500 iterations - wall clock of 100) / 400: set-up and graph capture cancel; nothing synchronises inside",
           "collectives_per_iter": 0 if n_gpus == 1 else 3, "loss_first": h[0]["loss"], "loss_last": h[-1]["loss"], "parity": parity}
    if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline:
        from oracle import first_order as FO
        from oracle import torch_ref as TR

        torch.set_num_threads(os.cpu_count() or 1)
        Tc = 20_000
        c = lambda x: x[:Tc].detach().double().cpu()
        Xc, Rc, tc = c(X0).requires_grad_(True), c(R).requires_grad_(True), c(t).requires_grad_(True)
        Kc, xc, cc = torch.tensor(d["K"]), c(d["x2d"]), c(d["conf"])
        best = 1e9
        for _ in range(3):
            for v in (Xc, Rc, tc):
                v.grad = None
            t1 = time.perf_counter()
            FO.total_loss(TR.ReferenceNames, Xc, Rc, tc, Kc, xc, cc, FO.DEFAULT_WEIGHTS)[0].backward()
            best = min(best, time.perf_counter() - t1)
        out["cpu_baseline"] = {"value": 1.0 / (best * T / Tc), "unit": "iters/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": f"forward + backward of the five loss terms (torch restatement of loss.py, float64, all host threads) on "
                                         f"{Tc} of the {T} frames, scaled linearly"}
    del d, R, t, X0
    torch.cuda.empty_cache()
    return out


def run_ba(a, dev, world, rank, barrier, dist):
    """BA LM iterations/s (second half of BASELINE's metric).  Strong scaling: the clip's frames are
    split over the ranks; per LM trial the packed reduced camera system and the 3 trial scalars are
    all-reduced (NCCL)."""
    import torch

    from skiing_analysis_pytorch_b200 import api, ba, synth

    out = {}
    peak, _ = hbm_peak()
    ref_path = ROOT / "profiles" / "ba_parity_n1.json"
    try:
        parity_ref = json.loads(ref_path.read_text())
    except Exception:
        parity_ref = {}
    for name, (rig, T_total, J) in BA_CONFIGS.items():
        T = T_total // world
        # the clip is a function of the GLOBAL frame index: N ranks hold exactly the frames one GPU would (synth.make_clip_device
        # shardable=True), so the trajectory at N GPUs can be checked against the recorded single-GPU one
        d = synth.make_clip_device(rig, T, J, dev, seed=100, shardable=True, frame_offset=rank * T)
        R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
        C = len(R0)
        kv = d["x2d"].permute(1, 0, 2, 3).contiguous()
        X0 = api.triangulate_reproject(kv, d["K"], R0, t0, want=("X",)).X  # BA init = DLT under the perturbed rig
        del kv
        iters = a.ba_iters
        calib = name.endswith("_calib")
        if calib:
            th = synth.perturb_intrinsics(d["K"])
            K_init, dist_init = synth.theta_to_K_dist(th)
            X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), K_init, R0, t0, want=("X",)).X
            s = ba.CalibratingBundleAdjuster(d["x2d"], d["conf"], K_init, R0, t0, X0, dist=dist_init, prior_rho=synth.CALIB_PRIOR_RHO,
                                             prior_theta=synth.theta_from_K(d["K"]), max_iters=iters + 8)
        else:
            s = ba.BundleAdjuster(d["x2d"], d["conf"], d["K"], R0, t0, X0, max_iters=iters + 8)
        graph = not a.no_ba_graph  # one trial (launches + NCCL all-reduces) captured and replayed at every N
        s.run(4, graph=graph)  # warm-up trials (also captures the graph)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s.run(iters, graph=graph)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms.item()) / iters
        hist = s.history
        alg = T * J * (2 * 12 * C + 36)  # per rank: two streaming passes over the observations + X read twice, written once
        note = ("latency / issue-bound (22 us of HBM time per trial)" if C == 2 else "CUDA-core (fp32 FMA pipe) bound: ~5k FMA per point")
        if calib:
            note = "issue-bound: the 24 x 24 reduced system + two 17 x 17 camera blocks cost ~4k warp instructions per 32 points"
        # ---- parity against the recorded single-GPU trajectory of the same clip (profiles/ba_parity_n1.json, written by
        #      `bench.py --record-ba-parity` on one GPU): cost per trial and the accept / reject decisions while decisive
        costs = [h["cost"] for h in hist] + [s.cost]
        acc = [bool(h["accepted"]) for h in hist]
        parity = {"reference": "unrecorded", "ok": None}
        ref = parity_ref.get(name)
        if ref is not None:
            n = min(len(ref["costs"]), len(costs))
            rel = max(abs(x - y) / abs(y) for x, y in zip(costs[:n], ref["costs"][:n]))
            decisive = [abs(h["cost"] - h["trial_cost"]) > 1e-3 * h["cost"] for h in hist]
            same = all(x == y for x, y, dz in zip(acc, ref["accepted"], decisive) if dz)
            parity = {"reference": f"profiles/ba_parity_n1.json ({ref.get('recorded', '?')})", "trials_compared": n, "max_rel_cost_dev": rel,
                      "decisions_equal_while_decisive": same, "tolerance": 1e-5, "ok": bool(rel <= 1e-5 and same)}
        if a.record_ba_parity and world == 1:
            parity_ref[name] = {"costs": costs, "accepted": acc, "recorded": f"{T_total} frames x {J} joints x {C} cameras, seed 100, {len(hist)} trials"}
        out[name] = {
            "metric": "ba_lm_iterations_per_sec",
            "value": 1e3 / ms,
            "unit": "iters/s",
            "ms_per_iter": ms,
            "scaling": "strong",
            "frames_total": T * world,
            "frames_per_gpu": T,
            "joints": J,
            "cameras": C,
            "free_params_per_camera": 15 if calib else 6,
            "parameters": ("points + extrinsics (camera 0 = gauge) + fx fy cx cy k1 k2 p1 p2 k3 of every camera, Gaussian prior on the intrinsics"
                           if calib else "points + extrinsics (camera 0 = gauge)"),
            "launches_per_iter": 6,
            "collectives_per_iter": 0 if world == 1 else 2,
            "exchange": "none (one GPU)" if world == 1 else ("single-CTA push / flag / sum kernel over NVLink peer memory (csrc/ska_peer.cu)"
                                                            if s.peer is not None else "NCCL all-reduce (torch.distributed)"),
            "cuda_graph": graph,
            "cost_first": hist[0]["cost"],
            "cost_last": s.cost,
            "accepted": int(sum(h["accepted"] for h in hist)),
            "trials": len(hist),
            "parity": parity,
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "bytes_per_iter_per_gpu": alg,
                         "note": note + ", not HBM-bound: DESIGN.md section 6"},
        }
        del s, d, X0
        torch.cuda.empty_cache()
    try:
        out.update(run_ba_regularised(a, dev, world, rank, barrier, dist, parity_ref))
    except Exception as e:  # an extra leg: never lose the line over it
        out["config3_regularised"] = {"failed": repr(e)[:300]}
    if a.record_ba_parity and world == 1 and rank == 0:
        out_dir = ROOT / "gpurun_out"
        out_dir.mkdir(exist_ok=True)
        (out_dir / "ba_parity_n1.json").write_text(json.dumps(parity_ref, indent=1))
    return out


def run_ba_regularised(a, dev, world, rank, barrier, dist, parity_ref):
    """Row N1 / e3: LM over the reference's full configured objective (reprojection + bone length + pose temporal + camera
    smoothness + baseline, configs/vggt.yaml weights) with PER-FRAME cameras, config 3's shape (100k frames x 17 joints x
    2 cameras) sharded by frame range over the ranks: one-frame halos of the CG direction / trial point and all-reduced
    dot products and cost sums (NCCL) inside the captured trial.  Modes: pose_only (the yaml default: points only) and
    full (every frame's R and t free)."""
    import math

    import torch

    from skiing_analysis_pytorch_b200 import api, ba_reg, synth

    out = {}
    T_total, J, rig = 100_000, 17, "2b"
    T = T_total // world
    d = synth.make_clip_device(rig, T, J, dev, seed=100, shardable=True, frame_offset=rank * T)
    R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
    C = len(R0)
    X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), d["K"], R0, t0, want=("X",)).X.double()
    # per-frame cameras: the perturbed rig plus a slow drift that is a function of the GLOBAL frame index
    tg = torch.arange(rank * T, (rank + 1) * T, dtype=torch.float64, device=dev)
    drift = torch.stack([0.01 * torch.sin(2 * math.pi * tg / 200.0 + c) for c in range(C)], 1)[..., None] * torch.tensor([1.0, 0.5, 0.25], dtype=torch.float64, device=dev)
    R = torch.tensor(R0, device=dev)[None].expand(T, C, 3, 3).contiguous()
    t = (torch.tensor(t0, device=dev)[None] + drift).contiguous()
    iters = a.ba_iters
    for mode, cg_iters in (("pose_only", 6), ("full", 48)):
        name = f"config3_regularised_{mode}"
        s = ba_reg.RegularisedBundleAdjuster(d["x2d"], d["conf"], d["K"], R, t, X0, mode=mode, max_iters=iters + 8, cg_iters=cg_iters,
                                             group=dist.group.WORLD if world > 1 else None, local_only=world == 1)
        graph = not a.no_ba_graph
        s.run(3, graph=graph)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s.run(iters, graph=graph)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms.item()) / iters
        hist = s.history
        costs = [h["cost"] for h in hist] + [s.cost_value]
        acc = [bool(h["accepted"]) for h in hist]
        parity = {"reference": "unrecorded", "ok": None}
        ref = parity_ref.get(name)
        if ref is not None:
            n = min(len(ref["costs"]), len(costs))
            rel = max(abs(x - y) / abs(y) for x, y in zip(costs[:n], ref["costs"][:n]))
            decisive = [abs(h["cost"] - h["trial_cost"]) > 1e-9 * h["cost"] for h in hist]
            same = all(x == y for x, y, dz in zip(acc, ref["accepted"], decisive) if dz)
            parity = {"reference": f"profiles/ba_parity_n1.json ({ref.get('recorded', '?')})", "trials_compared": n, "max_rel_cost_dev": rel,
                      "decisions_equal_while_decisive": same, "tolerance": 1e-9, "ok": bool(rel <= 1e-9 and same)}
        if a.record_ba_parity and world == 1:
            parity_ref[name] = {"costs": costs, "accepted": acc, "recorded": f"{T_total} frames x {J} joints x {C} per-frame cameras, seed 100, {len(hist)} trials, {mode}"}
        cg = [h["cg_iters"] for h in hist]
        out[name] = {
            "metric": "ba_lm_iterations_per_sec", "value": 1e3 / ms, "unit": "iters/s", "ms_per_iter": ms, "scaling": "strong",
            "frames_total": T * world, "frames_per_gpu": T, "joints": J, "cameras": C, "mode": mode, "dtype": "f64",
            "objective": "reprojection + bone_length + pose_temporal + camera_smooth + baseline_reg (configs/vggt.yaml:46-50), per-frame cameras",
            "solver": "matrix-free CG, per-frame Schur-complement preconditioner, relative residual 1e-8", "cg_iters_per_trial": cg,
            "cg_iters_captured": cg_iters, "collectives_per_cg_iter": 0 if world == 1 else 3, "cuda_graph": graph,
            "exchange": "none (one GPU)" if world == 1 else ("single-CTA push / flag / sum kernels over NVLink peer memory (csrc/ska_peer.cu)"
                                                            if s.peer is not None else "NCCL (torch.distributed)"),
            "cost_first": hist[0]["cost"], "cost_last": s.cost_value, "terms_last": {k: hist[-1][k] for k in ba_reg.HIST_KEYS[9:14]},
            "accepted": int(sum(acc)), "trials": len(hist), "parity": parity,
        }
        del s
        torch.cuda.empty_cache()
    return out


def run_tri_8view(a, dev, world, barrier, dist, T=1_000_000, J=17, key="tri_kernel_8view",
                  label="1M frames x 17 joints x 8 views per GPU, confidence-weighted DLT + distortion scoring"):
    """The north star's target shape for the fused kernel: 1M frames x 17 joints x 8 views, confidence weighted
    (140 B/joint), per GPU; with T=500k, J=70 it is BASELINE config 4's per-GPU shard (4M frames over 8 GPUs).
    Reported as extra objects; the headline `value` stays config 2."""
    import torch

    from skiing_analysis_pytorch_b200 import api, synth

    V = 8
    d = synth.make_clip_device("8", T, J, dev, seed=11, layout="CTJ2")
    outs = {"X": torch.empty((T, J, 3), dtype=torch.float32, device=dev), "err": torch.empty((V, T, J), dtype=torch.float32, device=dev)}
    kw = dict(K=d["K"], R=d["R"], t=d["t"], dist=synth.DIST_CALIB, want=("X", "err"))
    for _ in range(3):
        api.triangulate_reproject(d["x2d"], conf=d["conf"], out=outs, **kw)
    barrier()
    steps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        api.triangulate_reproject(d["x2d"], conf=d["conf"], out=outs, **kw)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item()) / steps
    peak, _ = hbm_peak()
    bpj = 8 * V + 4 * V + 12 + 4 * V
    ach = bpj * T * J / (ms * 1e-3) / 1e9
    del outs
    return {"workload": label, "ms_per_step": ms,
            "value": world * T * J / (ms * 1e-3), "unit": UNIT, "steps": steps,
            "roofline": {"bound": "hbm", "kernel": "ska::tri_kernel_cta_vp<8,...> (bulk-async staged, one point per lane, per-view work packed over view pairs)", "achieved": ach, "peak": peak,
                         "unit": "GB/s", "frac": ach / peak, "bytes_per_joint": bpj, "traffic": recorded_traffic(key),
                         "note": "fp32-pipe bound: ~670 FMA-pipe cycles per 32 points against ~420 cycles of HBM time"}}


def run_fusion(a, dev, world, barrier, dist):
    """Row N3: two-view 3D fusion + adaptive EMA of 1M frames x 70 joints per GPU (fp64 like the reference's numpy);
    frames shard by range with no collective (the EMA chunks replay their own halo).  Extra object `fusion`."""
    import torch

    from skiing_analysis_pytorch_b200 import fusion, synth

    T, J = 1_000_000, 70
    small = synth.make_fusion_clip(2000, J, seed=0)
    reps = (T + 1999) // 2000
    d = {k: torch.from_numpy(v).to(dev).repeat(reps, 1, 1)[:T].contiguous() for k, v in small.items()}

    def timed(fn, n):
        for _ in range(3):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    ms_f = timed(lambda: fusion.fuse_clip(d["Xl"], d["Xr"], d["Ul"], d["Ur"], want=(), strict=False), 5)
    fused = fusion.fuse_clip(d["Xl"], d["Xr"], d["Ul"], d["Ur"], want=(), strict=False).fused
    ms_e = timed(lambda: fusion.temporal_smooth_ema(fused), 5)
    ms_r = timed(lambda: fusion.rigid_fuse_clip(d["Xl"], d["Xr"], strict=False), 5)
    peak, _ = hbm_peak()
    b_f, b_e, b_r = T * J * 104, T * J * 48, T * J * 72
    out = {"workload": "1M frames x 70 joints per GPU: Kabsch alignment + weak-perspective / cross-view confidences + softmax fusion, then adaptive EMA (fp64)",
           "fuse_ms": ms_f, "ema_ms": ms_e, "rigid_transform_3d_ms": ms_r, "value": world * T / ((ms_f + ms_e) * 1e-3), "unit": "frames/s",
           "roofline_rigid_transform_3d": {"bound": "hbm", "achieved": b_r / ms_r / 1e6, "peak": peak, "unit": "GB/s", "frac": b_r / ms_r / 1e6 / peak,
                                           "bytes_per_joint": 72, "note": "bundle_adjustment/fuse/fuse.py rigid_transform_3D: Umeyama on the torso joints + threshold fusion"},
           "roofline_fuse": {"bound": "hbm", "achieved": b_f / ms_f / 1e6, "peak": peak, "unit": "GB/s", "frac": b_f / ms_f / 1e6 / peak,
                             "bytes_per_joint": 104, "note": "three launches (moments, per-frame parameters, per-joint fusion) read the inputs twice + a 448 B/frame workspace: ~190 B/joint of DRAM traffic against 104 algorithmic; the moments and fusion stages run at 55-65 % of HBM on their own traffic: DESIGN.md 3.6"},
           "roofline_ema": {"bound": "hbm", "achieved": b_e / ms_e / 1e6, "peak": peak, "unit": "GB/s", "frac": b_e / ms_e / 1e6 / peak,
                            "bytes_per_joint": 48, "note": "chunks of 512 frames replay a 70-sample halo (+14 % reads)"}}
    del d, fused
    torch.cuda.empty_cache()
    return out


def run_post(a, dev, world, barrier, dist):
    """Row N2: post-triangulation triage (+ per-frame report) and Savitzky-Golay smoothing of 1M frames x 17 joints per GPU."""
    import torch

    from skiing_analysis_pytorch_b200 import api, post, synth

    T, J = 1_000_000, 17
    d = synth.make_clip_device("2b", T, J, dev, seed=21, layout="CTJ2")
    X = api.triangulate_reproject(d["x2d"], d["K"], d["R"], d["t"], want=("X",)).X
    K, R, t = d["K"][0], d["R"][1], d["t"][1]

    def timed(fn, n=5):
        for _ in range(3):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / n

    ms_plain = timed(lambda: post.post_triage(X, d["x2d"], K, K, R, t))
    ms_und = timed(lambda: post.post_triage(X, d["x2d"], K, K, R, t, dist1=synth.DIST_CALIB, dist2=synth.DIST_CALIB, conf=d["conf"]))
    ms_sg = timed(lambda: post.smooth_skeleton(X, 9, 2))
    peak, _ = hbm_peak()
    N = T * J
    out = {"workload": "1M frames x 17 joints per GPU: triage (pinhole reprojection, depth / error / confidence gates, per-frame report) and Savitzky-Golay smoothing",
           "triage_ms": ms_plain, "triage_undistort_conf_ms": ms_und, "savgol_ms": ms_sg, "value": world * N / (ms_plain * 1e-3), "unit": "joints/s",
           "roofline": {"bound": "hbm", "achieved": N * 45 / ms_plain / 1e6, "peak": peak, "unit": "GB/s", "frac": N * 45 / ms_plain / 1e6 / peak,
                        "bytes_per_joint": 45, "note": "fp64 arithmetic like the reference's numpy (identical accept / reject decisions)"}}
    del d, X
    torch.cuda.empty_cache()
    return out


def post_cpu_rate(frames=300):
    """The reference's per-frame numpy triage (array form, oracle/postprocess.py) on one core."""
    from oracle import geometry as G
    from oracle import postprocess as PP
    from skiing_analysis_pytorch_b200 import synth

    clip = synth.make_clip("2b", frames, 17, seed=0)
    P = np.stack([G.make_P(clip.K[v], clip.R[v], clip.t[v]) for v in range(2)])
    X = G.dlt_triangulate(P, clip.x_vm.reshape(2, -1, 2)).reshape(frames, 17, 3).astype(np.float32)
    t0 = time.perf_counter()
    PP.post_triage_sequence(X, clip.x_vm[0], clip.x_vm[1], clip.K[0], clip.K[1], clip.R[1], clip.t[1])
    return frames * 17 / (time.perf_counter() - t0)


def fusion_cpu_rate(frames=600):
    """The reference's per-frame numpy fusion + EMA (array form, oracle/fusion.py) on one core."""
    from oracle import fusion as F
    from skiing_analysis_pytorch_b200 import synth

    d = synth.make_fusion_clip(frames, 70, seed=0)
    t0 = time.perf_counter()
    fz, *_ = F.fuse_clip(d["Xl"], d["Xr"], d["Ul"], d["Ur"])
    F.temporal_smooth_ema(fz)
    return frames / (time.perf_counter() - t0)


DUMP_BYTES = 32 << 20


def dump_outputs(out_dir, outs):
    """Write the arrays the timed step returns (X, err) as float32 .npy files, so that two builds run with the same
    arguments can be compared output for output.  Above DUMP_BYTES the same seeded sample of frames is taken every run."""
    import torch

    X, err = outs["X"], outs["err"]
    T = X.shape[0]
    n = min(T, DUMP_BYTES // ((X[0].numel() + err[:, 0].numel()) * 4))
    if n == 0:
        raise SystemExit(f"--dump-outputs: one frame of X and err is larger than {DUMP_BYTES} bytes")
    if n < T:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(T, n, replace=False))).to(X.device)
        X, err = X[idx], err[:, idx]
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "X.npy", X.cpu().numpy())
    np.save(d / "err.npy", err.cpu().numpy())


def run_ours(a, out_fd=1):
    import torch
    import torch.distributed as dist

    from skiing_analysis_pytorch_b200 import api, hostlink, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = hostlink.bind_to_device_numa(dev)  # before any pinned allocation: this rank's host buffers belong next to its GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    T, J = a.frames, a.joints
    clip = synth.make_clip(a.rig, T, J, seed=rank)
    V = len(clip.R)
    dist_coeffs = None if a.pinhole else synth.DIST_CALIB
    # host side: pinned buffers (the e2e arm copies from / to these every step)
    h_k = torch.from_numpy(clip.x_vm).pin_memory()
    h_c = torch.from_numpy(clip.conf_vm).pin_memory() if a.conf else None
    d_k = h_k.to(dev, non_blocking=True)
    d_c = h_c.to(dev, non_blocking=True) if a.conf else None
    outs = {
        "X": torch.empty((T, J, 3), dtype=torch.float32, device=dev),
        "err": torch.empty((V, T, J), dtype=torch.float32, device=dev),
    }
    kw = dict(K=clip.K, R=clip.R, t=clip.t, dist=dist_coeffs, solver=a.solver, want=("X", "err"))

    def step():
        api.triangulate_reproject(d_k, conf=d_c, out=outs, **kw)

    for _ in range(max(a.warmup, 3)):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        ev0.record()
        for _ in range(a.steps):
            step()
        ev1.record()
        barrier()
        kernel_ms = ev0.elapsed_time(ev1)

        # ---- end to end through the host-buffer API: pinned H2D + kernel + D2H, every step.  The result a caller of
        #      process_triangulate consumes is the 3D joints and the per-frame reprojection statistics (triangulate.py:111-118
        #      reads mean_err_L / mean_err_R and returns the joints): want=("X", "stats").  The per-joint error arrays - the
        #      contents of reproject_and_visualize's dict - cost another 4 V J bytes per frame over PCIe: timed as well
        #      (`e2e_per_joint_errors`).
        h_X = torch.empty((T, J, 3), dtype=torch.float32).pin_memory()
        h_err = torch.empty((V, T, J), dtype=torch.float32).pin_memory()
        h_stats = torch.empty((T, V, 4), dtype=torch.float32).pin_memory()
        e2e_steps = max(3, min(a.steps, 10))
        kw_host = dict(kw, chunk_frames=a.e2e_chunk, n_streams=a.e2e_streams, graph=a.e2e_graph)

        def e2e_timed(want, host_out):
            kwh = dict(kw_host, want=want)
            for _ in range(2):
                api.triangulate_reproject_host(h_k, conf=h_c, out=host_out, **kwh)
            barrier()
            ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev2.record()
            for _ in range(e2e_steps):
                api.triangulate_reproject_host(h_k, conf=h_c, out=host_out, **kwh)
            ev3.record()
            barrier()
            return ev2.elapsed_time(ev3)

        e2e_ms = e2e_timed(("X", "stats"), {"X": h_X, "stats": h_stats})
        e2e_full_ms = e2e_timed(("X", "err"), {"X": h_X, "err": h_err})
        # what the host side gives with all ranks copying at once: the ceiling of the end-to-end number at this N
        link = hostlink.measure_link(dev, barrier=barrier)

    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, outs)  # the host-buffer arm writes its own buffers: outs still holds the last timed step
    t_k = torch.tensor([kernel_ms, e2e_ms, e2e_full_ms], dtype=torch.float64, device=dev)
    t_l = torch.tensor([link["h2d_alone"], link["d2h_alone"], link["both_each"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_k, op=dist.ReduceOp.MAX)
        dist.all_reduce(t_l, op=dist.ReduceOp.MIN)  # the slowest rank's rates
    kernel_ms, e2e_ms, e2e_full_ms = (float(x) for x in t_k.cpu())
    link_min = [float(x) for x in t_l.cpu()]

    pts = T * J
    value = n_gpus * pts * a.steps / (kernel_ms * 1e-3)
    e2e_value = n_gpus * pts * e2e_steps / (e2e_ms * 1e-3)
    bytes_per_pt = 8 * V + (4 * V if a.conf else 0) + 12 + 4 * V
    peak, peak_src = hbm_peak()
    achieved = bytes_per_pt * pts / (kernel_ms * 1e-3 / a.steps) / 1e9
    h2d = h_k.numel() * 4 + (h_c.numel() * 4 if a.conf else 0)
    d2h = h_X.numel() * 4 + h_stats.numel() * 4
    d2h_full = h_X.numel() * 4 + h_err.numel() * 4

    line = {
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": n_gpus,
        "steps": a.steps,
        "warmup": max(a.warmup, 3),
        "ms_per_step": kernel_ms / a.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(a, V),
        "clocks": clocks.summary(),
        "e2e": {
            "value": e2e_value,
            "unit": UNIT,
            "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h,
            "steps": e2e_steps,
            "ms_per_step": e2e_ms / e2e_steps,
            "pipeline": f"{a.e2e_chunk}-frame chunks on {a.e2e_streams} streams, " + ("replayed as one CUDA graph (copies + kernels)" if a.e2e_graph else "enqueued call by call"),
            "result": "X (T,J,3) + per-(frame, view) rmse / mean / median / max of the pixel errors (T,V,4): what process_triangulate consumes",
            "host_link": {
                "per_rank_h2d_alone": link_min[0], "per_rank_d2h_alone": link_min[1], "per_rank_both_each_direction": link_min[2],
                "aggregate_both": 2 * link_min[2] * n_gpus, "unit": "GB/s", "ranks_copying_at_once": n_gpus,
                "note": "pinned 256 MB copies timed in this run with every rank copying at the same time (slowest rank): the "
                        "end-to-end step moves max(h2d, d2h) bytes at the both-at-once rate, so it tracks this, not the kernel",
            },
            "link_bound_ms_per_step": max(h2d, d2h) / (link_min[2] * 1e9) * 1e3,
            "numa": numa,
        },
        "e2e_per_joint_errors": {
            "value": n_gpus * pts * e2e_steps / (e2e_full_ms * 1e-3),
            "unit": UNIT,
            "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h_full,
            "steps": e2e_steps,
            "ms_per_step": e2e_full_ms / e2e_steps,
            "result": "X (T,J,3) + the per-joint pixel error of every view (V,T,J)",
        },
        "gpu_launches": a.steps,
        "roofline": {
            "bound": "hbm",
            "kernel": "ska::tri_kernel_cta (15 consumer warps + producer thread, one bulk-async copy per view and group of 15 tiles, packed FFMA2 pairs)",
            "achieved": achieved,
            "peak": peak,
            "peak_source": peak_src,
            "unit": "GB/s",
            "frac": achieved / peak,
            "bytes_per_joint": bytes_per_pt,
            "traffic": recorded_traffic("tri_kernel_config2"),
            "traffic_source": "profiles/traffic.json: dram bytes of one launch from the committed ncu --set full capture of this kernel (not re-measured in this run)",
        },
    }

    if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline and V == 2:
        frames = min(T, a.cpu_sample_frames)
        rate, dt = cpu_reference_rate(clip, dist_coeffs, frames, 1)
        line["cpu_baseline"] = {
            "value": rate,
            "unit": UNIT,
            "cores": 1,
            "kind": "port",
            "seconds": dt,
            "sample": f"first {frames} frames x {J} joints of the same clip, single-process per-frame "
            "cv2.triangulatePoints + cv2.projectPoints loop (oracle/reference_path.py), as the reference runs it",
        }
    del d_k, d_c, outs, h_k, h_c, h_X, h_err, h_stats
    api.clear_host_pipeline_cache()
    torch.cuda.empty_cache()
    if not a.no_extra:
        line["tri_8view"] = run_tri_8view(a, dev, world, barrier, dist)
        torch.cuda.empty_cache()
        line["tri_config4"] = run_tri_8view(a, dev, world, barrier, dist, T=500_000, J=70, key="tri_kernel_config4",
                                            label="config4 shard: 500k frames x 70 joints x 8 views per GPU (4M frames over 8 GPUs), "
                                                  "confidence-weighted DLT + distortion scoring")
        torch.cuda.empty_cache()
    if not a.no_extra:
        line["fusion"] = run_fusion(a, dev, world, barrier, dist)
        if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline:
            line["fusion"]["cpu_baseline"] = {"value": fusion_cpu_rate(), "unit": "frames/s", "cores": 1, "kind": "port",
                                              "sample": "600 frames x 70 joints through the reference's per-frame numpy path (oracle/fusion.py)"}
    if not a.no_extra:
        line["post"] = run_post(a, dev, world, barrier, dist)
        if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline:
            try:
                line["post"]["cpu_baseline"] = {"value": post_cpu_rate(), "unit": "joints/s", "cores": 1, "kind": "port",
                                                "sample": "300 frames x 17 joints through the reference's per-frame numpy triage (oracle/postprocess.py)"}
            except Exception as e:  # the CPU leg is a reported baseline, never the thing measured
                line["post"]["cpu_baseline"] = {"unavailable": repr(e)[:200]}
    if not a.no_ba:
        line["ba"] = run_ba(a, dev, world, rank, barrier, dist)
        line["gpu_launches_ba_per_iter"] = 6
        try:
            line["ba"]["first_order"] = run_first_order(a, dev, rank, n_gpus, dist)
        except Exception as e:  # an extra leg: never lose the line over it
            line["ba"]["first_order"] = {"failed": repr(e)[:300]}
        if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline:
            r = ba_cpu_iteration_rate()
            line["ba"]["cpu_baseline"] = {
                "value": r, "unit": "iters/s at 1500 frames x 17 joints x 2 cameras", "cores": 1, "kind": "port",
                "extrapolated_config3_iters_per_sec": r * 1500 / 100_000,
                "sample": "3 LM trials of the fp64 numpy Schur-LM oracle (oracle/lm.py) on a 1500-frame config-3 clip; cost is "
                "linear in the frame count",
            }
    if rank == 0:
        os.write(out_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        from skiing_analysis_pytorch_b200 import peer

        torch.cuda.synchronize(dev)
        peer.close_all()
        dist.destroy_process_group()
    return 0


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    # stdout carries exactly ONE line (the JSON): libraries that print to fd 1 from C (NCCL's version banner) are sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        return run_ours(a, real_stdout)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)


if __name__ == "__main__":
    sys.exit(main())
