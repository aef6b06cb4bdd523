"""Time one graph-captured LM trial per loss (l2 / huber / cauchy) on the full BASELINE shapes, one GPU:
    python tools/ba_robust_bench.py [--rounds R] [--reps N] [--cases c3,c3_calib,c5,c3_reg_pose_only,c3_reg_full]
Configurations: c3 (100k x 17 x 2), c3 calibrating (free intrinsics + distortion), c5 (1M x 70 x 8) - the static-rig
Schur LM - and c3_reg_pose_only / c3_reg_full: the regularised LM over per-frame cameras on config 3's shape, set up as
bench.py's config3_regularised legs (seed 100, a slow camera drift, 6 / 48 captured CG iterations).  The three losses of a
configuration are captured once each and their replays alternated in the same process (R rounds of N replays, CUDA events);
the median over rounds is reported.  Every trial reads the whole clip (c5: 4.5 GB of observations), far beyond the L2
cache.  The robust kernels take a select (Huber) or a reciprocal and a log (Cauchy) per observation, no divergence, so the
clip carries no injected outliers.  A regularised trial's time also depends on how many of its captured CG iterations
run before the convergence flag stops them (the mean count is printed beside it), so the launches that read the
observations - linearize, the matrix-vector product, the CG update with the preconditioner - are also timed one by one
at the starting point, the losses alternated in the same way."""
import argparse
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from skiing_analysis_pytorch_b200 import _cabi, api, ba, ba_reg, synth  # noqa: E402

CASES = [("c3", "2b", 100_000, 17, False), ("c3_calib", "2b", 100_000, 17, True), ("c5", "8", 1_000_000, 70, False)]
REG_CASES = [("c3_reg_pose_only", "pose_only", 6), ("c3_reg_full", "full", 48)]
LOSSES = (("l2", None), ("huber", 3.0), ("cauchy", 3.0))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the card name still identifies the measurement
        q = f"power limit not readable ({e})"
    return f"{name}, {q}"


def alternate(solvers, rounds, reps):
    """{loss: [ms per trial of each round]}: every solver's captured trial replayed `reps` times per round, in turn."""
    for s in solvers.values():
        s.run(2, graph=True)  # warm-up trial + capture + one replay
    torch.cuda.synchronize()
    times = {loss: [] for loss in solvers}
    for _ in range(rounds):
        for loss, s in solvers.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            s.run(reps, graph=True)
            e1.record()
            torch.cuda.synchronize()
            times[loss].append(e0.elapsed_time(e1) / reps)
    return times


def reg_launch_times(solvers, rounds, reps):
    """{(loss, launch): [ms per launch of each round]} at the solvers' current points, CG kept running (convergence flag 0)."""
    launches = {"linearize": lambda s: s.linearize(), "matvec": lambda s: s.cg(_cabi.BA_REG_CG_MATVEC),
                "precond": lambda s: s.cg(_cabi.BA_REG_CG_UPDATE)}
    times = {}
    for _ in range(rounds):
        for loss, s in solvers.items():
            for name, fn in launches.items():
                s.sc[13] = 0.0  # SC_DONE
                fn(s)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn(s)
                e1.record()
                torch.cuda.synchronize()
                times.setdefault((loss, name), []).append(e0.elapsed_time(e1) / reps)
    return times


def regularised(args, dev):
    T, J = 100_000, 17
    d = synth.make_clip_device("2b", T, J, dev, seed=100, shardable=True, frame_offset=0)
    R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
    C = len(R0)
    X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), d["K"], R0, t0, want=("X",)).X.double()
    tg = torch.arange(T, dtype=torch.float64, device=dev)
    drift = torch.stack([0.01 * torch.sin(2 * math.pi * tg / 200.0 + c) for c in range(C)], 1)[..., None] * torch.tensor([1.0, 0.5, 0.25], dtype=torch.float64, device=dev)
    R = torch.tensor(R0, device=dev)[None].expand(T, C, 3, 3).contiguous()
    t = (torch.tensor(t0, device=dev)[None] + drift).contiguous()
    for name, mode, cg_iters in REG_CASES:
        if name not in args.cases:
            continue
        nmax = 2 + args.rounds * args.reps
        solvers = {loss: ba_reg.RegularisedBundleAdjuster(d["x2d"], d["conf"], d["K"], R, t, X0, mode=mode, max_iters=nmax, cg_iters=cg_iters,
                                                          local_only=True, loss=loss, loss_scale=sc) for loss, sc in LOSSES}
        lt = reg_launch_times(solvers, args.rounds, args.reps)
        for (loss, launch), ts in lt.items():
            med, base = float(np.median(ts)), float(np.median(lt[("l2", launch)]))
            print(f"{name:16s} T={T} J={J} C={C} {loss:6s} {launch:9s}: {med:8.3f} ms/launch (median of {args.rounds} x {args.reps}; "
                  f"min {min(ts):.3f} max {max(ts):.3f})  {100.0 * (med / base - 1.0):+5.1f} % vs l2")
        times = alternate(solvers, args.rounds, args.reps)
        base = float(np.median(times["l2"]))
        for loss, ts in times.items():
            med = float(np.median(ts))
            cg = np.mean([h["cg_iters"] for h in solvers[loss].history])
            print(f"{name:16s} T={T} J={J} C={C} {loss:6s}: {med:8.3f} ms/trial (median of {args.rounds} x {args.reps}; min {min(ts):.3f} "
                  f"max {max(ts):.3f})  {100.0 * (med / base - 1.0):+5.1f} % vs l2   CG iterations/trial {cg:.1f} of {cg_iters}   "
                  f"final cost {solvers[loss].cost_value:.4f}")
        del solvers
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cases", default=",".join([c[0] for c in CASES] + [c[0] for c in REG_CASES]))
    args = ap.parse_args()
    args.cases = args.cases.split(",")
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    print(f"# {card()}")
    for name, rig, T, J, calib in CASES:
        if name not in args.cases:
            continue
        d = synth.make_clip_device(rig, T, J, dev, seed=0)
        R0, t0 = synth.perturb_cameras(d["R"], d["t"], seed=1)
        K = d["K"]
        kw = {}
        if calib:
            K, dist = synth.theta_to_K_dist(synth.perturb_intrinsics(d["K"]))
            kw = dict(dist=dist, prior_rho=synth.CALIB_PRIOR_RHO, prior_theta=synth.theta_from_K(d["K"]))
        X0 = api.triangulate_reproject(d["x2d"].permute(1, 0, 2, 3).contiguous(), K, R0, t0, want=("X",)).X
        cls = ba.CalibratingBundleAdjuster if calib else ba.BundleAdjuster
        nmax = 2 + args.rounds * args.reps
        solvers = {loss: cls(d["x2d"], d["conf"], K, R0, t0, X0, max_iters=nmax, loss=loss, loss_scale=sc, **kw) for loss, sc in LOSSES}
        times = alternate(solvers, args.rounds, args.reps)
        base = float(np.median(times["l2"]))
        for loss, ts in times.items():
            med = float(np.median(ts))
            print(f"{name:9s} T={T} J={J} C={len(R0)} {loss:6s}: {med:8.3f} ms/trial (median of {args.rounds} x {args.reps}; "
                  f"min {min(ts):.3f} max {max(ts):.3f})  {100.0 * (med / base - 1.0):+5.1f} % vs l2   final cost {solvers[loss].cost:.4f}")
        del solvers, d, X0
        torch.cuda.empty_cache()
    if any(c[0] in args.cases for c in REG_CASES):
        regularised(args, dev)


if __name__ == "__main__":
    main()
