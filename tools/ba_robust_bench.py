"""Time one graph-captured LM trial per loss (l2 / huber / cauchy) on the full BASELINE shapes, one GPU:
    python tools/ba_robust_bench.py [--rounds R] [--reps N]
Configurations: c3 (100k x 17 x 2), c3 calibrating (free intrinsics + distortion), c5 (1M x 70 x 8).  The three losses of a
configuration are captured once each and their replays alternated in the same process (R rounds of N replays, CUDA events);
the median over rounds is reported.  Every trial reads the whole clip (c5: 4.5 GB of observations), far beyond the L2
cache.  The robust kernels take a select (Huber) or a reciprocal and a log (Cauchy) per observation, no divergence, so the
clip carries no injected outliers."""
import argparse
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from skiing_analysis_pytorch_b200 import api, ba, synth  # noqa: E402

CASES = [("c3", "2b", 100_000, 17, False), ("c3_calib", "2b", 100_000, 17, True), ("c5", "8", 1_000_000, 70, False)]
LOSSES = (("l2", None), ("huber", 3.0), ("cauchy", 3.0))


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the card name still identifies the measurement
        q = f"power limit not readable ({e})"
    return f"{name}, {q}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda:0")
    print(f"# {card()}")
    for name, rig, T, J, calib in CASES:
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
        for s in solvers.values():
            s.run(2, graph=True)  # warm-up trial + capture + one replay
        torch.cuda.synchronize()
        times = {loss: [] for loss in solvers}
        for _ in range(args.rounds):
            for loss, s in solvers.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                s.run(args.reps, graph=True)
                e1.record()
                torch.cuda.synchronize()
                times[loss].append(e0.elapsed_time(e1) / args.reps)
        base = float(np.median(times["l2"]))
        for loss, ts in times.items():
            med = float(np.median(ts))
            print(f"{name:9s} T={T} J={J} C={len(R0)} {loss:6s}: {med:8.3f} ms/trial (median of {args.rounds} x {args.reps}; "
                  f"min {min(ts):.3f} max {max(ts):.3f})  {100.0 * (med / base - 1.0):+5.1f} % vs l2   final cost {solvers[loss].cost:.4f}")
        del solvers, d, X0
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
