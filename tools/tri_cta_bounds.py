"""Where config 2's time goes in tri_kernel_cta (1 M frames x 17 joints x 2 views, distortion scoring): CUDA-event times of
several builds of the library in ONE process, alternated, so that every arm sees the same box, clocks and neighbours.

    python tools/variants.py build cta_s6 cta_s8 cta_s12 cta_l2 cta_nomath cta_clocks   (no GPU needed)
    python tools/tri_cta_bounds.py [--reps 5] [ARM ...]                                  (on the GPU)

ARM is a variant name of tools/variants.py (lib/libska_<name>.so), `product` (lib/libska.so) or NAME=PATH for any other
build of the library, e.g. the parent commit's.  Default: product and every cta_* variant that is built.

  product      the shipped kernel
  cta_l2       the producer copies from a 32-group window that stays in L2: the same instructions without HBM reads,
               i.e. the bound set by issue and the FMA pipe
  cta_nomath   the consumers skip the arithmetic but keep the staging, the vote and every store: the staging bound
  cta_s<N>     N shared-memory stages instead of 4
  *clocks      clock64() spent on the `full` barrier per consumer warp, summed over a launch and printed by the kernel;
               not timed (the counters cost registers), run on its own after the timing

The clip (612 MB of traffic) is five times the 126 MB L2, so the timed launches stream from HBM without a flush.
"""
import argparse
import ctypes as C
import statistics
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from skiing_analysis_pytorch_b200 import _cabi, _lib, api, synth  # noqa: E402

LIBDIR = ROOT / "skiing_analysis_pytorch_b200" / "lib"


def load(path):
    lib = C.CDLL(str(path))  # a distinct path is a distinct copy of the library, kernels and all
    for name, (res, args) in _lib._SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ska_abi_version() != _cabi.ABI_VERSION:
        raise RuntimeError(f"{path}: ABI {lib.ska_abi_version()} != {_cabi.ABI_VERSION}")
    return lib


def arms_from(args):
    if not args:
        args = ["product"] + sorted(p.stem[len("libska_"):] for p in LIBDIR.glob("libska_cta_*.so"))
    arms = []
    for a in args:
        if "=" in a:
            name, path = a.split("=", 1)
        elif a == "product":
            name, path = a, LIBDIR / "libska.so"
        else:
            name, path = a, LIBDIR / f"libska_{a}.so"
        arms.append((name, load(path)))
    return arms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("arms", nargs="*")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tri_cta_bounds: no CUDA device")
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}", flush=True)
    arms = arms_from(a.arms)
    _lib._LIB = arms[0][1]
    T, J = 1_000_000, 17
    d = synth.make_clip_device("2b", T, J, dev, seed=0, layout="CTJ2")
    V = d["x2d"].shape[0]
    outs = {"X": torch.empty((T, J, 3), dtype=torch.float32, device=dev), "err": torch.empty((V, T, J), dtype=torch.float32, device=dev)}
    kw = dict(K=d["K"], R=d["R"], t=d["t"], dist=synth.DIST_CALIB, want=("X", "err"), out=outs)
    mb = (8 * V + 12 + 4 * V) * T * J / 1e6

    def run():
        api.triangulate_reproject(d["x2d"], conf=None, **kw)

    def timed(n):
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    timed_arms = [(n, lib) for n, lib in arms if not n.endswith("clocks")]
    ms = {n: [] for n, _ in timed_arms}
    for _ in range(a.reps):
        for n, lib in timed_arms:
            _lib._LIB = lib
            ms[n].append(timed(a.launches))
    print(f"config 2 (1M x 17 x 2, {mb:.0f} MB), {a.reps} alternated repeats of {a.launches} launches, ms per launch:")
    for n, v in ms.items():
        med = statistics.median(v)
        print(f"  {n:16s} median {med:.4f}  min {min(v):.4f}  max {max(v):.4f}  ({mb / med:.0f} GB/s)  " + " ".join(f"{x:.4f}" for x in v),
              flush=True)
    libc = C.CDLL(None)
    for n, lib in arms:
        if n.endswith("clocks"):
            _lib._LIB = lib
            print(f"  {n}: three launches", flush=True)
            for _ in range(3):
                run()
                torch.cuda.synchronize()
                libc.fflush(None)  # the kernel's printf lines, in order with ours


if __name__ == "__main__":
    main()
