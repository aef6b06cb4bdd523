"""Build experimental variants of libska.so so ONE gpurun call can time them side by side.  Only the translation
units named in TUS are recompiled with the variant's flags; every other object comes from the product build.

    python tools/variants.py build [names...]     (here, no GPU)
    python tools/variants.py run [names...]       (on the GPU box; BENCH = script + args, default tools/tri_bench.py c2 v8)
"""
import os
import shlex
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
TUS = ["ska_tri_v2.cu"]
VARIANTS = {
    "A": [],
    "B": ["-DSKA_FR_WARPS=10", "-DSKA_FR_PRODUCERS=2", "-DSKA_FR_STAGES=4"],
    "C": ["-DSKA_FR_STAGES=6"],
    # tri_kernel_cta on config 2 (tools/tri_cta_bounds.py): ring depth, and three builds that exist only to be measured
    "cta_s6": ["-DSKA_CTA_STAGES=6"],
    "cta_s8": ["-DSKA_CTA_STAGES=8"],
    "cta_s12": ["-DSKA_CTA_STAGES=12"],
    "cta_l2": ["-DSKA_CTA_L2_WINDOW"],
    "cta_nomath": ["-DSKA_CTA_NO_MATH"],
    "cta_clocks": ["-DSKA_CTA_WAIT_CLOCKS"],
}
LIBDIR = ROOT / "skiing_analysis_pytorch_b200" / "lib"


def build_variant(name):
    from skiing_analysis_pytorch_b200 import build as B

    B.build()  # product objects up to date
    vdir = B.CSRC / f"_obj_{name}"
    vdir.mkdir(exist_ok=True)
    objs = []
    for src in B.sources():
        if src.name in TUS:
            obj = vdir / (src.stem + ".o")
            cmd = [B._nvcc(), *B.ARCH_FLAGS, *B.NVCC_FLAGS, *VARIANTS[name], "-I", str(ROOT / "include"), "-c", str(src), "-o", str(obj)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(r.stderr)
            objs.append(obj)
        else:
            objs.append(B.OBJ / (src.stem + ".o"))
    out = LIBDIR / f"libska_{name}.so"
    r = subprocess.run([B._nvcc(), *B.ARCH_FLAGS, "-shared", "-o", str(out), *map(str, objs), "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(r.stderr)
    return out


def main():
    cmd = sys.argv[1]
    names = sys.argv[2:] or list(VARIANTS)
    if cmd == "build":
        from skiing_analysis_pytorch_b200 import build as B

        B.build()
        with ThreadPoolExecutor(max_workers=4) as ex:
            for n, p in zip(names, ex.map(build_variant, names)):
                print(n, p)
    else:
        bench = shlex.split(os.environ.get("BENCH", "tools/tri_bench.py c2 v8"))
        for n in names:
            env = dict(os.environ, SKA_LIB_PATH=str(LIBDIR / f"libska_{n}.so"))
            print(f"== {n}: {' '.join(VARIANTS[n])}", flush=True)
            r = subprocess.run([sys.executable, *bench], env=env, capture_output=True, text=True, cwd=ROOT)
            print(r.stdout.strip() if r.returncode == 0 else f"FAILED rc={r.returncode}\n{r.stdout[-500:]}\n{r.stderr[-800:]}", flush=True)


if __name__ == "__main__":
    main()
