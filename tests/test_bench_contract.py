"""bench.py contract checks: the reference arm prints ONE JSON line with the expected keys, the product arm
refuses to run without a CUDA device (there is no CPU fallback to time), and --dump-outputs writes what the timed
step computed."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-sample-frames", "256"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "triangulated_joints_per_sec" and j["unit"] == "joints/s"
    assert j["higher_is_better"] is True and j["value"] > 0 and j["steps"] == 1
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "joints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in j["config"] and "model" not in j["config"]


def test_product_arm_needs_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert "no CPU path" in (r.stderr + r.stdout)


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_dump_outputs_samples_the_same_frames_under_the_size_cap(tmp_path):
    import numpy as np
    import torch

    import bench

    T, J, V = 200_000, 17, 2
    g = torch.Generator().manual_seed(0)
    outs = {"X": torch.randn(T, J, 3, generator=g), "err": torch.rand(V, T, J, generator=g)}
    outs["X"][:, 0, 0] = torch.arange(T, dtype=torch.float32)  # names the frame
    bench.dump_outputs(tmp_path / "a", outs)
    bench.dump_outputs(tmp_path / "b", outs)
    X, err = np.load(tmp_path / "a" / "X.npy"), np.load(tmp_path / "a" / "err.npy")
    assert X.dtype == np.float32 and err.dtype == np.float32
    assert X.nbytes + err.nbytes <= bench.DUMP_BYTES and X.shape[1:] == (J, 3) and err.shape == (V, X.shape[0], J)
    assert X.shape[0] > T // 4
    rows = X[:, 0, 0].astype(np.int64)
    assert (np.diff(rows) > 0).all()
    assert np.array_equal(X, outs["X"].numpy()[rows]) and np.array_equal(err, outs["err"].numpy()[:, rows])
    for name in ("X.npy", "err.npy"):
        assert (tmp_path / "a" / name).read_bytes() == (tmp_path / "b" / name).read_bytes()
    small = {"X": outs["X"][:1000], "err": outs["err"][:, :1000]}
    bench.dump_outputs(tmp_path / "c", small)
    assert np.array_equal(np.load(tmp_path / "c" / "X.npy"), small["X"].numpy())
    assert np.array_equal(np.load(tmp_path / "c" / "err.npy"), small["err"].numpy())
    huge = {"X": torch.zeros(1, 2_000_000, 3), "err": torch.zeros(V, 1, 2_000_000)}  # 40 MB per frame: no sample fits
    with pytest.raises(SystemExit, match="larger than"):
        bench.dump_outputs(tmp_path / "d", huge)


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_steps_result(cuda, tmp_path):
    import numpy as np
    import torch

    from skiing_analysis_pytorch_b200 import api, synth

    T = 5000
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "1", "--frames", str(T), "--no-extra", "--no-ba",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-800:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    clip = synth.make_clip("2b", T, 17, seed=0)
    res = api.triangulate_reproject(torch.from_numpy(clip.x_vm).to(cuda), clip.K, clip.R, clip.t, dist=synth.DIST_CALIB, want=("X", "err"))
    assert np.array_equal(np.load(tmp_path / "X.npy"), res.X.cpu().numpy())
    assert np.array_equal(np.load(tmp_path / "err.npy"), res.err.cpu().numpy())
