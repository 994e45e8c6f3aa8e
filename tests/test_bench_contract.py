"""The CPU arm of bench.py (`--impl reference`) prints one JSON line with the contract's keys (runs without a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--grid", "200x300", "--nt", "50"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]
    # nothing extrapolated: ms_per_step is the measured time of the step that ran
    assert d["ms_per_step"] * d["steps"] < 60e3


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
                          "--grid", "200x300", "--nt", "50"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096)
    small = np.arange(12, dtype=np.float32).reshape(3, 4)
    big = np.arange(5000, dtype=np.float64).reshape(50, 100)
    bench.dump_outputs(str(tmp_path / "a"), {"small": small, "big": big})
    bench.dump_outputs(str(tmp_path / "b"), {"small": small, "big": big})
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)
    s = np.load(tmp_path / "a" / "big.npy")
    assert s.dtype == np.float64 and 0 < s.nbytes <= 2048
    assert np.all(np.diff(s) > 0) and np.all(np.isin(s, big))                    # distinct elements, in index order
    assert np.array_equal(s, np.load(tmp_path / "b" / "big.npy"))                 # the same sample on every run


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_rejected_arguments(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == "", out.stderr[-2000:]


@pytest.mark.gpu
def test_b200_arm_dumps_the_gradient_of_the_timed_steps(tmp_path):
    """--dump-outputs holds the gradient summed over the timed shots (the warm-up shots excluded) and is identical between
    runs with the same arguments."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import bench
    from full_waveform_inversion_b200 import acoustic as ac
    argv = ["--steps", "3", "--warmup", "2", "--grid", "200x300", "--nt", "120", "--settle-idle", "0",
            "--no-track-a", "--no-extras", "--no-configs", "--no-cpu-baseline"]
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv, "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
    got = np.load(tmp_path / "a" / "gradient.npy")
    assert np.array_equal(got, np.load(tmp_path / "b" / "gradient.npy"))

    class _Args:
        grid, nt = "200x300", 120
    w = bench.workload(_Args)
    dev = torch.device("cuda", 0)
    prop = ac.Propagator2D((w["nz"], w["nx"]), w["h"], w["dt"], nabs=w["nabs"], alpha=w["alpha"], device=0)
    v, wav = torch.from_numpy(w["v"]).to(dev), torch.from_numpy(w["wav"]).to(dev)
    grad = torch.zeros((w["nz"], w["nx"]), dtype=torch.float32, device=dev)
    for src, rec in w["shots"][2:5]:
        prop.set_geometry(src, rec)
        prop.set_model(v * 1.02)
        obs = prop.forward(wav).clone()
        prop.set_model(v)
        prop.gradient(wav, obs, grad=grad, want_misfit=False)
    want = grad.cpu().numpy()
    prop.close()
    assert got.dtype == np.float32 and got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
