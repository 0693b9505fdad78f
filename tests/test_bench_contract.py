"""bench.py contract on CPU: the reference arm runs without a GPU and prints one JSON line with
the keys the driver reads; the native arm refuses to run without CUDA (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c3", "--steps", "1", "--warmup", "1",
                          "--cpu-sample-pairs", "2e5"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "pairwise_loss_gpairs_per_s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_dumps_identical_outputs(tmp_path):
    import numpy as np

    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c3", "--steps", "2", "--warmup", "1",
                              "--cpu-sample-pairs", "2e5", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    assert sorted(dumps[0]) == ["loss", "loss_grad"]
    assert dumps[0]["loss_grad"].shape == (2493, 3) and dumps[0]["loss_grad"].dtype == np.float32
    assert dumps[0]["loss"].dtype == np.float64 and dumps[0]["loss"][0] > 0
    for name, a in dumps[0].items():
        assert np.array_equal(a, dumps[1][name]), name


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_native_arm_needs_cuda():
    import torch

    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_native_arm_dumps_the_last_timed_step(tmp_path):
    import numpy as np

    n = 2493
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c3", "--steps", "3", "--warmup", "3", "--train-steps", "2",
                          "--configs", "none", "--no-e2e", "--no-sparse", "--no-cpu-baseline", "--no-measure-copy", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    d = {f.stem: np.load(f) for f in sorted(tmp_path.glob("*.npy"))}
    assert sorted(d) == ["loss_grad", "loss_moments", "train_moments", "train_total"]
    assert d["loss_grad"].shape == (n, 3) and d["loss_grad"].dtype == np.float32 and np.isfinite(d["loss_grad"]).all()
    assert d["loss_moments"].dtype == np.float64 and d["loss_moments"][0] / n**2 == line["check"]["mse"]
    g = d["loss_grad"].astype(np.float64)
    assert np.abs(g.sum(0)).max() <= 1e-4 * np.abs(g).sum(0).max()  # translation invariance: sum_i grad_i = 0
    assert float(d["train_total"][0]) == line["train"]["total_loss"]


def test_committed_native_lines_carry_the_contract_keys():
    """The B200 lines committed under profiles/ (what DESIGN.md quotes) have every key the driver / judge reads, a
    roofline consistent with its own fields, a CPU baseline and an end-to-end number with real copies."""
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r1_bench_c*_n[0-9].json")))
    assert len(files) >= 4
    for f in files:
        line = json.loads(open(f).read().strip().splitlines()[-1])
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                    "config", "roofline", "e2e", "gpu_launches", "clocks"):
            assert key in line, (f, key)
        assert line["metric"] == "pairwise_loss_gpairs_per_s" and line["unit"] == "Gpairs/s" and line["higher_is_better"] is True
        assert line["warmup"] >= 3 and line["gpu_launches"] > 0 and "workload" in line["config"]
        r = line["roofline"]
        assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert abs(r["achieved"] - r["algorithmic_bytes"] / (r["kernel_ms"] * 1e-3) / 1e9) < 1e-6 * r["achieved"]
        assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0 and line["e2e"]["value"] < line["value"]
        bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(line["clocks"]["reasons"])
        assert not bad, (f, bad)
        if line["n_gpus"] == 1 and "c5" in os.path.basename(f):
            cb = line["cpu_baseline"]
            assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and "sample" in cb
