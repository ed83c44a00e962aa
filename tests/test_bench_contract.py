"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (the CPU oracle port, the one other place
bench.py may execute oracle/) prints exactly ONE JSON line with the keys the driver reads, also under torchrun (rank 0 only);
our arm refuses to run without a CUDA device instead of falling back to anything.  On a GPU: --dump-outputs writes the same
outputs of the last timed step run after run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "cpu_baseline", "e2e"}


def _json_lines(out):
    return [json.loads(l) for l in out.splitlines() if l.startswith("{")]


def _check_reference_line(line, n_gpus):
    assert REQUIRED <= set(line), REQUIRED - set(line)
    assert line["impl"] == "reference" and line["metric"] == "env-steps/s" and line["unit"] == "env-steps/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None and line["n_gpus"] == n_gpus
    assert line["config"]["workload"].startswith("QuadX-Hover") and line["config"]["global_envs"] == n_gpus * line["config"]["envs_per_gpu"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "oracle" in cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_reference_arm_prints_one_line():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "2", "--warmup", "3", "--envs", "512"], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1, r.stdout
    _check_reference_line(lines[0], 1)


def test_reference_arm_under_torchrun_rank0_only():
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "3", "--envs", "256"],
                       cwd=ROOT, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1, r.stdout  # the other rank exits 0 without work
    _check_reference_line(lines[0], 2)


def test_our_arm_fails_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("needs a box without a CUDA device")
    r = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "3", "--no-cpu-baseline"], cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode != 0
    assert not [l for l in _json_lines(r.stdout) if "value" in l]  # no number without the CUDA path


def test_dump_outputs_are_float32_and_sampled_above_the_limit(monkeypatch):
    import types

    import numpy as np
    import torch

    import bench

    n, obs_dim = 1000, 5
    g = torch.Generator().manual_seed(0)
    av = types.SimpleNamespace(num_drones=n, obs=torch.rand((n, obs_dim), generator=g), reward=torch.rand(n, generator=g),
                               term=torch.randint(0, 2, (n,), dtype=torch.uint8, generator=g),
                               trunc=torch.randint(0, 2, (n,), dtype=torch.uint8, generator=g),
                               info_bits=torch.randint(0, 8, (n,), dtype=torch.uint8, generator=g))
    env = types.SimpleNamespace(aviary=av)
    full = bench.timed_step_outputs(env)
    assert "env_index" not in full and all(a.dtype == np.float32 and len(a) == n for a in full.values())
    assert np.array_equal(full["obs"], av.obs.numpy()) and np.array_equal(full["terminated"], av.term.numpy())
    bits = av.info_bits.numpy()
    assert np.array_equal(full["info_out_of_bounds"], bits & 1) and np.array_equal(full["info_collision"], (bits >> 1) & 1)
    assert np.array_equal(full["info_env_complete"], (bits >> 2) & 1)

    row_bytes = (obs_dim + 6) * 4 + 8  # six per-env scalars and the float64 env index
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100 * row_bytes)
    part = bench.timed_step_outputs(env)
    keep = part.pop("env_index")
    assert keep.dtype == np.float64 and len(keep) == 100 and np.all(np.diff(keep) > 0)
    assert sum(a.nbytes for a in part.values()) + keep.nbytes <= bench.DUMP_LIMIT_BYTES
    for name, a in part.items():
        assert np.array_equal(a, full[name][keep.astype(np.int64)]), name
    assert np.array_equal(bench.timed_step_outputs(env)["env_index"], keep)  # the sample is fixed


@pytest.mark.gpu
def test_dump_outputs_repeat_run_after_run(tmp_path):
    import numpy as np

    cmd = [sys.executable, "bench.py", "--steps", "5", "--warmup", "3", "--envs", "8192", "--batches", "2", "--repeats", "2", "--no-cpu-baseline"]
    for run in ("a", "b"):
        r = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / run)], cwd=ROOT, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = _json_lines(r.stdout)
        assert len(lines) == 1 and lines[0]["steps"] == 5
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "obs.npy" in names and "reward.npy" in names
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float32 and len(a) == 8192 and np.array_equal(a, b), name
    assert np.isfinite(np.load(tmp_path / "a" / "obs.npy")).all()
