"""bench.py's contract: on the CPU the reference arm's JSON line, the host-thread sizing and the output dump; on the GPU a small
run of the GPU arm with --dump-outputs."""
import json
import os
import subprocess
import sys

import pytest

from tests.util import ROOT


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--preroll", "5"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["metric"].startswith("env-steps/sec") and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_host_threads_respects_affinity_and_quota():
    sys.path.insert(0, ROOT)
    import bench

    n, quota = bench.host_threads()
    assert 1 <= n <= len(os.sched_getaffinity(0))
    if quota is not None:
        assert n <= max(1, int(quota + 0.5))


def test_dump_outputs_writes_float_arrays_and_samples_the_same_rows_above_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np

    a = np.arange(40, dtype=np.float64).reshape(20, 2)
    b = np.arange(20, dtype=np.int32)
    bench.dump_outputs(str(tmp_path / "full"), {"a": a, "b": b})
    assert np.array_equal(np.load(tmp_path / "full" / "a.npy"), a) and np.load(tmp_path / "full" / "a.npy").dtype == np.float64
    got = np.load(tmp_path / "full" / "b.npy")
    assert got.dtype == np.float32 and np.array_equal(got, b)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", (a.nbytes + 4 * b.size) // 2)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"a": a, "b": b})
    sa, sb = np.load(tmp_path / "s1" / "a.npy"), np.load(tmp_path / "s1" / "b.npy")
    assert sa.shape == (10, 2) and sb.shape == (10,) and np.array_equal(sa[:, 0] // 2, sb)  # the same environments in every array
    assert np.array_equal(sa, np.load(tmp_path / "s2" / "a.npy"))


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert r.returncode != 0 and "GPU arm only" in r.stderr


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    """a small batch through bench.py: the steps count, and the dump holds the engine state and e2e outputs of every environment"""
    import numpy as np

    env = dict(os.environ, B2S_BENCH_SCALE="0.01")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--preroll", "2", "--no-cpu-baseline",
                        "--no-timeline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 4 and d["config"]["envs_per_gpu"] == 40
    names = sorted(os.listdir(tmp_path))
    assert names == sorted([f"Lift_Panda_{k}.npy" for k in ("qpos", "qvel", "qacc", "ctrl", "obs", "task_out")] + ["e2e_obs.npy", "e2e_reward.npy"])
    for n in names:
        a = np.load(tmp_path / n)
        assert a.dtype == np.float32 and a.shape[0] == 40 and np.isfinite(a).all(), n
    assert np.abs(np.load(tmp_path / "Lift_Panda_qvel.npy")).max() > 0


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
