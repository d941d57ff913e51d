"""bench.py's contract on CPU: the reference arm prints ONE JSON line with the required keys; the
GPU arm refuses to run without a device (no CPU fallback); under a multi-rank launch only rank 0
of the reference arm prints.  (The GPU arm's own line is checked where it runs, on the B200.)"""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env=None, timeout=600):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=timeout, env=e)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--vars-per-gpu", "2000"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["metric"] == "maxsum_edge_message_updates_per_s" and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["config"]["n_vars"] == 2000


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--vars-per-gpu", "500", "--gpus", "2"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_keeps_float_types_and_samples_to_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    small = {"value": np.arange(10, dtype=np.int32), "q": np.linspace(0, 1, 7, dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / "a"), small)
    v, q = np.load(tmp_path / "a" / "value.npy"), np.load(tmp_path / "a" / "q.npy")
    assert v.dtype == np.float64 and v.tolist() == list(range(10))
    assert q.dtype == np.float32 and np.array_equal(q, small["q"])
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    big = {"value": np.arange(100, dtype=np.int32), "r": np.arange(5000, dtype=np.float64)}
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), big)
    files = [tmp_path / "b" / "value.npy", tmp_path / "b" / "r.npy"]
    assert sum(np.load(f).nbytes for f in files) <= 4000
    assert np.load(files[0]).tolist() == list(range(100))          # under its share: kept whole
    r = np.load(files[1])
    assert len(r) == 250 and np.all(np.diff(r) > 0) and set(r) <= set(big["r"])
    assert np.array_equal(r, np.load(tmp_path / "c" / "r.npy"))     # the same sample every run


@pytest.mark.gpu
def test_gpu_arm_dumps_the_state_of_its_last_timed_step(tmp_path):
    """--steps K --warmup W runs exactly max(3, W) + K cycles: the dump equals a fresh engine stepped that often."""
    import numpy as np
    from pydcop_b200 import MaxSumEngine, build_layout
    from pydcop_b200.generators import config_c2
    r = _run(["--steps", "4", "--warmup", "3", "--vars-per-gpu", "20000", "--no-cpu-baseline", "--no-e2e",
              "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 4
    eng = MaxSumEngine(build_layout(**config_c2(seed=0, n_vars=20000)), device="cuda:0",
                       precision="f32").init().step(3 + 4)
    value, value_cost = eng.values()
    q, r_ = eng.messages()
    for name, want in (("value", value), ("value_cost", value_cost), ("q", q), ("r", r_)):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == (np.float64 if name == "value" else np.float32), name
        assert np.array_equal(got, want.astype(got.dtype)), name


def test_dump_outputs_is_refused_off_the_timed_gpu_path():
    r = _run(["--impl", "reference", "--steps", "1", "--dump-outputs", "out"])
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_reference_arm_sets_its_threads_explicitly_and_shares_the_gpu_arms_config():
    """torchrun exports OMP_NUM_THREADS=1: the CPU arm must not inherit it silently (VERDICT r1: it printed
    "128 threads" while running one), and its `config` is the dict the GPU arm prints at the same N."""
    import bench
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--vars-per-gpu", "1000", "--gpus", "2"],
             env={"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0", "OMP_NUM_THREADS": "1",
                  "PYDCOP_B200_CPU_THREADS": "3"})
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["cpu_baseline"]["cores"] == 3 and "OpenMP 3 threads" in d["cpu_baseline"]["sample"]
    assert "median of" in d["cpu_baseline"]["sample"]
    os.environ.pop("PYDCOP_B200_PARTITION", None)
    assert d["config"] == bench.workload_config(2000, 2)
    assert d["n_gpus"] == 2 and d["config"]["n_vars"] == 2000
