"""bench.py's reference arm runs on the host alone (it times the CPU oracle), so its contract can be
checked here: one JSON line with the keys the driver reads, rank > 0 silent."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                           "--warmup", "1", "--models", "2000"], capture_output=True, text=True, env=env,
                          timeout=240, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "model_source_travel_time_evals_per_s"
    assert d["unit"] == "evals/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_is_silent_on_other_ranks():
    r = _run({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_bench_refuses_zero_steps_and_a_dump_of_the_reference_arm(tmp_path):
    for extra in (["--steps", "0"], ["--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"] + extra,
                           capture_output=True, text=True, timeout=60, cwd=ROOT)
        assert r.returncode == 2 and "error:" in r.stderr
    assert not os.listdir(tmp_path)


def test_dump_outputs_is_exact_under_the_budget_and_a_fixed_sample_over_it(tmp_path):
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    flag = sys.dont_write_bytecode
    try:
        spec.loader.exec_module(bench)
    finally:
        sys.dont_write_bytecode = flag
    a = np.random.default_rng(1).normal(size=1000)
    bench.dump_outputs(str(tmp_path / "all"), {"logL": a}, budget=8000)
    got = np.load(tmp_path / "all" / "logL.npy")
    assert got.dtype == np.float64 and np.array_equal(got, a)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"logL": a}, budget=800)
    s1, s2 = np.load(tmp_path / "s1" / "logL.npy"), np.load(tmp_path / "s2" / "logL.npy")
    assert s1.nbytes <= 800 and s1.size == 100 and np.array_equal(s1, s2)
    assert np.array_equal(a[np.isin(a, s1)], s1)          # elements of the output, in index order
