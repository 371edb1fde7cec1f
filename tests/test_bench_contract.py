"""bench.py contract checks: the `--impl reference` arm (the CPU CG+AMG port timed on the host cores)
prints one JSON line with the keys the driver reads, and ranks other than 0 stay silent; `--steps` sets
the timed steps and `--dump-outputs` writes the same results on every run (gpu-marked: those of the
CUDA path, checked against the direct oracle)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--impl", "reference", "--rows", "90", "--cols", "90", "--pairs", "4", "--steps", "1", "--warmup", "0",
        "--cpu-sample", "2", "--ref-budget-s", "60"]


def _run(extra_env=None, args=ARGS):
    env = dict(os.environ)
    env.pop("RANK", None)
    env.pop("WORLD_SIZE", None)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    p = _run()
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    j = json.loads(lines[0])
    assert j["impl"] == "reference"
    assert j["metric"] == "pair_solves_per_sec" and j["unit"] == "pair-solves/s"
    assert j["higher_is_better"] is True and j["n_gpus"] == 1 and j["vs_baseline"] is None
    assert j["dtype"] == "f64" and j["data"] == "synthetic"
    for k in ("value", "steps", "warmup", "ms_per_step", "scaling"):
        assert k in j, k
    assert j["value"] > 0 and j["ms_per_step"] > 0
    assert "workload" in j["config"] and "90x90" in j["config"]["workload"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["sample"] and cb["value"] == j["value"]
    e = j["e2e"]
    assert e["value"] == j["value"] and e["unit"] == j["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ""


def _dumped(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_reference_arm_times_the_requested_steps_and_dumps_the_same_outputs(tmp_path):
    dumps = []
    for d in ("a", "b"):
        p = _run(args=ARGS + ["--steps", "3", "--dump-outputs", str(tmp_path / d)])
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout)["steps"] == 3
        dumps.append(_dumped(tmp_path / d))
    a, b = dumps
    assert list(a) == ["resistances"] and a["resistances"].shape == (2,)          # --cpu-sample 2
    assert a["resistances"].dtype == np.float64 and np.all(a["resistances"] > 0)
    assert np.array_equal(a["resistances"], b["resistances"])


def test_bench_rejects_zero_steps():
    p = _run(args=ARGS + ["--steps", "0"])
    assert p.returncode != 0 and "--steps" in p.stderr


def test_dump_samples_long_outputs_the_same_way_every_time(tmp_path):
    import bench
    n = bench.DUMP_SAMPLE + 1000
    x = np.arange(n, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "a"), {"x": x, "short": x[:10]})
    bench.dump_outputs(str(tmp_path / "b"), {"x": x})
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert a["x"].shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(a["x"]) > 0) and a["x"][-1] < n
    assert np.array_equal(a["x"], b["x"]) and np.array_equal(a["short"], x[:10])


@pytest.mark.gpu
def test_cuda_arm_dump_matches_the_direct_oracle(tmp_path):
    import bench
    from oracle import circuitscape_oracle as co
    p = _run(args=["--rows", "120", "--cols", "100", "--pairs", "6", "--steps", "2", "--warmup", "1",
                   "--skip-spmv1e7", "--skip-cpu", "--skip-direct", "--skip-e2e", "--dump-outputs", str(tmp_path)])
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == 2
    d = _dumped(tmp_path)
    L, src, dst = bench.workload(argparse.Namespace(rows=120, cols=100, precision="double"), 6)
    V = co.solve_pairs_direct(L, src, dst)
    R = V[dst, np.arange(len(src))]
    cur = np.column_stack([co.get_node_currents(L, V[:, c]) for c in range(len(src))])
    assert np.abs(d["resistances"] - R).max() <= 1e-6 * R.max()
    assert np.abs(d["cum_current"] - cur.sum(axis=1)).max() <= 1e-4 * cur.sum(axis=1).max()
    assert np.abs(d["max_current"] - cur.max(axis=1)).max() <= 1e-4 * cur.max()
