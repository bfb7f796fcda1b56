"""bench.py's command line: --steps sets the number of timed steps, and --dump-outputs writes what the timed plan
returned in its last step, from seeded inputs that are the same on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import term_b200 as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, rows=None):
    env = dict(os.environ)
    if rows is not None:
        env["TG_BENCH_ROWS"] = str(rows)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--steps", "-3"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_rejected_arguments(args):
    p = _bench(*args)
    assert p.returncode == 2 and "error:" in p.stderr, p.stderr


def test_dump_outputs_writes_float64_arrays_in_suite_order(tmp_path):
    S = T.ConstraintStatus
    results = [T.ConstraintResult(S.Success, 1e8, name="size"), T.ConstraintResult(S.Failure, -3.5, name="min"),
               T.ConstraintResult(S.Skipped, None, name="mean")]
    out = tmp_path / "a" / "b"
    bench.dump_outputs(results, str(out))
    assert sorted(os.listdir(out)) == ["metric.npy", "status.npy"]
    metric, status = np.load(out / "metric.npy"), np.load(out / "status.npy")
    assert metric.dtype == np.float64 and status.dtype == np.float64
    assert metric[0] == 1e8 and metric[1] == -3.5 and np.isnan(metric[2])
    assert status.tolist() == [0.0, 1.0, 2.0]


@pytest.mark.gpu
def test_steps_and_dumped_outputs_on_the_gpu(built_lib, tmp_path):
    n = 100_003
    lines = {}
    for steps in (2, 5):
        p = _bench("--steps", str(steps), "--warmup", "1", "--no-cpu", "--no-e2e", "--suites", "none",
                   "--dump-outputs", str(tmp_path / f"s{steps}"), rows=n)
        assert p.returncode == 0, p.stderr[-2000:]
        lines[steps] = json.loads(p.stdout.strip().splitlines()[-1])
        assert lines[steps]["steps"] == steps
    # every timed step launches the same kernels: the count over the timed region scales with --steps
    assert lines[2]["gpu_launches"] > 0 and lines[5]["gpu_launches"] * 2 == lines[2]["gpu_launches"] * 5
    got = {k: np.load(tmp_path / "s5" / f"{k}.npy") for k in ("metric", "status")}
    for k, v in got.items():  # the same seeded inputs on every run
        assert np.array_equal(v, np.load(tmp_path / "s2" / f"{k}.npy")), k
    assert got["status"].tolist() == [float(T.ConstraintStatus[r["status"]].value) for r in lines[5]["results"]]
    assert got["metric"].tolist() == [r["metric"] for r in lines[5]["results"]]
    # the C restatement of the suite on the same host table
    from oracle import cpu_scan as S
    cpu = S.numeric_suite({k: v for k, v in bench.make_host_table(n).items() if k != "_keep"}, n)
    size, mn, mean, corr, sat = got["metric"]
    assert size == cpu["size"] and mn == cpu["min_f0"] and sat == cpu["satisfies"]
    assert abs(mean - cpu["mean_f1"]) <= 1e-9 * abs(cpu["mean_f1"]) and abs(corr - cpu["corr_f0_f1"]) <= 1e-6
