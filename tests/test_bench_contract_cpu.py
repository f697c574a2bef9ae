"""bench.py's contract that can be checked without a GPU: the reference arm (the CPU oracle on the host cores,
`--impl reference`) prints one JSON line with the agreed keys, only rank 0 works under torchrun, the product arm
refuses to run without a CUDA device instead of falling back to anything, and arguments it cannot honour are refused."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, capture_output=True,
                          text=True, timeout=600)


def test_reference_arm_line():
    r = run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1", "--cpu-sample", "4"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "knot_evals_per_s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["dtype"] == "f64" and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("humanoid_kinodynamic single step flat ground (BASELINE config 3)")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "4 of the 1024 instances" in cb["sample"]
    assert d["steps"] == 1 and d["warmup"] == 1


def test_reference_arm_honours_steps_and_warmup():
    """--steps / --warmup are taken as given (round-1 verdict: they were clamped to 3 / 1); the per-step sample is
    what is bounded."""
    r = run(["--impl", "reference", "--gpus", "1", "--steps", "4", "--warmup", "2", "--cpu-sample", "4"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][0])
    assert d["steps"] == 4 and d["warmup"] == 2 and "(4 timed steps, 2 warm-up)" in d["cpu_baseline"]["sample"]


@pytest.mark.parametrize("args,message", [(["--steps", "0"], "--steps must be at least 1"),
                                          (["--impl", "reference", "--dump-outputs", "out"], "the reference arm keeps none")])
def test_arguments_that_are_refused(args, message):
    r = run(args)
    assert r.returncode == 2 and message in r.stderr and r.stdout == ""


def test_dump_rows_are_a_fixed_sample():
    import bench

    rows = bench.dump_rows(1024)
    assert len(rows) == bench.DUMP_INSTANCES and np.all(np.diff(rows) > 0) and rows[-1] < 1024
    assert np.array_equal(rows, bench.dump_rows(1024)) and np.array_equal(bench.dump_rows(5), np.arange(5))


def test_reference_arm_other_ranks_exit_quietly():
    r = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--cpu-sample", "4"],
            env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour WITHOUT a CUDA device")
def test_product_arm_has_no_cpu_fallback():
    r = run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "needs a CUDA device" in (r.stderr + r.stdout)
