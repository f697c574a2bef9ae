"""bench.py --dump-outputs on the GPU: the files hold what the timed path computed in its last step, for inputs that
--steps alone determines, within the size bound."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_last_timed_step(model, built_library, tmp_path):
    import bench
    from hippopt_b200.evaluator import ALL, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], cwd=ROOT, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert line["steps"] == 2
    names = {"f", "grad_f", "g", "jac", "hess"}
    assert {p.name for p in tmp_path.iterdir()} == {f"{n}.npy" for n in names}
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    got = {n: np.load(tmp_path / f"{n}.npy") for n in names}

    # the bench alternates two input sets; the last of two steps evaluates the second one (seed 1002 on rank 0)
    ev = KinoEvaluator(model, KinoSettings(horizon=bench.HORIZON))
    B = bench.INSTANCES_PER_GPU
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=1002)
    out = ev.eval(ALL, *(torch.tensor(a, device="cuda:0") for a in (x, p, lam, sigma)))
    rows = bench.dump_rows(B)
    for n in names:
        want = out[n].cpu().numpy()
        want = want if n == "f" else want[rows]
        assert got[n].dtype == np.float64 and got[n].shape == want.shape, n
        assert np.array_equal(got[n], want), n
