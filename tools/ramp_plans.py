"""Ramp plans end to end on one GPU: B plans of a step onto a ramp (``terrain="tilted_steps"``, one tilted step) with
slopes in U(0.05, 0.2) set up on the device (initial_guess.ramp_step_guess: keyframe poses on the ramp, interpolated
guess) and solved by the batched interior-point driver with the options of tools/stairs_plans.py.  Prints one JSON
line: converged / B, plans/s, median iterations, worst constraint violation of the converged plans, set-up time, and
the card name and power limit read in the same run.

    python tools/ramp_plans.py [--B 512] [--seed 0] [--max-iter 10000]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from stairs_plans import OPTIONS, constraint_violation, power_limit_w  # noqa: E402


def solve_ramp(model, B, seed=0, max_iter=10000, horizon=50):
    """-> (guess, result, kinodynamic evaluator, slopes, set-up seconds, solve seconds)."""
    from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
    from hippopt_b200.initial_guess import ramp_step_guess
    from hippopt_b200.ipsolver import BatchedInteriorPoint
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.pose_layout import PoseSettings

    tilted = dict(terrain="tilted_steps", n_terrain_params=10)
    pev = PoseEvaluator(model, PoseSettings(**tilted))
    ev = KinoEvaluator(model, KinoSettings(horizon=horizon, final_state_constraint=True, **tilted))
    s = np.random.default_rng(seed).uniform(0.05, 0.2, B)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gs = ramp_step_guess(model, pev, ev, s, force_z=100.0, mass_normalised=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    lb, ub = ev.layout.bounds(gs.parameters)
    ip = BatchedInteriorPoint(ev, kkt="stage", delta_c=1e-9, mu_init=1e-1, ipopt_options=dict(OPTIONS, max_iter=max_iter))
    res = ip.solve(gs.x0, torch.tensor(gs.parameters, device=gs.x0.device), lb, ub)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return gs, res, ev, s, t1 - t0, t2 - t1


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-iter", type=int, default=OPTIONS["max_iter"])
    a = ap.parse_args()
    from hippopt_b200.ipsolver import OptiFailure
    from hippopt_b200.robot_model import synthetic_ergocub

    model = synthetic_ergocub()
    try:  # warm-up: library load, allocator, first launches
        solve_ramp(model, 4, seed=a.seed + 1, max_iter=3)
    except OptiFailure:
        pass
    gs, res, ev, s, t_setup, t_solve = solve_ramp(model, a.B, seed=a.seed, max_iter=a.max_iter)
    ok = res.success.cpu().numpy()
    viol = constraint_violation(ev, res, gs.parameters)
    it = res.iterations.cpu().numpy()
    print(json.dumps({
        "workload": "ramp: one step onto a ramp, horizon 50, slopes U(0.05, 0.2)",
        "B": a.B, "converged": int(ok.sum()), "converged_fraction": float(ok.mean()),
        "keyframes_ok": int(gs.ok.sum().item()),
        "plans_per_s": a.B / t_solve, "solve_s": t_solve, "setup_s": t_setup,
        "median_iterations": float(np.median(it[ok])) if ok.any() else None,
        "max_iterations": int(it.max()),
        "worst_constr_viol_converged": float(viol[ok].max()) if ok.any() else None,
        "device": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w(),
    }))


if __name__ == "__main__":
    main()
