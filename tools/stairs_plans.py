"""Stairs plans (BASELINE config 5, walking on stairs) end to end on one GPU: B plans with step heights in
U(0.05, 0.15) set up on the device (initial_guess.stairs_step_guess: keyframe poses on the smooth steps, interpolated
guess) and solved by the batched interior-point driver with the stage-wise KKT sweep and the options of the
reference's stairs main (hessian_approximation = limited-memory, max_iter 10 000) and the tolerances config 4 is
solved with.  Prints one JSON line: converged / B, plans/s, median iterations, worst constraint violation of the
converged plans, set-up time, and the card name and power limit read in the same run.

    python tools/stairs_plans.py [--B 512] [--seed 0] [--max-iter 10000]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

OPTIONS = {"tol": 1e-3, "dual_inf_tol": 1000.0, "compl_inf_tol": 1e-2, "constr_viol_tol": 1e-4, "acceptable_tol": 10,
           "acceptable_iter": 2, "acceptable_compl_inf_tol": 1000.0, "acceptable_obj_change_tol": 1e0,
           "nlp_scaling_method": "gradient-based", "max_iter": 10000, "hessian_approximation": "limited-memory"}


def power_limit_w():
    """The enforced power limit of GPU 0 in W (a read-only query), or None where it cannot be read."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def solve_stairs(model, B, seed=0, max_iter=10000, horizon=50):
    """-> (guess, result, kinodynamic evaluator, step heights, set-up seconds, solve seconds)."""
    from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
    from hippopt_b200.initial_guess import stairs_step_guess
    from hippopt_b200.ipsolver import BatchedInteriorPoint
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.pose_layout import PoseSettings

    smooth = dict(terrain="smooth_steps", n_terrain_params=10)
    pev = PoseEvaluator(model, PoseSettings(**smooth))
    ev = KinoEvaluator(model, KinoSettings(horizon=horizon, final_state_constraint=True, **smooth))
    h = np.random.default_rng(seed).uniform(0.05, 0.15, B)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gs = stairs_step_guess(model, pev, ev, h, force_z=100.0, mass_normalised=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    lb, ub = ev.layout.bounds(gs.parameters)
    ip = BatchedInteriorPoint(ev, kkt="stage", delta_c=1e-9, mu_init=1e-1, ipopt_options=dict(OPTIONS, max_iter=max_iter))
    res = ip.solve(gs.x0, torch.tensor(gs.parameters, device=gs.x0.device), lb, ub)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return gs, res, ev, h, t1 - t0, t2 - t1


def constraint_violation(ev, res, parameters):
    from hippopt_b200.evaluator import G

    lb, ub = ev.layout.bounds(parameters)
    g = ev.eval(G, res.values, torch.tensor(parameters, device=res.values.device))["g"].cpu().numpy()
    return (np.maximum(lb - g, 0.0) + np.maximum(g - ub, 0.0)).max(axis=1)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--B", type=int, default=512)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max-iter", type=int, default=OPTIONS["max_iter"])
    a = ap.parse_args()
    from hippopt_b200.robot_model import synthetic_ergocub

    model = synthetic_ergocub()
    from hippopt_b200.ipsolver import OptiFailure

    try:  # warm-up: library load, allocator, first launches
        solve_stairs(model, 4, seed=a.seed + 1, max_iter=3)
    except OptiFailure:
        pass
    gs, res, ev, h, t_setup, t_solve = solve_stairs(model, a.B, seed=a.seed, max_iter=a.max_iter)
    ok = res.success.cpu().numpy()
    viol = constraint_violation(ev, res, gs.parameters)
    it = res.iterations.cpu().numpy()
    print(json.dumps({
        "workload": "config 5: walking on stairs, horizon 50, step heights U(0.05, 0.15)",
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
