"""The pose finder on the stairs (two smooth steps, BASELINE config 5) on the GPU: `pose_contact_kernel<1>` against
the oracle, determinism, the stairs plan set-up (`initial_guess.stairs_step_guess`) and stairs-plan solves."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-10
SMOOTH = dict(terrain="smooth_steps", n_terrain_params=10)
FIRST_EDGE, SECOND_EDGE = 0.225, 0.6975  # x of the first and second step edges of the stairs
# stairs-plan solves: 4 of these 16 plans converge within 3000 iterations (measured on an NVIDIA B200; the other 12
# stop at the iteration limit or shortly before it; DESIGN.md section 9.1, config 5)
STAIRS_MAX_ITER = 3000
STAIRS_MIN_CONVERGED = 4


def dev():
    return torch.device("cuda:0")


def run(ev, x, p, lam, sigma):
    from hippopt_b200.evaluator import ALL

    t = [torch.tensor(np.ascontiguousarray(a), device=dev()) for a in (x, p, lam, sigma)]
    out = ev.eval(ALL, *t)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def smooth_pose(model):
    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.pose_layout import PoseSettings

    return PoseEvaluator(model, PoseSettings(**SMOOTH))


def stairs_inputs(ev, model, B, seed):
    """Pose-finder inputs on the stairs with the points of each instance placed in one of the regions the terrain has:
    the ground, the first and the second tread, the transition bands of both edges, and all of them mixed."""
    from hippopt_b200.initial_guess import stairs_terrain
    from hippopt_b200.workloads import pose_batch

    rng = np.random.default_rng(seed)
    x, p, lam, sigma = pose_batch(ev.layout, model, B, seed=seed, noise=0.05)
    h = rng.uniform(0.05, 0.15, B)
    po = ev.layout.po
    p[:, po.terrain:po.terrain + 10] = stairs_terrain(h)
    regions = [(0.0, 0.1, 0.0), (0.45, 0.1, 1.0), (0.9, 0.1, 2.0), (FIRST_EDGE, 0.01, 0.5), (SECOND_EDGE, 0.01, 1.5)]
    for b in range(B):
        for i in range(8):
            cx, spread, level = regions[b % 5] if b % 6 != 5 else regions[rng.integers(5)]
            x[b, 6 * i] = cx + rng.uniform(-spread, spread)
            x[b, 6 * i + 1] = (0.1 if i < 4 else -0.1) + rng.uniform(-0.05, 0.05)
            x[b, 6 * i + 2] = level * h[b] + rng.normal(scale=0.01)
    sigma = np.linspace(0.3, 2.0, B)
    return x, p, lam, sigma


def check_against_oracle(ev, model, x, p, lam, sigma, out):
    import smooth_pose_oracle
    from oracle import parity

    nlp, _ = smooth_pose_oracle.build(model)
    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(out[k]).all() and np.isfinite(r).all(), k
    worst = parity.check_all(out, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2], x, rtol=RTOL)
    print("worst relative errors:", {k: f"{v:.2e}" for k, v in worst.items()})


def test_smooth_pose_finder_against_oracle(model, built_library):
    """All five outputs, per-instance parameters, a batch that is not a multiple of the kernel's four warps per CTA."""
    ev = smooth_pose(model)
    assert (ev.n_x, ev.n_p, ev.m) == (81, 212, 89)
    x, p, lam, sigma = stairs_inputs(ev, model, 11, seed=21)
    check_against_oracle(ev, model, x, p, lam, sigma, run(ev, x, p, lam, sigma))


def test_smooth_pose_finder_shared_parameters(model, built_library):
    """One parameter vector for the whole batch (p_stride = 0): the terrain parameters are read from it too."""
    ev = smooth_pose(model)
    x, p, lam, sigma = stairs_inputs(ev, model, 6, seed=22)
    out = run(ev, x, p[0], lam, sigma)
    check_against_oracle(ev, model, x, p[:1], lam, sigma, out)
    per_instance = run(ev, x, np.repeat(p[:1], 6, axis=0), lam, sigma)
    for k in out:
        assert np.array_equal(out[k], per_instance[k]), k


def test_smooth_pose_finder_is_deterministic(model, built_library):
    """Bit-identical outputs across two runs and across batch orders (fixed accumulation order of the Hessian)."""
    ev = smooth_pose(model)
    x, p, lam, sigma = stairs_inputs(ev, model, 1030, seed=23)
    out = run(ev, x, p, lam, sigma)
    again = run(ev, x, p, lam, sigma)
    perm = np.random.default_rng(4).permutation(1030)
    permuted = run(ev, x[perm], p[perm], lam[perm], sigma[perm])
    for k in out:
        assert np.isfinite(out[k]).all(), k
        assert np.array_equal(again[k], out[k]), k
        assert np.array_equal(permuted[k], out[k][perm]), k


def test_stairs_step_guess(model, built_library):
    """Keyframe poses on the stairs for 32 step heights in U(0.05, 0.15): every pose solve converges, every contact
    corner is on or above the terrain, the corners on a tread sit at its height and the guess is finite."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.initial_guess import stairs_step_guess
    from hippopt_b200.kino_layout import KinoSettings
    from oracle import expressions as ex

    B = 32
    h = np.random.default_rng(7).uniform(0.05, 0.15, B)
    ev = KinoEvaluator(model, KinoSettings(horizon=50, final_state_constraint=True, **SMOOTH))
    gs = stairs_step_guess(model, smooth_pose(model), ev, h, mass_normalised=True)
    assert bool(gs.ok.all()), f"{int(gs.ok.sum())} of {B} instances with all three keyframe poses converged"
    assert torch.isfinite(gs.x0).all() and np.isfinite(gs.parameters).all()
    key = gs.keyframes.cpu().numpy()  # (3, B, 105): per point (p, f, descriptor), ...
    assert np.array_equal(gs.parameters[:, ev.layout.po.terrain:ev.layout.po.terrain + 10],
                          np.stack([ex.TwoSmoothSteps.stairs_parameters(height=v) for v in h]))
    for kf in range(3):
        for i in range(8):
            pt = key[kf, :, 9 * i:9 * i + 3]
            assert (terrain_height(gs.parameters[:, ev.layout.po.terrain:ev.layout.po.terrain + 10], pt) >= -1e-6).all()
            on_tread = (i < 4 and kf >= 1) or (i >= 4 and kf == 2)
            assert np.abs(pt[:, 2] - (h if on_tread else 0.0)).max() < 1e-3, (kf, i)


def terrain_height(tp, pt):
    """h(p) = z - sum_s height_s exp(-g_s^20), g_s = (2 (x - ox_s) / l_s)^10 + (2 (y - oy_s) / w_s)^10 (numpy, (B,))."""
    out = pt[:, 2].copy()
    for s in range(2):
        l, w, hs, ox, oy = (tp[:, 5 * s + j] for j in range(5))
        g = (2.0 * (pt[:, 0] - ox) / l) ** 10 + (2.0 * (pt[:, 1] - oy) / w) ** 10
        out -= hs * np.exp(-np.minimum(g, 10.0) ** 20)
    return out


def load_stairs_tool():
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "stairs_plans.py")
    spec = importlib.util.spec_from_file_location("stairs_plans", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_stairs_plans_solve(model, built_library):
    """Config 5 end to end on a small batch: set-up on the device and limited-memory solves with the stairs main's
    options (tools/stairs_plans.py).  Converged plans satisfy the constraints to constr_viol_tol and end with both feet
    on the first tread."""
    tool = load_stairs_tool()
    B = 16
    gs, res, ev, h, _, _ = tool.solve_stairs(model, B, seed=3, max_iter=STAIRS_MAX_ITER)
    ok = res.success.cpu().numpy()
    print("stairs plans converged:", int(ok.sum()), "of", B, "iterations", res.iterations.cpu().numpy().tolist())
    assert ok.sum() >= STAIRS_MIN_CONVERGED, f"{int(ok.sum())} of {B} stairs plans converged"
    assert tool.constraint_violation(ev, res, gs.parameters)[ok].max() <= 1e-4
    N = ev.layout.N
    z = res.values.cpu().numpy()[ok][:, :189 * N].reshape(-1, N, 189)
    last = z[:, -1, :120].reshape(-1, 8, 15)[:, :, 6:9]  # the contact points' positions at the last knot
    assert np.abs(last[:, :, 2] - h[ok][:, None]).max() < 1e-3
    assert ((last[:, :, 0] > FIRST_EDGE + 0.02) & (last[:, :, 0] < SECOND_EDGE - 0.02)).all()
