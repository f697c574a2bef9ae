"""The general smooth-step terrain (``terrain="tilted_steps"``, the ramp's terrain) on the CPU: the oracle's tilted step
against SURVEY.md A.10's closed form, the K-step oracle against the stairs oracle, the layouts' patterns and bounds
against the oracle and the smooth_steps layouts, the stage-wise KKT solve on a tilted layout, the terrain parameter
builders and the rejection of inconsistent settings."""
import math

import numpy as np
import pytest
import torch

import tilted_oracle as to
from hippopt_b200.kino_layout import KinoLayout, KinoSettings, kernel_terrain
from hippopt_b200.kkt import StageKKT
from hippopt_b200.pose_layout import PoseLayout, PoseSettings
from hippopt_b200.workloads import kino_parameters
from oracle import expressions as ex
from oracle import sx


def _closed_form(pt, q):
    """A.10: h = p_z - exp(-g^20) pi(x_t, y_t) - o_z for one step q = (l, w, height, ox, oy, oz, yaw, nx, ny, nz)"""
    l, w, H, ox, oy, oz, yaw, nx, ny, nz = q
    c, s = math.cos(yaw), math.sin(yaw)
    dx, dy = pt[0] - ox, pt[1] - oy
    xt, yt = c * dx + s * dy, -s * dx + c * dy
    g = (2 * xt / l) ** 10 + (2 * yt / w) ** 10
    return pt[2] - math.exp(-g ** 20) * (H - nx / nz * xt - ny / nz * yt) - oz


STEPS = np.array([
    [0.9, 0.6, 0.1, 0.3, -0.1, 0.02, 0.4, -0.2, 0.1, 0.97],
    [1.2, 0.8, 0.05, -0.1, 0.2, -0.03, -1.1, 0.15, -0.25, 0.95],
    [0.5, 0.5, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0],
])
POINTS = np.array([[0.3, -0.1, 0.2], [0.6, 0.05, -0.1], [0.1, 0.3, 0.0], [0.7, -0.2, 0.05], [-0.4, 0.4, 0.3],
                   [0.25, 0.25, 0.1], [3.0, -2.0, 0.5]])


def _numeric(terrain, pt, tp):
    """terrain.height at a numeric point and parameters, through the oracle's tape"""
    p, q = sx.syms("p", 3), sx.syms("tp", len(tp))
    tape = sx.Tape([terrain.with_params(q).height(p)], list(p) + list(q))
    return float(tape.eval(np.concatenate([pt, tp])[None, :])[0, 0])


@pytest.mark.parametrize("s", range(len(STEPS)))
def test_oracle_tilted_step_matches_the_closed_form(s):
    for pt in POINTS:
        got = _numeric(to.TiltedSteps(1), pt, STEPS[s])
        ref = _closed_form(pt, STEPS[s])
        assert abs(got - ref) <= 1e-14 * max(1.0, abs(ref)), (pt, got, ref)


def test_oracle_tilted_steps_sum_the_steps():
    tp = STEPS.reshape(-1)
    for pt in POINTS:
        got = _numeric(to.TiltedSteps(3), pt, tp)
        ref = sum(_closed_form(pt, q) for q in STEPS) - 2 * pt[2]
        assert abs(got - ref) <= 1e-14 * max(1.0, abs(ref))


def test_tilted_steps_with_flat_axis_aligned_tops_equal_the_stairs():
    stairs = ex.TwoSmoothSteps.stairs_parameters(height=0.12)
    tilted = to.stairs_as_tilted(stairs)[0]
    for pt in np.concatenate([POINTS, [[0.225, 0.0, 0.1], [0.6975, 0.3, 0.2], [0.45, -0.4, 0.0]]]):
        a = _numeric(ex.TwoSmoothSteps(), pt, stairs)
        b = _numeric(to.TiltedSteps(2), pt, tilted)
        assert a == b or abs(a - b) <= 1e-15 * max(1.0, abs(a))


def test_kernel_terrain_names_and_counts():
    assert kernel_terrain("planar", 0) == 0
    assert kernel_terrain("smooth_steps", 10) == 1
    assert kernel_terrain("tilted_steps", 10) == kernel_terrain("tilted_steps", 30) == 2
    for name, n in (("ramp", 10), ("stairs", 10), ("tilted_steps", 0), ("tilted_steps", 15), ("tilted_steps", -10),
                    ("smooth_steps", 20), ("planar", 10)):
        with pytest.raises(ValueError):
            kernel_terrain(name, n)


@pytest.mark.parametrize("settings", [dict(terrain="ramp", n_terrain_params=10), dict(terrain="Planar"),
                                      dict(terrain="tilted_steps"), dict(terrain="tilted_steps", n_terrain_params=25),
                                      dict(terrain="smooth_steps", n_terrain_params=20)])
def test_layouts_reject_inconsistent_terrain_settings(model, settings):
    with pytest.raises(ValueError):
        KinoLayout(model, KinoSettings(horizon=3, **settings))
    with pytest.raises(ValueError):
        PoseLayout(model, PoseSettings(**settings))


@pytest.mark.parametrize("N,fin,per,K", [(3, False, False, 1), (3, True, False, 2), (4, False, True, 1),
                                         (4, True, True, 3)])
def test_kino_tilted_layout_matches_the_oracle_and_the_stairs_layout(model, N, fin, per, K):
    st = dict(horizon=N, final_state_constraint=fin, periodicity_constraint=per)
    lay = KinoLayout(model, KinoSettings(terrain="tilted_steps", n_terrain_params=10 * K, **st))
    stairs = KinoLayout(model, KinoSettings(terrain="smooth_steps", n_terrain_params=10, **st))
    assert lay.kernel_terrain == 2 and lay.n_p == stairs.n_p + 10 * (K - 1) and lay.po.terrain == stairs.po.terrain
    for a in ("jac_colind", "jac_row", "hess_colind", "hess_row"):
        assert np.array_equal(getattr(lay, a), getattr(stairs, a)), a
    assert (lay.m, lay.nnz_j, lay.nnz_h, lay.n_jc, lay.n_hc) == (stairs.m, stairs.nnz_j, stairs.nnz_h, stairs.n_jc,
                                                                 stairs.n_hc)
    nlp, _ = to.kino_build(model, K, **st)
    assert (lay.n_x, lay.n_p, lay.m) == (nlp.n_x, nlp.n_p, nlp.m)
    jc, jr = nlp.jac_structure()[:2]
    hc, hr = nlp.hess_structure()[:2]
    assert np.array_equal(lay.jac_colind, jc) and np.array_equal(lay.jac_row, jr)
    assert np.array_equal(lay.hess_colind, hc) and np.array_equal(lay.hess_row, hr)
    p = kino_parameters(lay, model, 2, np.random.default_rng(N + K))
    lb, ub = lay.bounds(p)
    olb, oub = nlp.eval_bounds(p)
    assert np.array_equal(lb, olb) and np.array_equal(ub, oub)


@pytest.mark.parametrize("K", [1, 2])
def test_pose_tilted_layout_matches_the_oracle_and_the_stairs_layout(model, K):
    lay = PoseLayout(model, PoseSettings(terrain="tilted_steps", n_terrain_params=10 * K))
    stairs = PoseLayout(model, PoseSettings(terrain="smooth_steps", n_terrain_params=10))
    nlp, olay = to.pose_build(model, K)
    assert (lay.n_x, lay.n_p, lay.m) == (nlp.n_x, nlp.n_p, nlp.m) == (81, 202 + 10 * K, 89)
    assert lay.po.terrain == olay.terrain - lay.n_x == 202 and lay.kernel_terrain == 2
    jc, jr = nlp.jac_structure()[:2]
    hc, hr = nlp.hess_structure()[:2]
    assert np.array_equal(lay.jac_colind, jc) and np.array_equal(lay.jac_row, jr)
    assert np.array_equal(lay.hess_colind, hc) and np.array_equal(lay.hess_row, hr)
    for a in ("jac_colind", "jac_row", "hess_colind", "hess_row"):
        assert np.array_equal(getattr(lay, a), getattr(stairs, a)), a
    p = np.random.default_rng(K).uniform(1.0, 2.0, (2, lay.n_p))
    lb, ub = lay.bounds(p)
    olb, oub = nlp.eval_bounds(p)
    assert np.array_equal(lb, olb) and np.array_equal(ub, oub)


def test_stage_solve_matches_dense_on_a_tilted_layout(model):
    N, K = 4, 2
    lay = KinoLayout(model, KinoSettings(horizon=N, final_state_constraint=True, terrain="tilted_steps",
                                         n_terrain_params=10 * K))
    p = kino_parameters(lay, model, 1, np.random.default_rng(0))
    lb, ub = lay.bounds(p)
    eq, ine = np.nonzero(lb[0] == ub[0])[0], np.nonzero(lb[0] != ub[0])[0]
    kkt = StageKKT(lay.n_x, lay.m, N, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine,
                   linalg="torch")
    B = 3
    g = torch.Generator().manual_seed(77)
    hv = torch.randn((B, lay.nnz_h), generator=g, dtype=torch.float64)
    jv = torch.randn((B, lay.nnz_j), generator=g, dtype=torch.float64)
    sig = torch.rand((B, len(ine)), generator=g, dtype=torch.float64) * 3.0
    delta = torch.tensor([40.0, 55.0, 70.0], dtype=torch.float64)
    rx = torch.randn((B, lay.n_x), generator=g, dtype=torch.float64)
    rE = torch.randn((B, len(eq)), generator=g, dtype=torch.float64)
    rE[:, kkt.dead_eq] = 0.0
    dx, dl = kkt.solve(hv, jv, sig, delta, 1e-6, rx, rE)
    Km = kkt.dense_matrix(hv, jv, sig, delta, 1e-6, eq, ine, lay.jac_colind, lay.jac_row, lay.hess_colind,
                          lay.hess_row)
    ref = torch.linalg.solve(Km, torch.cat([rx, rE], dim=1))
    u = torch.cat([dx, dl], dim=1)
    scale = ref.abs().amax(dim=1, keepdim=True)
    assert ((u - ref).abs() / scale).max().item() < 1e-9


def test_tilted_steps_terrain_builds_and_validates():
    from hippopt_b200.initial_guess import ramp_terrain, tilted_steps_terrain

    tp = tilted_steps_terrain([1.0, 2.0], [0.5, 0.6], [0.1, 0.2], [[0.1, 0.2, 0.3], [0.4, 0.5, 0.6]], [0.3, -0.3],
                              [[0.0, 0.0, 1.0], [0.1, 0.2, 0.9]])
    assert tp.shape == (1, 20)
    assert np.array_equal(tp[0, :10], [1.0, 0.5, 0.1, 0.1, 0.2, 0.3, 0.3, 0.0, 0.0, 1.0])
    assert np.array_equal(tp[0, 10:], [2.0, 0.6, 0.2, 0.4, 0.5, 0.6, -0.3, 0.1, 0.2, 0.9])
    one = tilted_steps_terrain(0.9, 0.8, 0.1, [0.3, 0.0, 0.0])
    assert np.array_equal(one, [[0.9, 0.8, 0.1, 0.3, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0]])
    for bad in (dict(length=0.0), dict(width=-1.0), dict(normal=[0.1, 0.0, 0.0]), dict(normal=[0.0, 0.0, -1.0]),
                dict(height=float("nan"))):
        args = dict(length=1.0, width=1.0, height=0.1, origin=[0.0, 0.0, 0.0], normal=[0.0, 0.0, 1.0])
        args.update(bad)
        with pytest.raises(ValueError):
            tilted_steps_terrain(**args)
    # the ramp: low edge at height 0, the top rises with the slope along +x
    s = np.array([0.1, 0.2])
    tp = ramp_terrain(s)
    assert tp.shape == (2, 10)
    for b in range(2):
        for x in (0.5, 1.0, 1.8):
            h = _closed_form([x, 0.0, 0.0], tp[b])
            assert abs(-h - s[b] * (x - 0.225)) < 1e-12
