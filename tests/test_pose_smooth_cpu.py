"""The pose finder on the stairs (smooth-step terrain, BASELINE config 5 keyframes), on the CPU: the layout's patterns
against the oracle's structural derivation, the planar layout unchanged, the plugin's template match, and the
stage-wise KKT solve on smooth-terrain kinodynamic layouts (whose height, normal-force and CoM-height rows stay
general rows) against a dense solve."""
import numpy as np
import pytest
import torch

from hippopt_b200.kino_layout import KinoLayout, KinoSettings
from hippopt_b200.kkt import StageKKT
from hippopt_b200.pose_layout import PoseLayout, PoseSettings
from hippopt_b200.workloads import kino_parameters

SMOOTH = PoseSettings(terrain="smooth_steps", n_terrain_params=10)


def test_smooth_pose_layout_patterns_match_the_oracle(model):
    import smooth_pose_oracle

    lay = PoseLayout(model, SMOOTH)
    nlp, olay = smooth_pose_oracle.build(model)
    assert (lay.n_x, lay.n_p, lay.m) == (nlp.n_x, nlp.n_p, nlp.m) == (81, 212, 89)
    assert lay.po.terrain == olay.terrain - lay.n_x == 202
    jc, jr = nlp.jac_structure()[:2]
    hc, hr = nlp.hess_structure()[:2]
    assert np.array_equal(lay.jac_colind, jc) and np.array_equal(lay.jac_row, jr)
    assert np.array_equal(lay.hess_colind, hc) and np.array_equal(lay.hess_row, hr)
    assert (lay.nnz_j, lay.nnz_h, lay.n_jc, lay.n_hc) == (680, 449, 355, 255)
    p = np.random.default_rng(0).uniform(1.0, 2.0, (2, lay.n_p))
    lb, ub = lay.bounds(p)
    olb, oub = nlp.eval_bounds(p)
    assert np.array_equal(lb, olb) and np.array_equal(ub, oub)


def test_planar_pose_layout_is_unchanged(model):
    """The planar layout against the oracle (the parent's derivation) and its known sizes; the terrain settings
    default to the planar terrain."""
    from oracle import pose_finder as pf

    lay = PoseLayout(model)
    assert lay.st.terrain == "planar" and lay.st.n_terrain_params == 0 and not lay.smooth
    assert (lay.n_p, lay.nnz_j, lay.nnz_h, lay.n_jc, lay.n_hc) == (202, 584, 385, 259, 191)
    nlp, _ = pf.build(model)
    assert np.array_equal(lay.jac_colind, nlp.jac_structure()[0]) and np.array_equal(lay.jac_row, nlp.jac_structure()[1])
    assert np.array_equal(lay.hess_colind, nlp.hess_structure()[0])
    assert np.array_equal(lay.hess_row, nlp.hess_structure()[1])


def test_smooth_pose_layout_keeps_the_planar_local_orders(model):
    """Everything but the per-point terrain rows keeps its local order: the smooth layout's scatter maps of the
    kinematics kernel and of the robot rows are those of the planar layout, shifted past the longer point blocks."""
    pl, sl = PoseLayout(model), PoseLayout(model, SMOOTH)
    assert np.array_equal(pl.zmap, sl.zmap) and pl.fam == sl.fam
    jp, js = pl._enumerate_jp(), sl._enumerate_jp()
    assert jp[8 * 13:] == js[8 * 25:]
    assert [jp[13 * i + 7:13 * i + 13] for i in range(8)] == [js[25 * i + 19:25 * i + 25] for i in range(8)]
    assert pl._enumerate_jk() == sl._enumerate_jk()


@pytest.mark.parametrize("settings", [dict(terrain="smooth_steps"), dict(n_terrain_params=10),
                                      dict(terrain="ramp", n_terrain_params=10)])
def test_pose_layout_rejects_inconsistent_terrain_settings(model, settings):
    with pytest.raises(ValueError):
        PoseLayout(model, PoseSettings(**settings))


def test_match_template_finds_the_smooth_pose_finder():
    from hippopt_b200.plugin import match_template

    m = match_template(81, 212, 89)
    assert m.kind == "pose_finder" and m.smooth_terrain and m.n_terrain_params == 10
    m = match_template(81, 202, 89)
    assert m.kind == "pose_finder" and not m.smooth_terrain and m.n_terrain_params == 0
    assert match_template(81, 207, 89) is None


@pytest.mark.parametrize("N,final", [(3, False), (3, True), (4, False), (4, True)])
def test_stage_solve_matches_dense_on_the_smooth_terrain(model, N, final):
    lay = KinoLayout(model, KinoSettings(horizon=N, final_state_constraint=final, terrain="smooth_steps",
                                         n_terrain_params=10))
    p = kino_parameters(lay, model, 1, np.random.default_rng(0))
    lb, ub = lay.bounds(p)
    eq, ine = np.nonzero(lb[0] == ub[0])[0], np.nonzero(lb[0] != ub[0])[0]
    planar = KinoLayout(model, KinoSettings(horizon=N, final_state_constraint=final))
    plb, pub = planar.bounds(kino_parameters(planar, model, 1, np.random.default_rng(0)))
    assert lay.m == planar.m and len(ine) == int((plb[0] != pub[0]).sum())
    kkt = StageKKT(lay.n_x, lay.m, N, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine,
                   linalg="torch")
    B = 3
    g = torch.Generator().manual_seed(10 + N)
    hv = torch.randn((B, lay.nnz_h), generator=g, dtype=torch.float64)
    jv = torch.randn((B, lay.nnz_j), generator=g, dtype=torch.float64)
    sig = torch.rand((B, len(ine)), generator=g, dtype=torch.float64) * 3.0
    delta = torch.tensor([40.0, 55.0, 70.0], dtype=torch.float64)
    rx = torch.randn((B, lay.n_x), generator=g, dtype=torch.float64)
    rE = torch.randn((B, len(eq)), generator=g, dtype=torch.float64)
    rE[:, kkt.dead_eq] = 0.0
    dx, dl = kkt.solve(hv, jv, sig, delta, 1e-6, rx, rE)
    K = kkt.dense_matrix(hv, jv, sig, delta, 1e-6, eq, ine, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row)
    ref = torch.linalg.solve(K, torch.cat([rx, rE], dim=1))
    u = torch.cat([dx, dl], dim=1)
    scale = ref.abs().amax(dim=1, keepdim=True)
    assert ((u - ref).abs() / scale).max().item() < 1e-9
    res = torch.einsum("bij,bj->bi", K, u) - torch.cat([rx, rE], dim=1)
    assert res.abs().max().item() < 1e-8 * max(1.0, float(scale.max()))
