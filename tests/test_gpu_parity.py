"""Parity tests proper: the CUDA path, called through the C ABI, against the committed golden
fixtures, against the CPU oracle on seeded inputs, and -- at BASELINE.json's full sizes -- through
size-independent properties.  Tolerance: 1e-10 RELATIVE (north_star); the floor under entries that
cancel is the scale of the row / column the entry belongs to, never the constant 1 (oracle/parity.py)."""
import glob
import os

import numpy as np
import pytest

from tests_support import golden_files
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden")
RTOL = 1e-10
RTOL_SMOOTH = RTOL  # config 5 (smooth-step terrain): same bar


def close(got, ref, rtol=RTOL):
    """Two evaluations of the SAME array by the CUDA path (two algorithms / two masks): relative to the
    largest magnitude of the instance's array."""
    got, ref = np.atleast_2d(got), np.atleast_2d(ref)
    err = np.abs(got - ref) / np.maximum(np.abs(ref), np.abs(ref).max(axis=1, keepdims=True))
    assert err.max() <= rtol, f"max relative error {err.max():.3e} at {np.unravel_index(err.argmax(), err.shape)}"


def check(out, ref, jac_pattern, hess_pattern, x, keys=("f", "grad_f", "g", "jac", "hess"), rtol=RTOL):
    """CUDA outputs against reference values with the row-scaled relative metric of oracle/parity.py."""
    from oracle import parity

    worst = parity.check_all(out, ref, jac_pattern, hess_pattern, x, rtol=rtol, keys=keys)
    print("worst relative errors:", {k: f"{v:.2e}" for k, v in worst.items()})
    return worst


def check_nlp(out, nlp, x, p, lam, sigma, **kw):
    from oracle import parity

    return check(out, parity.reference_outputs(nlp, x, p, lam, sigma), nlp.jac_structure()[:2], nlp.hess_structure()[:2], x, **kw)


def dev():
    return torch.device("cuda:0")


def run(ev, x, p, lam, sigma, mask=None):
    from hippopt_b200.evaluator import ALL

    t = [torch.tensor(np.ascontiguousarray(a), device=dev()) for a in (x, p, lam, sigma)]
    out = ev.eval(ALL if mask is None else mask, *t)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


@pytest.mark.parametrize("path", golden_files("kino"))
def test_kino_golden(model, built_library, path):
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings

    d = np.load(path)
    smooth = bool(d["smooth"]) if "smooth" in d else False
    ev = KinoEvaluator(model, KinoSettings(horizon=int(d["horizon"]), final_state_constraint=bool(d["final"]),
                                           periodicity_constraint=bool(d["periodicity"]),
                                           terrain="smooth_steps" if smooth else "planar",
                                           n_terrain_params=10 if smooth else 0))
    assert np.array_equal(ev.jac_sparsity()[1], d["jac_row"]) and np.array_equal(ev.hess_sparsity()[1], d["hess_row"])
    out = run(ev, d["x"], d["p"], d["lam"], d["sigma"])
    check(out, d, (d["jac_colind"], d["jac_row"]), (d["hess_colind"], d["hess_row"]), d["x"])


@pytest.mark.parametrize("path", golden_files("toy"))
def test_toy_golden(built_library, path):
    from hippopt_b200.evaluator import ToyEvaluator

    d = np.load(path)
    ev = ToyEvaluator(int(d["horizon"]), "euler" if "euler" in path else "trapezoid", float(d["dt"]))
    jc, jr = ev.jac_sparsity()
    hc, hr = ev.hess_sparsity()
    assert np.array_equal(jc, d["jac_colind"]) and np.array_equal(jr, d["jac_row"])
    assert np.array_equal(hc, d["hess_colind"]) and np.array_equal(hr, d["hess_row"])
    lb, ub = ev.bounds(d["p"])
    assert np.array_equal(lb, d["lbg"]) and np.array_equal(ub, d["ubg"])
    out = run(ev, d["x"], d["p"], d["lam"], d["sigma"])
    check(out, d, (jc, jr), (hc, hr), d["x"])


def test_toy_reference_solution(built_library):
    """/root/reference/test/test_multiple_shooting.py:336-353 at the test's own size (N = 100)."""
    from hippopt_b200.evaluator import F, G, GRAD_F, ToyEvaluator
    from oracle import toy

    N, dt, g, x0, v0 = 100, 0.01, -9.81, 1.0, 0.0
    ev = ToyEvaluator(N, "euler", dt)
    assert (ev.n_x, ev.m) == (900, 703)
    x = toy.closed_form_solution(N, dt, g, x0, v0)[None]
    p = np.array([[g, x0, v0]])
    out = run(ev, x, p, np.zeros((1, ev.m)), np.ones(1), F | G | GRAD_F)
    lb, ub = ev.bounds(p)
    assert np.all(out["g"] >= lb - 1e-12) and np.all(out["g"] <= ub + 1e-12)
    assert out["f"][0] == pytest.approx(3 * (98 * 25.0 + 36.0), rel=1e-14)
    assert np.abs(out["grad_f"][0, :600]).max() < 1e-12


# (60, True, True): a horizon twice the bench's -- the knot-relative scatter tables (first / interior / last classes) over 58
# interior knots, with the final-state and periodicity rows
@pytest.mark.parametrize("N,fin,per,noise", [(2, False, False, 0.3), (6, True, True, 0.05), (3, True, False, 1.0),
                                             (60, True, True, 0.05)])
def test_kino_against_oracle(model, built_library, N, fin, per, noise):
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch
    from oracle import kinodynamic as kd

    ev = KinoEvaluator(model, KinoSettings(horizon=N, final_state_constraint=fin, periodicity_constraint=per))
    B = 3 if N < 30 else 2
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=100 + N, noise=noise, spread=2.0)
    sigma = np.array([0.0, 1.0, 3.5])[:B]
    nlp, _ = kd.build(model, kd.Settings(horizon=N, final_state_constraint=fin, periodicity_constraint=per))
    out = run(ev, x, p, lam, sigma)
    check_nlp(out, nlp, x, p, lam, sigma)


@pytest.mark.parametrize("N,fin,noise", [(3, True, 0.05), (4, False, 0.15)])
def test_kino_smooth_terrain_against_oracle(model, built_library, N, fin, noise):
    """BASELINE config 5: two smooth steps (SmoothTerrain.step + SmoothTerrain.step) with the terrain
    parameters as runtime data.  Far from a step the reference's formula evaluates 0 * inf = NaN in fp64 in the
    high derivatives (exp(-g^20) underflows while products of powers of g overflow); the long-double oracle has
    the exponent range to stay finite there, so every entry is compared."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch
    from oracle import expressions as ex
    from oracle import kinodynamic as kd

    ev = KinoEvaluator(model, KinoSettings(horizon=N, terrain="smooth_steps", n_terrain_params=10,
                                           final_state_constraint=fin))
    x, p, lam, sigma = kino_batch(ev.layout, model, 3, seed=40 + N, noise=noise)
    sigma = np.array([1.0, 0.3, 2.0])
    nlp, _ = kd.build(model, kd.Settings(horizon=N, terrain=ex.TwoSmoothSteps(), terrain_params=10,
                                         final_state_constraint=fin))
    assert np.array_equal(ev.jac_sparsity()[1], nlp.jac_structure()[1])
    assert np.array_equal(ev.hess_sparsity()[1], nlp.hess_structure()[1])
    out = run(ev, x, p, lam, sigma)
    from oracle import parity

    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(out[k]).all() and np.isfinite(r).all(), k
    check(out, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2], x, rtol=RTOL_SMOOTH)


@pytest.mark.parametrize("noise", [0.05, 0.4])
def test_pose_finder_against_oracle(model, built_library, noise):
    """BASELINE config 2: humanoid_pose_finder static pose, single knot, exact Hessian."""
    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.workloads import pose_batch
    from oracle import pose_finder as pf

    ev = PoseEvaluator(model)
    assert (ev.n_x, ev.n_p, ev.m) == (81, 202, 89)  # SURVEY.md Appendix B.4
    nlp, _ = pf.build(model)
    assert np.array_equal(ev.jac_sparsity()[0], nlp.jac_structure()[0])
    assert np.array_equal(ev.jac_sparsity()[1], nlp.jac_structure()[1])
    assert np.array_equal(ev.hess_sparsity()[1], nlp.hess_structure()[1])
    x, p, lam, sigma = pose_batch(ev.layout, model, 6, seed=9, noise=noise)
    sigma = np.linspace(0.2, 2.0, 6)
    lb, ub = ev.bounds(p)
    olb, oub = nlp.eval_bounds(p)
    assert np.array_equal(lb, olb) and np.array_equal(ub, oub)
    out = run(ev, x, p, lam, sigma)
    check_nlp(out, nlp, x, p, lam, sigma)


def test_pose_finder_config2_batch(model, built_library):
    """Config 2 at its stated batch (4096): deterministic, batch-order independent, finite."""
    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.workloads import pose_batch

    ev = PoseEvaluator(model)
    x, p, lam, sigma = pose_batch(ev.layout, model, 4096, seed=1)
    out = run(ev, x, p, lam, sigma)
    perm = np.random.default_rng(3).permutation(4096)
    again = run(ev, x[perm], p[perm], lam[perm], sigma[perm])
    for k in out:
        assert np.isfinite(out[k]).all()
        assert np.array_equal(again[k], out[k][perm]), k


def test_kino_edge_cases(model, built_library):
    """Single instance, shared parameter vector, zero multipliers, partial masks, argument errors."""
    from hippopt_b200 import _capi
    from hippopt_b200.evaluator import ALL, F, G, GRAD_F, HESS_L, JAC_G, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    ev = KinoEvaluator(model, KinoSettings(horizon=4))
    x, p, lam, sigma = kino_batch(ev.layout, model, 5, seed=7, noise=0.1)
    p[:] = p[0]
    full = run(ev, x, p, lam, sigma)
    X, P1, L, S = (torch.tensor(a, device=dev()) for a in (x, p[0].copy(), lam, sigma))
    shared = ev.eval(ALL, X, P1, L, S)
    torch.cuda.synchronize()
    for k in full:
        assert np.array_equal(shared[k].cpu().numpy(), full[k]), k  # bit-identical
    one = run(ev, x[2:3], p[2:3], lam[2:3], sigma[2:3])
    for k in full:
        assert np.array_equal(one[k][0], full[k][2]), k  # batching does not change results
    part = run(ev, x, p, lam, sigma, F | G)
    assert set(part) == {"f", "g"} and np.array_equal(part["g"], full["g"]) and np.array_equal(part["f"], full["f"])
    # The kinematic rows of jac_g come from the forward tangents of the direction lanes whatever the mask ...
    jac_only = run(ev, x, p, lam, sigma, JAC_G)
    assert np.array_equal(jac_only["jac"], full["jac"])
    jac_grad = run(ev, x, p, lam, sigma, JAC_G | GRAD_F)
    assert np.array_equal(jac_grad["jac"], full["jac"]) and np.array_equal(jac_grad["grad_f"], full["grad_f"])
    # ... and, as an option, from the row-per-lane adjoint sweep: two algorithms, equal to rounding
    ev.set_option("JAC_ADJOINT", 1)
    adj = run(ev, x, p, lam, sigma, JAC_G | GRAD_F)
    ev.set_option("JAC_ADJOINT", 0)
    assert not np.array_equal(adj["jac"], full["jac"])
    close(adj["jac"], full["jac"], rtol=1e-13)
    close(adj["grad_f"], full["grad_f"], rtol=1e-12)
    with pytest.raises(_capi.EvaluationError):
        _capi.check(_capi.lib().hb_set_option(ev._h, 99, 1), "hb_set_option")
    again = run(ev, x, p, lam, sigma)
    for k in full:
        assert np.array_equal(again[k], full[k]), k  # same mask: bit-reproducible
    zero = run(ev, x, p, np.zeros_like(lam), np.zeros_like(sigma), HESS_L)
    assert np.abs(zero["hess"]).max() == 0.0
    with pytest.raises(ValueError):
        ev.eval(ALL, X[:, :-1].contiguous(), P1, L, S)
    with pytest.raises(ValueError):
        ev.eval(HESS_L, X, P1)
    with pytest.raises(_capi.EvaluationError):
        ev.eval(0, X, P1)


@pytest.fixture(scope="module")
def config3(model):
    """BASELINE.json config 3: single step on flat ground, N = 30, batch of 1024."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    ev = KinoEvaluator(model, KinoSettings(horizon=30))
    x, p, lam, sigma = kino_batch(ev.layout, model, 1024, seed=2)
    return ev, x, p, lam, sigma


def _spmv_ccs(colind, row, vals, d, n_rows, transpose=False):
    """y = A d (or A^T d) for a batch of CCS value arrays sharing one pattern."""
    col = np.repeat(np.arange(len(colind) - 1), np.diff(colind))
    y = np.zeros((vals.shape[0], n_rows if not transpose else len(colind) - 1))
    if not transpose:
        np.add.at(y, (slice(None), row), vals * d[:, col])
    else:
        np.add.at(y, (slice(None), col), vals * d[:, row])
    return y


def test_config3_full_size_properties(config3):
    """Full-size checks that need no oracle: directional derivatives of g / of the Lagrangian gradient
    reproduce J d and H d; results are deterministic and independent of the batch order."""
    from hippopt_b200.evaluator import G, GRAD_F, JAC_G

    ev, x, p, lam, sigma = config3
    lay = ev.layout
    out = run(ev, x, p, lam, sigma)
    again = run(ev, x, p, lam, sigma)
    for k in out:
        assert np.array_equal(out[k], again[k]), f"{k} is not deterministic"
    perm = np.random.default_rng(0).permutation(x.shape[0])
    shuffled = run(ev, x[perm], p[perm], lam[perm], sigma[perm])
    for k in out:
        assert np.array_equal(shuffled[k], out[k][perm]), f"{k} depends on the batch order"
    assert np.isfinite(out["jac"]).all() and np.isfinite(out["hess"]).all()
    rng = np.random.default_rng(1)
    d = rng.normal(size=x.shape)
    eps = 1e-6
    plus = run(ev, x + eps * d, p, lam, sigma, G | GRAD_F | JAC_G)
    minus = run(ev, x - eps * d, p, lam, sigma, G | GRAD_F | JAC_G)
    Jd = _spmv_ccs(lay.jac_colind, lay.jac_row, out["jac"], d, lay.m)
    fd = (plus["g"] - minus["g"]) / (2 * eps)
    assert np.abs(fd - Jd).max() <= 1e-5 * max(1.0, np.abs(Jd).max())

    def lag_grad(o):
        return sigma[:, None] * o["grad_f"] + _spmv_ccs(lay.jac_colind, lay.jac_row, o["jac"], lam, lay.m, transpose=True)

    fdh = (lag_grad(plus) - lag_grad(minus)) / (2 * eps)
    col = np.repeat(np.arange(lay.n_x), np.diff(lay.hess_colind))
    Hd = _spmv_ccs(lay.hess_colind, lay.hess_row, out["hess"], d, lay.n_x)
    off = lay.hess_row != col
    strict = out["hess"] * off  # mirror the strictly-upper part
    np.add.at(Hd, (slice(None), col), strict * d[:, lay.hess_row])
    assert np.abs(fdh - Hd).max() <= 2e-5 * max(1.0, np.abs(Hd).max())


def test_config4_periodic_step_full_size(model, built_library):
    """BASELINE config 4: periodic walking step (final-state and periodicity constraints), 4096 instances;
    the 512-instance shard one of 8 GPUs owns is evaluated, plus two instances against the oracle."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.sharding import shard_range
    from hippopt_b200.workloads import kino_batch
    from oracle import kinodynamic as kd

    ev = KinoEvaluator(model, KinoSettings(horizon=30, final_state_constraint=True, periodicity_constraint=True))
    assert ev.m == 8142 + 105 + 84 - 6
    lo, hi = shard_range(4096, 3, 8)
    x, p, lam, sigma = kino_batch(ev.layout, model, hi - lo, seed=3)
    out = run(ev, x, p, lam, sigma)
    again = run(ev, x[::-1].copy(), p[::-1].copy(), lam[::-1].copy(), sigma[::-1].copy())
    for k in out:
        assert np.isfinite(out[k]).all()
        assert np.array_equal(again[k][::-1], out[k]), k
    idx = np.array([5, 400])
    nlp, _ = kd.build(model, kd.Settings(horizon=30, final_state_constraint=True, periodicity_constraint=True))
    check_nlp({k: v[idx] for k, v in out.items()}, nlp, x[idx], p[idx], lam[idx], sigma[idx])


def test_config5_stairs_full_size(model, built_library):
    """BASELINE config 5: walking on stairs, horizon 50, randomised step heights as runtime terrain
    parameters; one 512-instance shard: finite, deterministic, first-order consistent (J d vs central
    differences of g), and four instances against the oracle at this size (f, g, grad_f, jac_g, hess_l)."""
    from hippopt_b200.evaluator import G, JAC_G, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    ev = KinoEvaluator(model, KinoSettings(horizon=50, terrain="smooth_steps", n_terrain_params=10,
                                           final_state_constraint=True))
    assert ev.n_x == 189 * 50 + 6
    x, p, lam, sigma = kino_batch(ev.layout, model, 512, seed=4)
    assert len(np.unique(p[:, ev.layout.po.terrain + 2])) == 512  # a different step height per instance
    out = run(ev, x, p, lam, sigma)
    again = run(ev, x, p, lam, sigma)
    for k in out:
        assert np.isfinite(out[k]).all(), k
        assert np.array_equal(out[k], again[k]), k
    lay = ev.layout
    d = np.random.default_rng(2).normal(size=x.shape)
    eps = 1e-6
    gp = run(ev, x + eps * d, p, lam, sigma, G)["g"]
    gm = run(ev, x - eps * d, p, lam, sigma, G)["g"]
    Jd = _spmv_ccs(lay.jac_colind, lay.jac_row, run(ev, x, p, lam, sigma, JAC_G)["jac"], d, lay.m)
    assert np.abs((gp - gm) / (2 * eps) - Jd).max() <= 1e-4 * max(1.0, np.abs(Jd).max())
    # oracle samples AT THE FULL SIZE (N = 50, all five outputs): instances spread over the shard, incl. first / last
    from oracle import expressions as ex
    from oracle import kinodynamic as kd

    nlp, _ = kd.build(model, kd.Settings(horizon=50, terrain=ex.TwoSmoothSteps(), terrain_params=10,
                                         final_state_constraint=True))
    assert np.array_equal(lay.jac_row, nlp.jac_structure()[1]) and np.array_equal(lay.jac_colind, nlp.jac_structure()[0])
    assert np.array_equal(lay.hess_row, nlp.hess_structure()[1]) and np.array_equal(lay.hess_colind, nlp.hess_structure()[0])
    idx = np.array([0, 137, 300, 511])
    from oracle import parity

    # long double: finite where the fp64 graph forms 0 * inf far from a step (see the smooth-terrain test above)
    ref = parity.reference_outputs(nlp, x[idx], p[idx], lam[idx], sigma[idx], dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(r).all(), k
    check({k: v[idx] for k, v in out.items()}, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2], x[idx],
          rtol=RTOL_SMOOTH)


@pytest.mark.parametrize("config", [4, 5])
def test_configs_4_and_5_at_their_stated_batch(model, built_library, config):
    """BASELINE configs 4 and 5 at the stated batch of 4096 instances on ONE GPU (the bench shards them over 8):
    every instance evaluated, shard-by-shard results identical to the whole batch (sharding by instance changes
    nothing), oracle samples from the first, a middle and the last shard."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.sharding import shard_range
    from hippopt_b200.workloads import kino_batch
    from oracle import expressions as ex
    from oracle import kinodynamic as kd
    from oracle import parity

    if config == 4:
        st = KinoSettings(horizon=30, final_state_constraint=True, periodicity_constraint=True)
        ks = kd.Settings(horizon=30, final_state_constraint=True, periodicity_constraint=True)
    else:
        st = KinoSettings(horizon=50, terrain="smooth_steps", n_terrain_params=10, final_state_constraint=True)
        ks = kd.Settings(horizon=50, terrain=ex.TwoSmoothSteps(), terrain_params=10, final_state_constraint=True)
    ev = KinoEvaluator(model, st)
    B = 4096
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=40 + config)
    X, P, L, S = (torch.tensor(a, device=dev()) for a in (x, p, lam, sigma))
    from hippopt_b200.evaluator import ALL

    out = ev.eval(ALL, X, P, L, S)
    torch.cuda.synchronize()
    whole = {k: v.clone() for k, v in out.items()}
    for k, v in whole.items():
        assert bool(torch.isfinite(v).all()), k
    for r in (0, 3, 7):
        lo, hi = shard_range(B, r, 8)
        part = ev.eval(ALL, X[lo:hi].contiguous(), P[lo:hi].contiguous(), L[lo:hi].contiguous(), S[lo:hi].contiguous())
        torch.cuda.synchronize()
        for k, v in part.items():
            assert torch.equal(v, whole[k][lo:hi]), (k, r)
    idx = np.array([0, 2049, 4095])
    nlp, _ = kd.build(model, ks)
    ref = parity.reference_outputs(nlp, x[idx], p[idx], lam[idx], sigma[idx], dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(r).all(), k
    check({k: whole[k][idx].cpu().numpy() for k in ref}, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2],
          x[idx], rtol=RTOL_SMOOTH)


def test_config3_samples_against_oracle(model, config3):
    """Two instances of the full-size batch against the CPU oracle (finishes in seconds)."""
    from oracle import kinodynamic as kd

    ev, x, p, lam, sigma = config3
    idx = np.array([0, 517])
    out = run(ev, x[idx], p[idx], lam[idx], sigma[idx])
    nlp, _ = kd.build(model, kd.Settings(horizon=30))
    check_nlp(out, nlp, x[idx], p[idx], lam[idx], sigma[idx])


@pytest.mark.parametrize("B", [1, 3, 5, 130])
def test_kino_batch_sizes_not_multiple_of_the_cta(model, built_library, B):
    """Ragged batches: B * N is not a multiple of the 4 warps per CTA; every instance must still be
    written, identically to evaluating it alone."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    ev = KinoEvaluator(model, KinoSettings(horizon=3))
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=60 + B, noise=0.1)
    out = run(ev, x, p, lam, sigma)
    last = run(ev, x[-1:], p[-1:], lam[-1:], sigma[-1:])
    for k in out:
        assert np.isfinite(out[k]).all()
        assert np.array_equal(out[k][-1], last[k][0]), k


def test_non_finite_inputs_are_passed_through(model, built_library):
    """NaN / Inf are not trapped (include/hippopt_b200.h): a NaN in one instance poisons only that
    instance's outputs -- IPOPT handles it by rejecting the step [ext]."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch

    ev = KinoEvaluator(model, KinoSettings(horizon=3))
    x, p, lam, sigma = kino_batch(ev.layout, model, 3, seed=77, noise=0.1)
    clean = run(ev, x, p, lam, sigma)
    x[1, 189 + 157] = np.nan  # a joint position of knot 1 of instance 1
    out = run(ev, x, p, lam, sigma)
    assert np.isnan(out["g"][1]).any() and np.isnan(out["hess"][1]).any()
    for k in out:
        assert np.array_equal(out[k][0], clean[k][0]) and np.array_equal(out[k][2], clean[k][2]), k


def test_minimal_horizon(model, built_library):
    """Horizon 2 (one interval): first and last knot only, with final state and periodicity rows."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch
    from oracle import kinodynamic as kd

    ev = KinoEvaluator(model, KinoSettings(horizon=2, final_state_constraint=True, periodicity_constraint=True))
    x, p, lam, sigma = kino_batch(ev.layout, model, 2, seed=5, noise=0.2)
    nlp, _ = kd.build(model, kd.Settings(horizon=2, final_state_constraint=True, periodicity_constraint=True))
    out = run(ev, x, p, lam, sigma)
    check_nlp(out, nlp, x, p, lam, sigma)


def test_other_joint_orders(built_library):
    """The kernels take the tree as data (parents, sub-tree masks, the host-built sweep schedule): a joint list
    with the limbs in another order -- other body numbers, foot / chest bodies, branch slots -- must give the
    same agreement with the oracle; an interleaved list, which would need a branch accumulator per body, is
    refused at creation with a message, not at launch."""
    from hippopt_b200 import _capi
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.robot_model import ERGOCUB_JOINTS, RobotModel, synthetic_ergocub_urdf
    from hippopt_b200.workloads import kino_batch
    from oracle import kinodynamic as kd

    torso, l_arm, r_arm, l_leg, r_leg = (ERGOCUB_JOINTS[0:3], ERGOCUB_JOINTS[3:7], ERGOCUB_JOINTS[7:11],
                                         ERGOCUB_JOINTS[11:17], ERGOCUB_JOINTS[17:23])
    frames = ["l_sole", "r_sole", "chest"]
    urdf = synthetic_ergocub_urdf(seed=7)
    model2 = RobotModel.from_urdf(urdf, l_leg + r_leg + torso + r_arm + l_arm, "root_link", frames=frames)
    assert list(model2.parent[:8]) == [-1, 0, 1, 2, 3, 4, 5, 0]
    ev = KinoEvaluator(model2, KinoSettings(horizon=3, final_state_constraint=True))
    nlp, _ = kd.build(model2, kd.Settings(horizon=3, final_state_constraint=True))
    assert np.array_equal(ev.jac_sparsity()[1], nlp.jac_structure()[1])
    assert np.array_equal(ev.hess_sparsity()[1], nlp.hess_structure()[1])
    x, p, lam, sigma = kino_batch(ev.layout, model2, 3, seed=4, noise=0.2)
    out = run(ev, x, p, lam, sigma)
    check_nlp(out, nlp, x, p, lam, sigma)
    jac_only = run(ev, x, p, lam, sigma, 8)
    close(jac_only["jac"], out["jac"], rtol=1e-13)

    interleaved = [j for grp in zip(l_leg, r_leg) for j in grp] + torso + [j for grp in zip(l_arm, r_arm) for j in grp]
    model3 = RobotModel.from_urdf(urdf, interleaved, "root_link", frames=frames)
    with pytest.raises(_capi.EvaluationError, match="branch accumulators"):
        KinoEvaluator(model3, KinoSettings(horizon=2))


@pytest.mark.parametrize("smooth", [False, True])
def test_named_cost_values_against_oracle(model, built_library, smooth):
    """Row f4 / a30: `hb_eval_cost_terms` gives the value of every NAMED cost expression
    (opti_solver.py:526-529); per name against the oracle's recording of the planner's minimize calls, and the
    sum against f."""
    from hippopt_b200 import naming
    from hippopt_b200.evaluator import F, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.workloads import kino_batch
    from oracle import expressions as ex
    from oracle import kinodynamic as kd

    N, B = 4, 3
    ev = KinoEvaluator(model, KinoSettings(horizon=N, terrain="smooth_steps" if smooth else "planar",
                                           n_terrain_params=10 if smooth else 0))
    extra = dict(terrain=ex.TwoSmoothSteps(), terrain_params=10) if smooth else {}
    nlp, _ = kd.build(model, kd.Settings(horizon=N, **extra))
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=21, noise=0.2)
    X, P = (torch.tensor(a, device=dev()) for a in (x, p))
    terms = ev.cost_terms(X, P).cpu().numpy()
    f = ev.eval(F, X, P)["f"].cpu().numpy()
    ref = nlp.eval_cost_terms(x, p)  # (B, applications), recording order
    slots = naming.cost_slots(ev.layout)
    assert set(slots) == set(nlp.cost_names)
    scale = np.abs(ref).max(axis=1)
    for j, name in enumerate(nlp.cost_names):
        k, s = slots[name]
        err = np.abs(terms[:, k, s] - ref[:, j]) / np.maximum(np.abs(ref[:, j]), 1e-300)
        ok = (err <= RTOL) | (np.abs(terms[:, k, s] - ref[:, j]) <= 2.3e-16 * scale)
        assert ok.all(), f"{name}: {terms[:, k, s]} vs {ref[:, j]}"
    named = np.zeros_like(terms, dtype=bool)
    for k, s in slots.values():
        named[:, k, s] = True
    assert np.all(terms[~named] == 0.0)  # expressions that do not exist at knot 0
    assert np.allclose(terms.sum(axis=(1, 2)), f, rtol=1e-13, atol=0)
    for b in range(B):
        by_name = naming.cost_values(ev.layout, terms[b])
        assert by_name["com_velocity_error[0]"] == terms[b, 0, 32]
