"""The oracle's `dtype` keyword: float64 by default, bit for bit what it always computed, and np.longdouble as an
extended-precision reference for the smooth-step terrain, whose fp64 tapes form 0 * inf far from a step.  CPU only."""
import os

import mpmath
import numpy as np
import pytest

from oracle import expressions as ex
from oracle import kinodynamic as kd
from oracle import parity
from oracle import sx

GOLD = os.path.join(os.path.dirname(__file__), "golden")
STAIRS = os.path.join(GOLD, "kino_n3_stairs.npz")
KEYS = ("f", "grad_f", "g", "jac", "hess")

extended = pytest.mark.skipif(np.finfo(np.longdouble).eps > 2.0 ** -63,
                              reason="long double is not an 80-bit extended type on this platform")


@pytest.fixture(scope="module")
def stairs(model):
    d = np.load(STAIRS)
    nlp, _ = kd.build(model, kd.Settings(horizon=int(d["horizon"]), final_state_constraint=bool(d["final"]),
                                         periodicity_constraint=bool(d["periodicity"]), terrain=ex.TwoSmoothSteps(),
                                         terrain_params=10))
    return nlp, d


def test_default_dtype_is_bit_identical_to_explicit_float64(stairs):
    nlp, d = stairs
    args = (d["x"], d["p"], d["lam"], d["sigma"])
    default = parity.reference_outputs(nlp, *args)
    explicit = parity.reference_outputs(nlp, *args, dtype=np.float64)
    for k in KEYS:
        assert default[k].dtype == np.float64 and explicit[k].dtype == np.float64, k
        assert np.array_equal(default[k], explicit[k]), k
    lb, ub = nlp.eval_bounds(d["p"])
    assert lb.dtype == np.float64 and np.array_equal(lb, d["lbg"]) and np.array_equal(ub, d["ubg"])


@extended
def test_longdouble_outputs_are_longdouble_and_agree_with_float64(stairs):
    nlp, d = stairs
    args = (d["x"], d["p"], d["lam"], d["sigma"])
    f64 = parity.reference_outputs(nlp, *args)
    ld = parity.reference_outputs(nlp, *args, dtype=np.longdouble)
    for k in KEYS:
        assert ld[k].dtype == np.longdouble, k
        assert np.isfinite(ld[k]).all(), k
    worst = parity.check_all(f64, ld, nlp.jac_structure()[:2], nlp.hess_structure()[:2], d["x"], rtol=1e-12)
    print("float64 oracle against the long-double oracle:", {k: f"{v:.2e}" for k, v in worst.items()})
    lb, ub = nlp.eval_bounds(d["p"], dtype=np.longdouble)
    assert lb.dtype == np.longdouble and np.array_equal(lb, d["lbg"]) and np.array_equal(ub, d["ubg"])


@extended
def test_longdouble_is_finite_where_float64_forms_nan(stairs, model):
    """Contact points moved far behind both steps (g > 1e6): exp(-g^20) underflows to 0 while the products of powers
    of g in the Hessian's graph overflow fp64, so the float64 tapes evaluate 0 * inf = NaN.  The long-double tapes
    have the exponent range to keep those products finite."""
    from hippopt_b200.kino_layout import NZ, P

    nlp, d = stairs
    x, p = d["x"].copy(), d["p"]
    N = int(d["horizon"])
    tp = p[:, -10:]  # the ten terrain parameters close the parameter vector
    for k in range(N):
        for i in (0, 5):
            x[:, NZ * k + 15 * i + P] = -3.0
            x[:, NZ * k + 15 * i + P + 1] = 0.35 if i == 0 else -0.35
    X, Y = x[:, P], x[:, P + 1]
    for s in range(2):
        l, w, ox, oy = tp[:, 5 * s], tp[:, 5 * s + 1], tp[:, 5 * s + 3], tp[:, 5 * s + 4]
        assert np.all((2 * (X - ox) / l) ** 10 + (2 * (Y - oy) / w) ** 10 > 1e6)
    args = (x, p, d["lam"], d["sigma"])
    with np.errstate(all="ignore"):
        f64 = parity.reference_outputs(nlp, *args)
    ld = parity.reference_outputs(nlp, *args, dtype=np.longdouble)
    assert not np.isfinite(f64["hess"]).all(), "the float64 oracle no longer forms 0 * inf far from a step"
    for k in KEYS:
        assert np.isfinite(ld[k]).all(), k
    # wherever float64 is finite the two agree
    ok = np.isfinite(f64["hess"])
    scale = np.abs(ld["hess"]).max()
    assert np.abs(f64["hess"][ok] - ld["hess"][ok]).max() <= 1e-12 * scale
    print(f"{(~ok).sum()} Hessian entries are NaN in float64 and finite in long double")


def _exact(v):
    n, d = v.as_integer_ratio()  # exact: mpmath.mpf(np.longdouble) would round through float
    return mpmath.mpf(n) / d


def _mp_step(v):
    """h = z - height exp(-g^20) of one step and its gradient in x, y, at 50 digits."""
    x, y, z, l, w, height, ox, oy = (mpmath.mpf(float(t)) for t in v)
    X, Y = 2 * (x - ox) / l, 2 * (y - oy) / w
    g = X ** 10 + Y ** 10
    e = mpmath.exp(-g ** 20)
    h = z - height * e
    dg = 20 * g ** 19 * height * e
    return [h, dg * 10 * X ** 9 * 2 / l, dg * 10 * Y ** 9 * 2 / w]


@extended
def test_longdouble_tapes_carry_a_64_bit_mantissa():
    """Height and gradient of one step, in the band, against mpmath: the long-double tapes are accurate to well below
    fp64's 1.1e-16, so every intermediate really holds 64 mantissa bits."""
    v = sx.syms("v", 8)
    step = ex.SmoothStep(v[3], v[4], v[5], origin=(v[6], v[7], 0.0))
    h = step.height(v[:3])
    grad = sx.gradient(h, [v[0], v[1]])
    tape = sx.Tape([h, *grad], list(v))
    rng = np.random.default_rng(11)
    pts = []
    for gx, gy in [(0.9, 0.01), (0.7, 0.2), (0.5, 0.45), (0.05, 0.85)]:
        l, w, height, ox, oy = 0.9, 0.8, rng.uniform(0.05, 0.15), 0.675, 0.1
        x = ox + 0.5 * l * gx ** 0.1
        y = oy - 0.5 * w * gy ** 0.1
        pts.append([x, y, 0.0, l, w, height, ox, oy])
    pts = np.array(pts)
    got = tape.eval(pts, dtype=np.longdouble)
    got64 = tape.eval(pts)
    worst = worst64 = 0.0
    with mpmath.workdps(50):
        for b in range(len(pts)):
            ref = _mp_step(pts[b])
            for j in range(3):
                worst = max(worst, float(abs((_exact(got[b, j]) - ref[j]) / ref[j])))
                worst64 = max(worst64, float(abs((_exact(got64[b, j]) - ref[j]) / ref[j])))
    print(f"worst relative error: long double {worst:.2e}, float64 {worst64:.2e}")
    assert worst < 1e-17
