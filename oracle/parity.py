"""Parity metric of the tests (TEST INFRASTRUCTURE: imported by tests/, __graft_entry__.smoke() only).

north_star asks for 1e-10 RELATIVE agreement with the reference's evaluation.  An entry-wise relative error
needs a floor for entries that are structurally present but (nearly) cancel -- d h_ang / d pb_dot, a defect of
an almost feasible iterate -- and the floor must come from the scale of the data the entry was formed from,
not from the constant 1:

  f        |got - ref| <= rtol * |ref|
  grad_f   |got - ref| <= rtol * max(|ref_i|, ||grad_f||_inf of the instance)
  jac_g    |got - ref| <= rtol * max(|ref_e|, ||row of e||_inf)               (row = one constraint)
  g        |got - ref| <= rtol * max(|ref_i|, ||row i of jac_g||_inf * max(1, ||x||_inf))
           (a rounding-level relative perturbation of x moves g_i by that much)
  hess_l   |got - ref| <= rtol * max(|ref_e|, sqrt(S_r S_c)),  S_v = largest |entry| in row/column v of the
           symmetric matrix (invariant under a diagonal rescaling of the variables)

On top of the relative bound every check allows ONE UNIT OF ROUNDING of the largest entry of the instance's
array (eps * ||array||_inf, eps = 2.2e-16): entries that are structurally present but exactly zero in exact
arithmetic (all of d2L / d vb d s: the momentum map is linear in the base velocity) come out as +-1e-17 noise of
cancelling O(1) terms in any evaluation order, and a whole row of them has no scale of its own.  (For scale: the
round-1 metric had an absolute floor of 1e-10 * 1; this one is 2.2e-16 * ||array||_inf.)

Every function takes batched arrays [B, ...] and patterns in compressed-column form (colind, row).
"""
from __future__ import annotations

import numpy as np

RTOL = 1e-10


EPS = float(np.finfo(np.float64).eps)


def _rel(got, ref, floor, rtol=RTOL):
    """|got - ref| / max(|ref|, floor), after removing one unit of rounding of the instance's largest entry
    (expressed so that the result compares against rtol: err <= rtol  <=>  |d| <= rtol * den + eps * max|ref|)."""
    got, ref = np.asarray(got, dtype=float), np.asarray(ref, dtype=float)
    den = np.maximum(np.abs(ref), floor)
    r2 = np.atleast_2d(ref)
    noise = EPS * (np.abs(r2).max(axis=1, keepdims=True) if r2.size else 0.0)
    noise = np.broadcast_to(noise, r2.shape).reshape(ref.shape) if ref.ndim else float(np.max(noise))
    with np.errstate(divide="ignore", invalid="ignore"):
        err = np.maximum(np.abs(got - ref) - noise, 0.0) / den
    err = np.where((got == ref) | ((den == 0) & (got == ref)), 0.0, err)
    return err


def _report(name, err, rtol):
    worst = float(np.nanmax(err)) if err.size else 0.0
    if not np.isfinite(worst) or np.isnan(err).any():
        raise AssertionError(f"{name}: non-finite error (got or reference contains NaN/Inf)")
    assert worst <= rtol, (f"{name}: max relative error {worst:.3e} > {rtol:.1e} at "
                           f"{np.unravel_index(int(np.nanargmax(err)), err.shape)}")
    return worst


def jac_row_scale(jac_ref, row, m):
    """[B, m]: inf-norm of every Jacobian row."""
    jac_ref = np.atleast_2d(np.abs(jac_ref))
    S = np.zeros((jac_ref.shape[0], m))
    np.maximum.at(S, (slice(None), np.asarray(row)), jac_ref)
    return S


def hess_var_scale(hess_ref, colind, row):
    """[B, n]: largest |entry| in row/column v of the symmetric matrix stored as its upper triangle."""
    hess_ref = np.atleast_2d(np.abs(hess_ref))
    n = len(colind) - 1
    col = np.repeat(np.arange(n), np.diff(colind))
    S = np.zeros((hess_ref.shape[0], n))
    np.maximum.at(S, (slice(None), col), hess_ref)
    np.maximum.at(S, (slice(None), np.asarray(row)), hess_ref)
    return S, col


def check_f(got, ref, rtol=RTOL):
    return _report("f", _rel(got, ref, 0.0), rtol)


def check_grad(got, ref, rtol=RTOL):
    ref = np.atleast_2d(ref)
    return _report("grad_f", _rel(np.atleast_2d(got), ref, np.abs(ref).max(axis=1, keepdims=True)), rtol)


def check_jac(got, ref, jac_pattern, m, rtol=RTOL):
    ref = np.atleast_2d(ref)
    row = np.asarray(jac_pattern[1])
    S = jac_row_scale(ref, row, m)
    return _report("jac_g", _rel(np.atleast_2d(got), ref, S[:, row]), rtol)


def check_g(got, ref, jac_ref, jac_pattern, x, rtol=RTOL):
    ref = np.atleast_2d(ref)
    S = jac_row_scale(jac_ref, jac_pattern[1], ref.shape[1])
    xs = np.maximum(1.0, np.abs(np.atleast_2d(x)).max(axis=1, keepdims=True))
    return _report("g", _rel(np.atleast_2d(got), ref, S * xs), rtol)


def check_hess(got, ref, hess_pattern, rtol=RTOL):
    ref = np.atleast_2d(ref)
    S, col = hess_var_scale(ref, hess_pattern[0], hess_pattern[1])
    floor = np.sqrt(S[:, col] * S[:, np.asarray(hess_pattern[1])])
    return _report("hess_l", _rel(np.atleast_2d(got), ref, floor), rtol)


def check_all(got: dict, ref: dict, jac_pattern, hess_pattern, x, rtol=RTOL, keys=("f", "grad_f", "g", "jac", "hess")):
    """Compare the evaluator's outputs with reference values; returns {key: worst relative error}."""
    worst = {}
    m = np.atleast_2d(ref["g"]).shape[1] if "g" in ref else int(np.max(jac_pattern[1])) + 1
    for k in keys:
        if k not in got or k not in ref:
            continue
        if k == "f":
            worst[k] = check_f(got[k], ref[k], rtol)
        elif k == "grad_f":
            worst[k] = check_grad(got[k], ref[k], rtol)
        elif k == "jac":
            worst[k] = check_jac(got[k], ref[k], jac_pattern, m, rtol)
        elif k == "g":
            worst[k] = check_g(got[k], ref[k], ref["jac"], jac_pattern, x, rtol)
        elif k == "hess":
            worst[k] = check_hess(got[k], ref[k], hess_pattern, rtol)
    return worst


def reference_outputs(nlp, x, p, lam, sigma, dtype=np.float64):
    """The five nlpsol oracle functions evaluated by the CPU oracle (oracle/nlp.py) in floating type ``dtype``."""
    return {"f": nlp.eval_f(x, p, dtype), "grad_f": nlp.eval_grad_f(x, p, dtype), "g": nlp.eval_g(x, p, dtype),
            "jac": nlp.eval_jac(x, p, dtype), "hess": nlp.eval_hess(x, p, lam, sigma, dtype)}
