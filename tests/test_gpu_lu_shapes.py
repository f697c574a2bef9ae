"""Batched LU kernels (csrc/lu.cu) at the sizes and batch sizes where their variants change, against references that
do not depend on the kernels' summation order:

A. planted dyadic factorisations (tests/lu_reference.py): pivots, factors and solutions are known bit for bit;
B. Gaussian, saddle-point (the shape of a KKT stage block) and diagonally dominant matrices: the backward error, with
   the residual in extended precision, is within max(n eps, 8 x LAPACK's), and the pivots are LAPACK's up to the first
   near-tie of LAPACK's choice;
C. a batch of 1 (MB = 1 build of the factor kernel) and batches above the SM count (MB = 2 up to n = 436) return the
   same bits: the instruction sequence is the same, only the register budget differs;
D. a singular or NaN matrix inside a batch above the SM count reports its column in `info` and leaves every other
   matrix of the batch bit-identical to the clean run.

Every case asserts which kernel variant it runs (hb_debug_lu_plan, the function both launch paths use), and
test_plan_coverage checks that the cases together run all five factor instantiations and every solve tile count."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sla
import torch

import lu_reference as R

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
# both sides of every dispatch boundary (RPT 256/257, 512/513; MB 436/437; solve tiles 352/353, 442/443, 715/716),
# every last-panel width 1..15 (17..31) and the largest size
SIZES = sorted({1, 16, *range(17, 32), 255, 256, 257, 337, 352, 353, 436, 437, 442, 443, 512, 513, 715, 716, 768})
NRHS = (1, 9, 33, 88, 172)
NRHS_ETA = (1, 9)
FAMILIES = ("planted-reversed", "planted-random", "planted-identity", "gaussian", "saddle", "diag-dominant")
TIE = 1e-6  # LAPACK pivot margins below this are near-ties: the pivots are compared up to the first one
WORST = {}  # family -> worst eta_kernel / eta_LAPACK seen


def dev():
    return torch.device("cuda:0")


def sm_count():
    return torch.cuda.get_device_properties(dev()).multi_processor_count


def batches(sms):
    return (1, sms + 1, 2 * sms + 3)


def plan(lib, n, batch, nrhs, sms):
    out = (ctypes.c_int32 * 4)()
    assert lib.hb_debug_lu_plan(n, batch, nrhs, sms, out) == 0, lib.hb_last_error().decode()
    return tuple(out)


def _references(n):
    """The six matrices of one size and their CPU references."""
    rng = np.random.default_rng(n)
    P = [R.planted(n, perm, rng=rng) for perm in ("reversed", "random", "identity")]
    A = np.stack([p["A"] for p in P] + [R.gaussian(n, rng), R.saddle(n, rng), R.diag_dominant(n, rng)])
    X = rng.integers(-8, 9, size=(n, max(NRHS))) / 4.0
    B = A @ X  # exact for the planted matrices
    ref = dict(A=A, X=X, B=B, planted=P, lapack={})
    for t in range(3, 6):
        lu, piv = sla.lu_factor(A[t])
        eta = {r: R.backward_error(A[t], sla.lu_solve((lu, piv), B[t][:, :r]), B[t][:, :r]) for r in NRHS_ETA}
        ref["lapack"][t] = (piv, R.pivot_margins(lu), eta)
    return ref


def _check(ref, t, F, piv, info, X, what):
    """A and B on one matrix: F (n x n, the kernel's layout), piv, info, solutions X[r] (n x r), all on the CPU."""
    n = F.shape[0]
    fam = FAMILIES[t]
    assert info == 0, what
    if t < 3:
        P = ref["planted"][t]
        assert np.array_equal(piv, P["ipiv"]), what
        assert np.array_equal(R.to_lapack(F, piv), np.tril(P["L"], -1) + P["U"]), what
        for r, x in X.items():
            assert np.array_equal(x, ref["X"][:, :r]), (what, r)
        return
    lpiv, margin, eta_l = ref["lapack"][t]
    tie = np.nonzero(margin < TIE)[0]
    upto = int(tie[0]) if len(tie) else n  # steps after a near-tie may legitimately differ
    if t == 5:
        assert upto == n and np.array_equal(piv, np.arange(n)), what
    assert np.array_equal(piv[:upto], lpiv[:upto]), (what, upto, np.nonzero(piv[:upto] != lpiv[:upto])[0][:4])
    for r in NRHS_ETA:
        eta = R.backward_error(ref["A"][t], X[r], ref["B"][t][:, :r])
        assert eta <= max(n * EPS, 8.0 * eta_l[r]), (what, r, eta, eta_l[r])
        WORST[fam] = max(WORST.get(fam, 0.0), eta / max(eta_l[r], 1e-300))


def _run(A, B):
    from hippopt_b200.kkt import lu_factor, lu_solve

    F, piv, info = lu_factor(A)  # factors a transposed copy: A is left as it is
    X = {r: lu_solve(F, piv, B[:, :, :r]) for r in NRHS}
    return F.transpose(1, 2), piv, info, X  # F: L\U with rows first


@pytest.mark.parametrize("n", SIZES)
def test_lu_shapes(built_library, n):
    sms = sm_count()
    ref = _references(n)
    k = len(FAMILIES)
    A_d = torch.tensor(ref["A"], device=dev())
    B_d = torch.tensor(ref["B"], device=dev())
    one = None
    for batch in batches(sms):
        for r in NRHS:
            assert plan(built_library, n, batch, r, sms) == R.expected_plan(n, batch, r, sms), (n, batch, r)
        if batch == 1:
            runs = [_run(A_d[t:t + 1], B_d[t:t + 1]) for t in range(k)]
            F = torch.cat([u[0] for u in runs])
            piv = torch.cat([u[1] for u in runs])
            info = torch.cat([u[2] for u in runs])
            X = {r: torch.cat([u[3][r] for u in runs]) for r in NRHS}
        else:
            idx = torch.arange(batch, device=dev()) % k
            F, piv, info, X = _run(A_d[idx], B_d[idx])
        Fc, pc, ic = F[:k].cpu().numpy(), piv[:k].cpu().numpy(), info[:k].cpu().numpy()
        Xc = {r: X[r][:k].cpu().numpy() for r in NRHS}
        for t in range(k):
            _check(ref, t, Fc[t], pc[t], int(ic[t]), {r: Xc[r][t] for r in NRHS}, (FAMILIES[t], n, batch))
        if batch == 1:
            one = (F, piv, info, X)
            continue
        # C: every instance bit-identical to its batch-of-1 run
        idx = torch.arange(batch, device=dev()) % k
        assert torch.equal(piv, one[1][idx]) and torch.equal(info, one[2][idx]), (n, batch)
        assert torch.equal(F, one[0][idx]), (n, batch, "factors")
        for r in NRHS:
            assert torch.equal(X[r], one[3][r][idx]), (n, batch, r)
        if batch == sms + 1:
            _errors_inside_a_large_batch(n, A_d, B_d, (F, piv, info, X[1]))


def _errors_inside_a_large_batch(n, A_d, B_d, clean):
    """D, in a batch of sms + 1: planted singular matrices at several columns, an all-NaN column, a single NaN."""
    from hippopt_b200.kkt import lu_factor, lu_solve

    batch = clean[0].shape[0]
    k = len(FAMILIES)
    idx = torch.arange(batch, device=dev()) % k
    A = A_d[idx].clone()
    special = {}
    rng = np.random.default_rng(10_000 + n)
    last_panel = ((n - 1) // R.NB) * R.NB
    for j, c in enumerate(sorted({0, n // 2, last_panel + (n - 1 - last_panel) // 2, n - 1})):
        P = R.planted(n, "identity", rng=rng, singular_col=c)
        slot = 5 + 17 * j
        A[slot] = torch.tensor(P["A"], device=dev())
        special[slot] = ("singular", c, np.tril(P["L"], -1) + P["U"])
    c_nan = n // 3
    slot = batch - 1  # the last CTA of the launch
    A[slot] = A_d[3]
    A[slot, :, c_nan] = float("nan")
    special[slot] = ("nan-column", c_nan, None)
    slot = batch // 2
    A[slot] = A_d[3]
    A[slot, n // 2, n // 3] = float("nan")
    special[slot] = ("nan-entry", None, None)
    Fk, piv, info = lu_factor(A)
    x = lu_solve(Fk, piv, B_d[idx][:, :, :1])
    F = Fk.transpose(1, 2)
    info_c = info.cpu().numpy()
    for slot, (kind, c, LU) in special.items():
        if kind == "singular":
            assert info_c[slot] == c + 1, (n, kind, c)
            assert np.array_equal(piv[slot].cpu().numpy(), np.arange(n)), (n, kind, c)
            assert np.array_equal(F[slot].cpu().numpy(), LU), (n, kind, c)
        elif kind == "nan-column":
            assert info_c[slot] == c + 1, (n, kind, c)
        else:
            assert not torch.isfinite(x[slot]).all(), (n, kind)
    keep = torch.ones(batch, dtype=torch.bool, device=dev())
    keep[list(special)] = False
    assert torch.equal(F[keep], clean[0][keep]) and torch.equal(piv[keep], clean[1][keep]), n
    assert torch.equal(info[keep], clean[2][keep]) and torch.equal(x[keep], clean[3][keep]), n


def test_plan_coverage(built_library):
    """The cases of test_lu_shapes run all five factor instantiations and every solve tile count reachable for
    n <= 768 (4 and 3, each at two CTAs and at one CTA per SM)."""
    sms = sm_count()
    by_factor, by_ct = {}, {}
    for n in SIZES:
        for batch in batches(sms):
            rpt, mb, ct, _ = plan(built_library, n, batch, 1, sms)
            by_factor.setdefault((rpt, mb), set()).add((n, batch))
            by_ct.setdefault(ct, set()).add(n)
    print(f"\nLU plan coverage ({sms} SMs): factor <RPT, MB> -> sizes (batches)")
    for key in sorted(by_factor):
        cases = sorted(by_factor[key])
        ns = sorted({n for n, _ in cases})
        print(f"  lu_factor_kernel<{key[0]},{key[1]}>: {len(cases)} cases, n = {ns}, "
              f"batches {sorted({b for _, b in cases})}")
    for ct in sorted(by_ct):
        print(f"  lu_solve_staged_kernel<{ct}>: n = {sorted(by_ct[ct])}")
    assert set(by_factor) == {(1, 1), (1, 2), (2, 1), (2, 2), (3, 1)}
    assert set(by_ct) == {3, 4}
    # each tile count at both residencies: two CTAs per SM below 443, one above
    assert {(ct, min(by_ct[ct]) <= 442, max(by_ct[ct]) > 442) for ct in by_ct} == {(3, True, True), (4, True, True)}
    if WORST:
        print("worst eta_kernel / eta_LAPACK: " + ", ".join(f"{f} {v:.3g}" for f, v in sorted(WORST.items())))
