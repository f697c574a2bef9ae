"""Batched LU kernels (csrc/lu.cu), the parts that need no GPU: the variant each (n, batch, nrhs) is dispatched to
(hb_debug_lu_plan, the function both launch paths use), and the reference helpers of tests/test_gpu_lu_shapes.py --
the layout conversion to LAPACK, the blocked model of the kernel's pivoting and the planted dyadic factorisations."""
import ctypes

import numpy as np
import pytest
import scipy.linalg as sla

import lu_reference as R

SMS = 148  # SM count of a B200; the plan takes it as an argument


def plan(lib, n, batch, nrhs, sms=SMS):
    out = (ctypes.c_int32 * 4)()
    rc = lib.hb_debug_lu_plan(n, batch, nrhs, sms, out)
    assert rc == 0, lib.hb_last_error().decode()
    return tuple(out)


@pytest.mark.parametrize("n", [1, 16, 255, 256, 257, 337, 352, 353, 436, 437, 442, 443, 512, 513, 715, 716, 768])
@pytest.mark.parametrize("sms", [SMS, 132])
def test_plan_at_the_dispatch_boundaries(built_library, n, sms):
    for batch in (1, sms, sms + 1, 2 * sms, 2 * sms + 3):
        assert plan(built_library, n, batch, 1, sms) == R.expected_plan(n, batch, 1, sms), (n, batch)


def test_plan_regimes_over_every_size(built_library):
    """RPT changes at 256/257 and 512/513, MB = 2 stops at 436/437, the solve's tile count at 352/353, 442/443 and
    715/716 -- and nowhere else."""
    plans = [plan(built_library, n, SMS + 1, 1) for n in range(1, 769)]
    change = [n for n in range(2, 769) if plans[n - 1][:3] != plans[n - 2][:3]]
    assert change == [257, 353, 437, 443, 513, 716]
    assert {p[:3] for p in plans} == {(1, 2, 4), (2, 2, 4), (2, 2, 3), (2, 1, 3), (2, 1, 4), (3, 1, 4), (3, 1, 3)}
    assert all(plan(built_library, n, SMS, 1)[1] == 1 for n in range(1, 769))


@pytest.mark.parametrize("nrhs", [1, 24, 25, 32, 33, 88, 172])
@pytest.mark.parametrize("n", [337, 400, 600, 768])
def test_plan_column_chunks(built_library, n, nrhs):
    got = plan(built_library, n, SMS + 1, nrhs)
    assert got == R.expected_plan(n, SMS + 1, nrhs, SMS)
    assert got[3] == {4: {1: 1, 24: 1, 25: 1, 32: 1, 33: 2, 88: 3, 172: 6},
                      3: {1: 1, 24: 1, 25: 2, 32: 2, 33: 2, 88: 4, 172: 8}}[got[2]][nrhs]


def test_plan_rejects_bad_arguments(built_library):
    out = (ctypes.c_int32 * 4)()
    for args in [(0, 1, 1, SMS), (769, 1, 1, SMS), (16, 0, 1, SMS), (16, 1, 0, SMS), (16, 1, 1, 0)]:
        assert built_library.hb_debug_lu_plan(*args, out) != 0, args
    assert built_library.hb_debug_lu_plan(16, 1, 1, SMS, None) != 0


def test_permutation_round_trip():
    rng = np.random.default_rng(0)
    for n in (1, 2, 17, 100):
        perm = rng.permutation(n)
        ipiv = R.perm_to_ipiv(perm)
        assert np.all(ipiv >= np.arange(n))
        assert np.array_equal(R.ipiv_to_perm(ipiv), perm)


NS_CPU = [1, 2, 15, 16, *range(17, 32), 33, 48, 64, 100]


@pytest.mark.parametrize("n", NS_CPU)
def test_to_lapack_matches_scipy_on_gaussian(n):
    """The blocked model in the kernel's layout, converted, is scipy's getrf: same pivots, same factors to rounding.
    The conversion only moves entries within a column."""
    A = R.gaussian(n, rng=n)
    F, piv, info = R.blocked_lu(A)
    lu, ref_piv = sla.lu_factor(A)
    assert info == 0
    assert np.array_equal(piv, ref_piv)
    G = R.to_lapack(F, piv)
    assert np.array_equal(np.sort(G, axis=0), np.sort(F, axis=0))
    assert np.abs(G - lu).max() <= 1e-12 * max(1.0, np.abs(lu).max())
    if n > R.NB and np.any(piv[R.NB:] != np.arange(R.NB, n)):
        assert not np.array_equal(F, G)  # the conversion is not vacuous here


@pytest.mark.parametrize("perm", ["reversed", "random", "identity"])
@pytest.mark.parametrize("n", [1, 2, 7, 16, 17, 31, 45, 100, 337])
def test_planted_factorisation_is_exact(n, perm):
    """Planted dyadic LU: scipy and the blocked model both return the planted L, U, pivots and solution bit for bit."""
    P = R.planted(n, perm, rng=1000 + n)
    LU = np.tril(P["L"], -1) + P["U"]
    lu, piv = sla.lu_factor(P["A"])
    assert np.array_equal(piv, P["ipiv"]) and np.array_equal(lu, LU)
    F, bpiv, info = R.blocked_lu(P["A"])
    assert info == 0 and np.array_equal(bpiv, P["ipiv"]) and np.array_equal(R.to_lapack(F, bpiv), LU)
    X, B = R.planted_rhs(P["A"], 3, rng=n)
    assert np.array_equal(sla.lu_solve((lu, piv), B), X)
    assert R.backward_error(P["A"], X, B) == 0.0


@pytest.mark.parametrize("n", [768])
def test_planted_factorisation_is_exact_at_the_largest_size(n):
    for perm in ("reversed", "random"):
        P = R.planted(n, perm, rng=n)
        lu, piv = sla.lu_factor(P["A"])
        assert np.array_equal(piv, P["ipiv"]) and np.array_equal(lu, np.tril(P["L"], -1) + P["U"])


def test_planted_random_permutation_fills_the_interchange_list():
    """A random permutation makes a full panel's composed interchange list 32 rows long (16 pivot rows, 16 rows they
    came from): the longest list the kernel's gather handles."""
    P = R.planted(337, "random", rng=5)
    ipiv = P["ipiv"]
    longest = 0
    for j0 in range(0, 337 - R.NB, R.NB):
        rows = set(range(j0, j0 + R.NB)) | {int(p) for p in ipiv[j0:j0 + R.NB]}
        longest = max(longest, len(rows))
    assert longest == 2 * R.NB


@pytest.mark.parametrize("c", [0, 5, 16, 40])
def test_planted_singular_factorisation(c):
    """U's row c and L's column c below the diagonal zero, identity permutation: partial pivoting keeps row c,
    stores zero multipliers and reports column c; every other value is exact."""
    n = 45
    P = R.planted(n, "identity", rng=c, singular_col=c)
    F, piv, info = R.blocked_lu(P["A"])
    assert info == c + 1
    assert np.array_equal(piv, np.arange(n))
    assert np.array_equal(F, np.tril(P["L"], -1) + P["U"])


def test_backward_error_definition():
    A = np.array([[2.0, 0.0], [0.0, 4.0]])
    x = np.array([1.0, 1.0])
    b = np.array([2.0, 4.0 + 1e-3])
    assert R.backward_error(A, x, b) == pytest.approx(1e-3 / (4.0 * 1.0 + 4.001))
    # the residual is accumulated in extended precision: 1 + 2^-60 - 1 is not lost where long double is wider
    if np.finfo(np.longdouble).eps < 2.0 ** -60:
        A = np.array([[1.0, 2.0 ** -60]])
        assert R.backward_error(A, np.array([1.0, 1.0]), np.array([1.0])) > 0.0


def test_diag_dominant_and_saddle_families():
    n = 100
    A = R.diag_dominant(n, rng=0)
    _, piv = sla.lu_factor(A)
    assert np.array_equal(piv, np.arange(n))
    K = R.saddle(R.SADDLE_N, rng=0)
    nx = R.SADDLE_NX
    assert np.array_equal(K, K.T)
    assert np.array_equal(K[nx:, nx:], -R.SADDLE_DELTA_C * np.eye(R.SADDLE_N - nx))
    _, piv = sla.lu_factor(K)
    assert np.any(piv - np.arange(R.SADDLE_N) > 2 * R.NB)  # pivots come from far below the diagonal


def test_saddle_split_is_the_kinodynamic_stage_block(model):
    from hippopt_b200.kino_layout import KinoLayout, KinoSettings
    from hippopt_b200.kkt import StageKKT
    from hippopt_b200.workloads import kino_parameters

    N = 5
    lay = KinoLayout(model, KinoSettings(horizon=N))
    lb, ub = lay.bounds(kino_parameters(lay, model, 1, np.random.default_rng(0)))
    eq, ine = np.nonzero(lb[0] == ub[0])[0], np.nonzero(lb[0] != ub[0])[0]
    kkt = StageKKT(lay.n_x, lay.m, N, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine,
                   linalg="torch")
    # the stage blocks are nb-square: nx variable slots, then the equality rows of the stage
    assert kkt.nb == R.SADDLE_N and kkt.nx == R.SADDLE_NX
    assert max(len(e) for e in kkt.eq_stage_rows) == R.SADDLE_N - R.SADDLE_NX
    assert R.saddle_split(R.SADDLE_N) == R.SADDLE_NX
