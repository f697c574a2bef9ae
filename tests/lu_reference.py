"""Reference helpers for the batched LU kernels (csrc/lu.cu): layout conversion, a numpy model of the kernel's blocked
partial pivoting, backward errors in extended precision and the test-matrix families.

Factor layout.  The kernel factors 16-column panels and applies a panel's interchanges to the panel and the trailing
columns only: the L columns of earlier panels keep the row order they had when their panel was factored (LINPACK-style
across panels).  `to_lapack` applies the later interchanges to them, which gives LAPACK getrf's layout.

Planted dyadic LU.  P A = L U with a unit lower L whose off-diagonal entries are multiples of 1/8 with |L_ij| <= 1/2,
U's diagonal in {+-1, +-2} and its off-diagonal entries multiples of 1/4, x multiples of 1/4 and b = A x.  Every value
partial pivoting and the substitutions form is then a dyadic far inside fp64's 53 bits, whatever the summation order,
and every pivot is unambiguous (|L| <= 1/2 < 1).  The factors, the pivots and the solution are therefore known bit for
bit for any kernel variant, tile shape or tensor-core accumulation order.  The family cannot see lost precision (a
float32 detour is exact on these values too): the Gaussian and saddle-point families are there for that."""
from __future__ import annotations

import numpy as np

NB = 16  # panel width of lu_factor_kernel (LU_NB)

# split of a kinodynamic stage block (n = 337): 195 variable slots, 142 equality rows (tests/test_lu_plan_cpu.py
# checks it against a real StageKKT)
SADDLE_N, SADDLE_NX = 337, 195
SADDLE_DELTA, SADDLE_DELTA_C = 1e-2, 1e-9


# ---------------------------------------------------------------------------------------------------- layouts
def perm_to_ipiv(perm) -> np.ndarray:
    """Row permutation (row i of P A = row perm[i] of A) -> LAPACK interchange sequence (0-based, ipiv[j] >= j)."""
    perm = np.asarray(perm)
    n = len(perm)
    cur = np.arange(n)
    where = np.arange(n)  # where[r] = position of original row r in cur
    ipiv = np.empty(n, dtype=np.int64)
    for j in range(n):
        p = where[perm[j]]
        ipiv[j] = p
        rj, rp = cur[j], cur[p]
        cur[j], cur[p] = rp, rj
        where[rp], where[rj] = j, p
    return ipiv


def ipiv_to_perm(ipiv) -> np.ndarray:
    perm = np.arange(len(ipiv))
    for j, p in enumerate(ipiv):
        perm[[j, p]] = perm[[p, j]]
    return perm


def to_lapack(F, piv, nb: int = NB) -> np.ndarray:
    """Kernel factors (n x n, L\\U in one matrix, LINPACK-style across nb-column panels) -> LAPACK getrf layout: the
    interchanges of every panel are applied to the L columns left of it.  Moves entries only."""
    F = np.array(F, copy=True)
    for j, p in enumerate(np.asarray(piv)):
        j0 = (j // nb) * nb
        if p != j and j0 > 0:
            F[[j, p], :j0] = F[[p, j], :j0]
    return F


def blocked_lu(A, nb: int = NB):
    """numpy model of lu_factor_kernel's arithmetic order: per nb-column panel, unblocked partial pivoting (ties to the
    lowest row) with the rows exchanged in the panel and the trailing columns only, U12 = L11^{-1} A12, then
    A22 -= L21 U12.  Returns (F in the kernel's layout, piv, info)."""
    F = np.array(A, dtype=np.float64, copy=True)
    n = F.shape[0]
    piv = np.arange(n)
    info = 0
    for j0 in range(0, n, nb):
        j1 = min(j0 + nb, n)
        for c in range(j0, j1):
            p = c + int(np.argmax(np.abs(F[c:, c])))
            piv[c] = p
            if not (abs(F[p, c]) > 0.0) and info == 0:
                info = c + 1
            if p != c:
                F[[c, p], j0:] = F[[p, c], j0:]
            inv = 1.0 / F[c, c] if F[c, c] != 0.0 else 0.0
            F[c + 1:, c] *= inv
            F[c + 1:, c + 1:j1] -= np.outer(F[c + 1:, c], F[c, c + 1:j1])
        if j1 < n:
            L11 = np.tril(F[j0:j1, j0:j1], -1) + np.eye(j1 - j0)
            F[j0:j1, j1:] = np.linalg.solve(L11, F[j0:j1, j1:])
            F[j1:, j1:] -= F[j1:, j0:j1] @ F[j0:j1, j1:]
    return F, piv, info


def split_lu(F):
    n = F.shape[0]
    return np.tril(F, -1) + np.eye(n), np.triu(F)


# ---------------------------------------------------------------------------------------------------- errors
def backward_error(A, x, b) -> float:
    """eta = ||b - A x||_inf / (||A||_inf ||x||_inf + ||b||_inf) per right-hand side (max over columns), with the
    residual accumulated in np.longdouble."""
    A = np.asarray(A)
    x = np.asarray(x).reshape(A.shape[1], -1)
    b = np.asarray(b).reshape(A.shape[0], -1)
    r = b.astype(np.longdouble) - A.astype(np.longdouble) @ x.astype(np.longdouble)
    num = np.abs(r).max(axis=0).astype(np.float64)
    den = np.abs(A).sum(axis=1).max() * np.abs(x).max(axis=0) + np.abs(b).max(axis=0)
    return float((num / np.where(den > 0.0, den, 1.0)).max())  # x = b = 0: zero residual


def pivot_margins(lu_lapack) -> np.ndarray:
    """Per step j of LAPACK's partial pivoting: 1 - max_{i > j} |L_ij|, the relative gap between the chosen pivot and
    the largest other candidate of the column (the candidates are L_ij U_jj).  A margin near zero is a near-tie that
    another summation order may resolve the other way."""
    n = lu_lapack.shape[0]
    L = np.abs(np.tril(lu_lapack, -1))
    m = np.ones(n)
    if n > 1:
        m[:-1] = 1.0 - L[:, :-1].max(axis=0)
    return m


# ---------------------------------------------------------------------------------------------------- families
def planted(n: int, perm="random", rng=None, singular_col: int | None = None):
    """Planted dyadic LU.  perm: "identity", "reversed", "random" or an explicit permutation (row i of P A = row
    perm[i] of A).  singular_col = c: U's row c and L's column c below the diagonal are zero, so that partial pivoting
    keeps row c as the pivot of column c, stores zero multipliers and reports column c (use with the identity).
    Returns dict(A, L, U, ipiv, x) with P A = L U exactly."""
    rng = np.random.default_rng(rng)
    if isinstance(perm, str):
        perm = {"identity": np.arange(n), "reversed": np.arange(n)[::-1], "random": rng.permutation(n)}[perm]
    perm = np.asarray(perm)
    L = np.tril(rng.integers(-4, 5, size=(n, n)) / 8.0, -1) + np.eye(n)
    U = np.triu(rng.integers(-8, 9, size=(n, n)) / 4.0, 1)
    U[np.diag_indices(n)] = rng.choice([-2.0, -1.0, 1.0, 2.0], size=n)
    if singular_col is not None:
        U[singular_col, :] = 0.0
        L[singular_col + 1:, singular_col] = 0.0
    A = np.empty((n, n))
    A[perm] = L @ U  # exact: every sum is a multiple of 1/32 far below 2^53
    x = rng.integers(-8, 9, size=n) / 4.0
    return dict(A=A, L=L, U=U, ipiv=perm_to_ipiv(perm), x=x)


def planted_rhs(A, nrhs: int, rng=None):
    """Dyadic solutions X (n x nrhs, multiples of 1/4) and B = A X, exact."""
    rng = np.random.default_rng(rng)
    X = rng.integers(-8, 9, size=(A.shape[0], nrhs)) / 4.0
    return X, A @ X


def gaussian(n: int, rng=None):
    return np.random.default_rng(rng).standard_normal((n, n))


def saddle_split(n: int) -> int:
    """Variable slots of an n-square saddle-point block, in the proportion of the kinodynamic stage block."""
    return max(1, min(n - 1, round(n * SADDLE_NX / SADDLE_N))) if n > 1 else 1


def saddle(n: int, rng=None, delta: float = SADDLE_DELTA, delta_c: float = SADDLE_DELTA_C):
    """[[H + delta I, J^T], [J, -delta_c I]] with H symmetric: the shape of a KKT stage block.  The pivots of the
    J columns come from rows far below the diagonal."""
    rng = np.random.default_rng(rng)
    if n == 1:
        return np.array([[rng.standard_normal() + delta]])
    nx = saddle_split(n)
    me = n - nx
    H = rng.standard_normal((nx, nx))
    H = 0.5 * (H + H.T)
    J = rng.standard_normal((me, nx))
    K = np.zeros((n, n))
    K[:nx, :nx] = H + delta * np.eye(nx)
    K[:nx, nx:] = J.T
    K[nx:, :nx] = J
    K[nx:, nx:] = -delta_c * np.eye(me)
    return K


def diag_dominant(n: int, rng=None):
    """Column-wise strictly diagonally dominant: partial pivoting keeps every diagonal pivot."""
    rng = np.random.default_rng(rng)
    A = rng.uniform(-1.0, 1.0, size=(n, n))
    A[np.diag_indices(n)] = (np.abs(A).sum(axis=0) + 1.0) * rng.choice([-1.0, 1.0], size=n)
    return A


# ---------------------------------------------------------------------------------------------------- dispatch
def expected_plan(n: int, batch: int, nrhs: int, sms: int) -> tuple[int, int, int, int]:
    """(RPT, MB, ct, column chunks) hb_debug_lu_plan should report, restated from the kernels' limits:
    RPT = ceil(n / 256) panel rows per thread; MB = 2 when the batch exceeds one CTA per SM and two factor CTAs fit
    an SM (2 (lu_factor_smem + 2048) <= 227 KB: n <= 436); the staged solve runs 32 right-hand sides per CTA at two
    CTAs per SM up to n = 352, 24 at two CTAs per SM up to 442, 32 at one CTA per SM up to 715 and 24 above."""
    rpt = 1 if n <= 256 else 2 if n <= 512 else 3
    mb = 2 if batch > sms and n <= 436 else 1
    ct = 4 if n <= 352 else 3 if n <= 442 else 4 if n <= 715 else 3
    return rpt, mb, ct, -(-nrhs // (8 * ct))
