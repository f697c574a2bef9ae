"""Stage-wise solve of the primal-dual Newton (KKT) system of a multiple-shooting OCP (SURVEY.md 8(f), row f2).

The step on the other side of the evaluation path: IPOPT hands `jac_g` / `hess_l` to a sparse symmetric
indefinite solver (MUMPS [ext]) once per iteration.  For the problems of this repository the matrix

        K = [ W + J_I^T Sigma J_I + delta I      J_E^T   ]        W   block diagonal per knot (hess_l)
            [ J_E                             -delta_c I ]        J_I rows local to one knot
                                                                  J_E rows touch knot k, or knots k-1 and k
                                                                      (integrator defects)

is block tridiagonal once unknowns are ordered by stage, u_k = (dx_k, dlam_E,k): the only coupling between
stage k-1 and stage k are the defect rows of stage k acting on dx_{k-1}.  The solve is a block LU sweep
over the stages (Riccati-like), batched over instances: per stage one dense LU of an
(n_k + m_E,k)-square block and one solve with the ~87 coupling columns -- O(N) blocks instead of one
(n_x + m_E)-square factorisation.  With linalg="hb" (CUDA only, no fallback) every stage is assembled by
one kernel (csrc/kkt_assemble.cu) and factored and solved by this library's batched LU kernels (csrc/lu.cu
through `lu_factor` / `lu_solve`); linalg="torch", the comparison baseline and what the CPU-side structural
tests use, assembles the stages with torch indexing and solves them with torch.linalg.  What this module
owns is the structure: the assignment of rows to
stages and the gather maps from the CCS value arrays the kernels write to the dense stage blocks.

Checked against a dense solve of the same system (tests/test_kkt_cpu.py on random values in the real
pattern, tests/test_gpu_kkt.py on evaluated values).  Periodicity rows (knot 0 with knot N-1) make
the matrix cyclic: they are kept as a border of the block-tridiagonal part and eliminated with a Schur
complement (one sweep with 1 + 84 right-hand sides).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _capi


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def lu_factor(A: torch.Tensor, symmetric: bool = False):
    """Batched LU with partial pivoting of A (B, n, n) on the GPU (csrc/lu.cu through the C ABI).
    Returns (factors, piv, info); `factors` is only meaningful to ``lu_solve``.  symmetric=True skips the
    transposition to the kernel's column-major storage (and factors A in place)."""
    if not A.is_cuda or A.dtype != torch.float64 or A.dim() != 3 or A.shape[1] != A.shape[2]:
        raise ValueError("lu_factor needs a (B, n, n) float64 CUDA tensor")
    B, n = A.shape[0], A.shape[1]
    F = A if (symmetric and A.is_contiguous()) else (A.contiguous() if symmetric else A.transpose(1, 2).contiguous())
    piv = torch.empty((B, n), dtype=torch.int32, device=A.device)
    info = torch.empty((B,), dtype=torch.int32, device=A.device)
    st = torch.cuda.current_stream(A.device).cuda_stream
    _capi.check(_capi.lib().hb_lu_factor_batched(_ptr(F), _ptr(piv), _ptr(info), n, B, ctypes.c_void_p(st)),
                "hb_lu_factor_batched")
    return F, piv, info


def lu_solve(F: torch.Tensor, piv: torch.Tensor, rhs: torch.Tensor, inplace: bool = False) -> torch.Tensor:
    """Solve with the factors of ``lu_factor``; rhs (B, n, r) -> solution (B, n, r) (a new tensor, or `rhs` itself
    with inplace=True, which needs it contiguous)."""
    if rhs.dim() != 3 or rhs.shape[0] != F.shape[0] or rhs.shape[1] != F.shape[1] or not rhs.is_cuda:
        raise ValueError("lu_solve needs a (B, n, r) CUDA right-hand side matching the factors")
    if inplace and not rhs.is_contiguous():
        raise ValueError("lu_solve(inplace=True) needs a contiguous right-hand side")
    X = rhs if inplace else rhs.contiguous().clone()
    st = torch.cuda.current_stream(F.device).cuda_stream
    _capi.check(_capi.lib().hb_lu_solve_batched(_ptr(F), _ptr(piv), _ptr(X), F.shape[1], X.shape[2], F.shape[0],
                                                ctypes.c_void_p(st)), "hb_lu_solve_batched")
    return X


class StageKKT:
    def __init__(self, n_x: int, m: int, horizon: int, knot_size: int, jac_colind, jac_row, hess_colind, hess_row,
                 eq_rows, ine_rows, device="cpu", linalg: str = "hb", max_border: int = 128):
        """eq_rows / ine_rows: sorted global row indices of the equality / inequality constraints (the
        ordering of the multiplier vectors handed to ``solve``).  Variables beyond horizon*knot_size
        (initial-state decision variables) join stage 0.

        linalg: "hb" = the batched LU kernels of this library (CUDA tensors only, no fallback);
        "torch" = torch.linalg (cuSOLVER on the GPU, LAPACK on the CPU): the comparison baseline, and what
        the CPU-side structural tests use."""
        if linalg not in ("hb", "torch"):
            raise ValueError("linalg must be 'hb' or 'torch'")
        self.linalg = linalg
        self.n_x, self.m, self.N, self.nz = n_x, m, horizon, knot_size
        self.device = torch.device(device)
        N, nz = horizon, knot_size
        n_extra = n_x - N * nz
        if n_extra < 0:
            raise ValueError("n_x is smaller than horizon * knot_size")
        self.nx = nx = nz + n_extra  # local variable slots of a stage (the extras are padding for k > 0)
        jac_colind, jac_row = np.asarray(jac_colind), np.asarray(jac_row)
        hess_colind, hess_row = np.asarray(hess_colind), np.asarray(hess_row)
        eq_rows, ine_rows = np.asarray(eq_rows, dtype=np.int64), np.asarray(ine_rows, dtype=np.int64)
        self.mE, self.mI = len(eq_rows), len(ine_rows)

        def stage_of(c):
            return np.where(c < N * nz, c // nz, 0)

        def local_of(c):
            return np.where(c < N * nz, c % nz, nz + (c - N * nz))

        jcol = np.repeat(np.arange(n_x), np.diff(jac_colind))
        jst = stage_of(jcol)
        hi = np.full(m, -1)
        lo = np.full(m, N + 1)
        np.maximum.at(hi, jac_row, jst)
        np.minimum.at(lo, jac_row, jst)
        live = hi >= 0  # rows with an empty Jacobian (parameter-only rows) take no part in the Newton system
        # rows that couple non-adjacent knots (periodicity: knot 0 with knot N-1) make the matrix cyclic; they
        # are kept out of the stages and handled as a BORDER: K = [[K_bt, P^T], [P, -delta_c I]], solved with
        # one block-tridiagonal sweep over 1 + n_border right-hand sides and a small Schur complement
        far = live & ((hi - lo) > 1)
        if np.any(far[ine_rows]):
            raise NotImplementedError("an inequality row couples non-adjacent knots")
        if np.any((hi - lo)[ine_rows][live[ine_rows]] > 0):
            raise NotImplementedError("an inequality row couples two knots")
        if far.sum() > max_border:
            raise NotImplementedError(f"{int(far.sum())} constraint rows couple non-adjacent knots (limit {max_border})")
        hi = np.where(far, -2, hi)  # not in any stage
        hcol = np.repeat(np.arange(n_x), np.diff(hess_colind))
        if np.any(stage_of(hcol) != stage_of(hess_row)):
            raise NotImplementedError("hess_l couples two knots")

        # ---- rows -> stages
        is_eq = np.zeros(m, dtype=bool)
        is_eq[eq_rows] = True
        pos_E = np.full(m, -1)
        pos_E[eq_rows] = np.arange(self.mE)
        pos_I = np.full(m, -1)
        pos_I[ine_rows] = np.arange(self.mI)
        self.eq_stage_rows, self.ine_stage_rows, self.cpl_local = [], [], []
        for k in range(N):
            e = eq_rows[(hi[eq_rows] == k)]
            i = ine_rows[(hi[ine_rows] == k)]
            self.eq_stage_rows.append(e)
            self.ine_stage_rows.append(i)
            self.cpl_local.append(np.nonzero(lo[e] < k)[0])  # positions (inside the stage's eq rows) of the defect rows
        self.dead_eq = pos_E[eq_rows[~live[eq_rows]]]  # multipliers of empty rows: left at zero
        border = eq_rows[far[eq_rows]]
        self.n_border = len(border)
        self.mEk = max(len(e) for e in self.eq_stage_rows)
        self.mIk = max(max(len(i) for i in self.ine_stage_rows), 1)
        self.mCk = max(max(len(c) for c in self.cpl_local), 1)
        self.nb = nb = nx + self.mEk
        row_stage = hi
        loc_E = np.full(m, -1)
        loc_I = np.full(m, -1)
        for k in range(N):
            loc_E[self.eq_stage_rows[k]] = np.arange(len(self.eq_stage_rows[k]))
            loc_I[self.ine_stage_rows[k]] = np.arange(len(self.ine_stage_rows[k]))
        loc_C = np.full(m, -1)
        for k in range(N):
            loc_C[self.eq_stage_rows[k][self.cpl_local[k]]] = np.arange(len(self.cpl_local[k]))

        dev = self.device

        def t(a):
            return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.long, device=dev)

        # ---- gather maps: for every stage, (value index, flat position in the dense block)
        self.maps = []
        hst = stage_of(hcol)
        hr_l, hc_l = local_of(hess_row), local_of(hcol)
        jc_l = local_of(jcol)
        for k in range(N):
            sel = np.nonzero(hst == k)[0]
            w_idx, w_pos, w_pos_t = sel, hr_l[sel] * nb + hc_l[sel], hc_l[sel] * nb + hr_l[sel]
            # equality rows of this stage, columns of this stage -> C (rows nx + loc_E) and its transpose
            je = np.nonzero(is_eq[jac_row] & (row_stage[jac_row] == k) & (jst == k))[0]
            c_pos = (nx + loc_E[jac_row[je]]) * nb + jc_l[je]
            c_pos_t = jc_l[je] * nb + (nx + loc_E[jac_row[je]])
            # equality rows of this stage, columns of stage k-1 -> A (mCk x nx)
            ja = np.nonzero(is_eq[jac_row] & (row_stage[jac_row] == k) & (jst == k - 1))[0] if k > 0 else np.zeros(0, int)
            a_pos = loc_C[jac_row[ja]] * nx + jc_l[ja]
            # inequality rows -> J_I (mIk x nx)
            ji = np.nonzero((~is_eq[jac_row]) & (pos_I[jac_row] >= 0) & (row_stage[jac_row] == k))[0]
            i_pos = loc_I[jac_row[ji]] * nx + jc_l[ji]
            var = (np.arange(nz) + k * nz) if k > 0 else np.concatenate([np.arange(nz), N * nz + np.arange(n_extra)])
            self.maps.append({
                "w_idx": t(w_idx), "w_pos": t(w_pos), "w_pos_t": t(w_pos_t),
                "c_idx": t(je), "c_pos": t(c_pos), "c_pos_t": t(c_pos_t),
                "a_idx": t(ja), "a_pos": t(a_pos),
                "i_idx": t(ji), "i_pos": t(i_pos),
                "var": t(var), "n_var": len(var),
                "eq": t(pos_E[self.eq_stage_rows[k]]), "n_eq": len(self.eq_stage_rows[k]),
                "ine": t(pos_I[self.ine_stage_rows[k]]), "n_ine": len(self.ine_stage_rows[k]),
                "cpl": t(nx + self.cpl_local[k]), "n_cpl": len(self.cpl_local[k]),
            })
        # ---- border rows: nnz index, local border row, global column; positions in the multiplier vector
        loc_B = np.full(m, -1)
        loc_B[border] = np.arange(self.n_border)
        jb = np.nonzero(far[jac_row] & is_eq[jac_row])[0]
        self.border = {"idx": t(jb), "row": t(loc_B[jac_row[jb]]), "col": t(jcol[jb]), "eq": t(pos_E[border])}
        # ---- tables of the fused assembly kernel (hb_kkt_assemble_stage), in the order include/hippopt_b200.h lists.
        # The fused sweep sizes every stage block by ITS variables and equality rows (nb_k = n_var_k + n_eq_k) instead
        # of the padded maximum: with a final-state constraint the last stage has 81 more rows than the others
        # (config 4: 418 against 331), and a padded block costs (418 / 331)^3 = 2 x the factorisation on 29 of 30 stages.
        self._stage_np = []
        self.stage_nx = [len(mp_["var"]) for mp_ in self.maps]
        self.stage_nb = [self.stage_nx[k] + len(self.eq_stage_rows[k]) for k in range(N)]
        for k in range(N):
            nxk, nbk = self.stage_nx[k], self.stage_nb[k]
            sel = np.nonzero(hst == k)[0]
            je = np.nonzero(is_eq[jac_row] & (row_stage[jac_row] == k) & (jst == k))[0]
            direct_val = np.concatenate([sel, sel, ~je, ~je])
            direct_pos = np.concatenate([hr_l[sel] * nbk + hc_l[sel], hc_l[sel] * nbk + hr_l[sel],
                                         (nxk + loc_E[jac_row[je]]) * nbk + jc_l[je], jc_l[je] * nbk + (nxk + loc_E[jac_row[je]])])
            if len(sel) and max(hr_l[sel].max(), hc_l[sel].max()) >= nxk or len(je) and jc_l[je].max() >= nxk:
                raise AssertionError("a stage references a variable slot beyond its own variables")
            # J_I^T Sigma J_I: ordered pairs of the entries of every inequality row, grouped by destination
            ji = np.nonzero((~is_eq[jac_row]) & (pos_I[jac_row] >= 0) & (row_stage[jac_row] == k))[0]
            by_row: dict[int, list] = {}
            for e in ji:
                by_row.setdefault(int(jac_row[e]), []).append(int(e))
            contrib: dict[int, list] = {}
            for r in sorted(by_row):
                for e1 in by_row[r]:
                    for e2 in by_row[r]:
                        contrib.setdefault(int(jc_l[e1]) * nbk + int(jc_l[e2]), []).append((int(pos_I[r]), e1, e2))
            tgt_pos = np.asarray(sorted(contrib), dtype=np.int64)
            tgt_ptr = np.zeros(len(tgt_pos) + 1, dtype=np.int64)
            flat = []
            for i, pos in enumerate(tgt_pos):
                flat += contrib[int(pos)]
                tgt_ptr[i + 1] = len(flat)
            flat = np.asarray(flat, dtype=np.int64).reshape(-1, 3)

            def coupling_rows(kk):  # (row inside the coupling rows of stage kk, jac_vals index, variable slot of stage kk-1)
                if kk <= 0 or kk >= N:
                    return np.zeros((0, 3), dtype=np.int64)
                ja = np.nonzero(is_eq[jac_row] & (row_stage[jac_row] == kk) & (jst == kk - 1))[0]
                out = np.stack([loc_C[jac_row[ja]], ja, jc_l[ja]], axis=1)
                return out[np.lexsort((out[:, 2], out[:, 0]))]

            a = coupling_rows(k)
            n_cpl = len(self.cpl_local[k])
            a_ptr = np.zeros(n_cpl + 1, dtype=np.int64)
            np.add.at(a_ptr, a[:, 0] + 1, 1)
            a_ptr = np.cumsum(a_ptr)
            an = coupling_rows(k + 1)
            var = self.maps[k]["var"].cpu().numpy()
            eqk = pos_E[self.eq_stage_rows[k]]
            tables = [direct_val, direct_pos, tgt_pos, tgt_ptr, flat[:, 0], flat[:, 1], flat[:, 2], var, eqk,
                      nxk + self.cpl_local[k], a_ptr, a[:, 1], a[:, 2], an[:, 1], an[:, 0], an[:, 2]]
            hdr = [nbk, nxk, len(var), len(eqk), 0, n_cpl, len(self.cpl_local[k + 1]) if k + 1 < N else 0, len(direct_val),
                   len(tgt_pos), len(flat), len(a), len(an), self.stage_nb[k - 1] if k > 0 else 0]
            self._stage_np.append((hdr, np.concatenate([np.asarray(t, dtype=np.int64).ravel() for t in tables]).astype(np.int32)))
        self._stage_dev = None

    @classmethod
    def for_evaluator(cls, ev, lbg, ubg, device="cpu", linalg: str = "hb"):
        """Kinodynamic evaluator (KinoEvaluator) + one instance's bounds -> solver and the (eq, ine) row lists."""
        lbg, ubg = np.asarray(lbg, dtype=np.float64).ravel(), np.asarray(ubg, dtype=np.float64).ravel()
        eq = np.nonzero(lbg == ubg)[0]
        ine = np.nonzero((lbg != ubg) & ~(np.isinf(lbg) & np.isinf(ubg)))[0]
        jc, jr = ev.jac_sparsity()
        hc, hr = ev.hess_sparsity()
        lay = ev.layout
        if not hasattr(lay, "knot_size"):
            raise ValueError(f"{type(ev).__name__} has no multiple-shooting stage structure (layout.knot_size)")
        return cls(ev.n_x, ev.m, lay.N, lay.knot_size, jc, jr, hc, hr, eq, ine, device=device, linalg=linalg), eq, ine

    # ------------------------------------------------------------------ solve
    def solve(self, hess_vals, jac_vals, sigma_I, delta, delta_c, rhs_x, rhs_E, chunk: int | None = None):
        """Solve K [dx; dlam_E] = [rhs_x; rhs_E] for every instance.

        hess_vals (B, nnz_h), jac_vals (B, nnz_j): CCS value arrays as written by hb_eval;
        sigma_I (B, m_I) >= 0: barrier diagonal of the inequality rows; delta (B,): Hessian shift;
        delta_c: scalar >= 0 on the (2,2) block.  Returns dx (B, n_x), dlam_E (B, m_E).
        Instances are processed `chunk` at a time: the forward sweep keeps, per stage, the substituted
        right-hand sides and the nb x 87 coupling solve for the back substitution (chunk * N * nb * 88 * 8
        bytes, 1.8 GB for 256 instances of the 30-knot problem); the factors themselves live for one stage.

        Border rows (periodicity): K = [[K_bt, P^T], [P, -delta_c I]].  One sweep solves K_bt [y0 | Y] =
        [rhs | P^T] (1 + n_border right-hand sides), then (-delta_c I - P Y) lam_p = rhs_p - P y0 and
        u = y0 - Y lam_p."""
        B = hess_vals.shape[0]
        if chunk is None:  # one CTA per stage block: whole waves of the factor kernel (1 CTA per SM)
            chunk = 2 * torch.cuda.get_device_properties(hess_vals.device).multi_processor_count if hess_vals.is_cuda else 256
        if B > chunk:
            parts = [self.solve(hess_vals[i:i + chunk], jac_vals[i:i + chunk], sigma_I[i:i + chunk], delta[i:i + chunk],
                                delta_c, rhs_x[i:i + chunk], rhs_E[i:i + chunk], chunk) for i in range(0, B, chunk)]
            return torch.cat([a for a, _ in parts]), torch.cat([b for _, b in parts])
        nbr = self.n_border
        multi = rhs_x.dim() == 3  # (B, n_x, R) / (B, m_E, R): several right-hand sides (L-BFGS low-rank correction)
        if not multi:
            rhs_x, rhs_E = rhs_x[:, :, None], rhs_E[:, :, None]
        R0 = rhs_x.shape[2]
        if nbr == 0:
            DX, DL = self._sweep(hess_vals, jac_vals, sigma_I, delta, delta_c, rhs_x, rhs_E)
            return (DX, DL) if multi else (DX[:, :, 0], DL[:, :, 0])
        dev, dt = hess_vals.device, hess_vals.dtype
        bd = self.border
        pv = jac_vals[:, bd["idx"]]  # (B, nnz of P)
        RX = torch.zeros((B, self.n_x, R0 + nbr), dtype=dt, device=dev)
        RX[:, :, :R0] = rhs_x
        RX[:, bd["col"], R0 + bd["row"]] = pv  # P^T
        RE = torch.zeros((B, self.mE, R0 + nbr), dtype=dt, device=dev)
        RE[:, :, :R0] = rhs_E
        RE[:, bd["eq"], :R0] = 0.0  # border rows are not part of K_bt
        DX, DL = self._sweep(hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE)
        # P X for X = [y0 | Y] (dx part only: P has no multiplier columns).  Every border row has one entry per
        # side (x_0 term, x_{N-1} term): at most two additions per element, order-independent
        PX = torch.zeros((B, nbr, R0 + nbr), dtype=dt, device=dev)
        PX.index_add_(1, bd["row"], pv[:, :, None] * DX[:, bd["col"], :])
        S = -PX[:, :, R0:] - delta_c * torch.eye(nbr, dtype=dt, device=dev)
        # small (n_border^2) library solve; a singular / non-finite Schur complement (a stage block that failed
        # to factor) gives NaN for that instance, which the caller treats like any failed solve
        S = torch.where(torch.isfinite(S), S, torch.zeros_like(S))
        lam_p, info = torch.linalg.solve_ex(S, rhs_E[:, bd["eq"], :] - PX[:, :, :R0], check_errors=False)
        bad = (info != 0) | ~torch.isfinite(PX).all(dim=2).all(dim=1)
        lam_p = torch.where(bad[:, None, None], torch.full_like(lam_p, float("nan")), lam_p)
        dx = DX[:, :, :R0] - torch.bmm(DX[:, :, R0:], lam_p)
        dl = DL[:, :, :R0] - torch.bmm(DL[:, :, R0:], lam_p)
        dl[:, bd["eq"], :] = lam_p
        return (dx, dl) if multi else (dx[:, :, 0], dl[:, :, 0])

    def _sweep(self, hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE):
        """Block-tridiagonal part: K_bt [DX; DL] = [RX; RE] for R right-hand sides (B, n_x | m_E, R)."""
        if self.linalg == "hb":
            if not hess_vals.is_cuda:
                raise ValueError("linalg='hb' runs on CUDA tensors only")
            return self._sweep_fused(hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE)
        B, R = hess_vals.shape[0], RX.shape[2]
        dev, dt = hess_vals.device, hess_vals.dtype
        nx, nb, N = self.nx, self.nb, self.N
        DX = torch.zeros((B, self.n_x, R), dtype=dt, device=dev)
        DL = torch.zeros((B, self.mE, R), dtype=dt, device=dev)
        Wv, Zs = [], []
        w_prev = None
        A = Z = None
        for k in range(N):
            mp = self.maps[k]
            D, b = self._assemble(k, hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE)
            Zs.append(Z)
            if Z is not None:  # Z = S_{k-1}^{-1} [A_k^T; 0] came out of the previous stage's solve
                cp = mp["cpl"]
                D[:, cp[:, None], cp[None, :]] -= torch.bmm(A, Z[:, :nx, :])
                b[:, cp, :] -= torch.bmm(A, w_prev[:, :nx, :])
            fac = torch.linalg.lu_factor_ex(D)[:2]
            # one solve per stage: the stage's right-hand sides and the coupling columns of the next stage
            if k + 1 < N and self.maps[k + 1]["n_cpl"]:
                A = self._coupling(k + 1, jac_vals)
                rhs = torch.zeros((B, nb, R + A.shape[1]), dtype=dt, device=dev)
                rhs[:, :, :R] = b
                rhs[:, :nx, R:] = A.transpose(1, 2)
                sol = torch.linalg.lu_solve(*fac, rhs)
                w_prev, Z = sol[:, :, :R], sol[:, :, R:]
            else:
                A = Z = None
                w_prev = torch.linalg.lu_solve(*fac, b)
            Wv.append(w_prev)
        u_next = None
        for k in range(N - 1, -1, -1):
            mp = self.maps[k]
            u = Wv[k]
            if k < N - 1 and Zs[k + 1] is not None:
                u = u - torch.bmm(Zs[k + 1], u_next[:, self.maps[k + 1]["cpl"], :])
            DX[:, mp["var"], :] = u[:, :mp["n_var"], :]
            DL[:, mp["eq"], :] = u[:, nx:nx + mp["n_eq"], :]
            u_next = u
        return DX, DL

    def _sweep_fused(self, hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE):
        """The sweep of `_sweep` with every stage assembled by ONE kernel (csrc/kkt_assemble.cu): block, right-hand
        sides, J_I^T Sigma J_I and the coupling terms come straight from the CCS value arrays; the stage's solution
        [w | Z] (B, nb, R + n_cpl_next) is the next stage's input and is kept for the back substitution."""
        B, R = hess_vals.shape[0], RX.shape[2]
        dev, dt = hess_vals.device, hess_vals.dtype
        nx, nb, N = self.nx, self.nb, self.N
        if self._stage_dev is None or self._stage_dev[0] != dev:
            self._stage_dev = (dev, [torch.as_tensor(tab, device=dev) for _, tab in self._stage_np])
        L = _capi.lib()
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        hv, jv, sg, dl = hess_vals.contiguous(), jac_vals.contiguous(), sigma_I.contiguous(), delta.contiguous()
        rx, re = RX.contiguous(), RE.contiguous()
        sols, prev = [], None
        for k in range(N):
            hdr, _ = self._stage_np[k]
            hdr = list(hdr)
            hdr[4] = R
            nbk = hdr[0]
            D = torch.empty((B, nbk, nbk), dtype=dt, device=dev)
            rhs = torch.empty((B, nbk, R + hdr[6]), dtype=dt, device=dev)
            _capi.check(L.hb_kkt_assemble_stage((ctypes.c_int32 * len(hdr))(*hdr), _ptr(self._stage_dev[1][k]), _ptr(hv),
                                                hv.shape[1], _ptr(jv), jv.shape[1], _ptr(sg), max(sg.shape[1], 1), _ptr(dl),
                                                float(delta_c), _ptr(rx), self.n_x, _ptr(re), self.mE,
                                                _ptr(prev) if (prev is not None and hdr[5]) else None, _ptr(D), _ptr(rhs), B, st),
                        "hb_kkt_assemble_stage")
            F, piv, _ = lu_factor(D, symmetric=True)  # in place
            prev = lu_solve(F, piv, rhs, inplace=True)
            sols.append(prev)
        DX = torch.zeros((B, self.n_x, R), dtype=dt, device=dev)
        DL = torch.zeros((B, self.mE, R), dtype=dt, device=dev)
        u_next = None
        for k in range(N - 1, -1, -1):
            mp = self.maps[k]
            nxk = self.stage_nx[k]
            u = sols[k][:, :, :R]
            if k < N - 1 and self.maps[k + 1]["n_cpl"]:
                nxn = self.stage_nx[k + 1]
                cp_next = u_next[:, nxn + self._cpl_local_dev(k + 1, dev), :]
                u = u - torch.bmm(sols[k][:, :, R:], cp_next)
            DX[:, mp["var"], :] = u[:, :nxk, :]
            DL[:, mp["eq"], :] = u[:, nxk:nxk + mp["n_eq"], :]
            u_next = u
        return DX, DL

    def _cpl_local_dev(self, k, dev):
        cache = self.__dict__.setdefault("_cpl_dev", {})
        key = (k, str(dev))
        if key not in cache:
            cache[key] = torch.as_tensor(np.ascontiguousarray(self.cpl_local[k]), dtype=torch.long, device=dev)
        return cache[key]

    # ------------------------------------------------------------------ torch assembly of a stage
    def _assemble(self, k, hess_vals, jac_vals, sigma_I, delta, delta_c, RX, RE):
        """Stage block D_k (B, nb, nb) and right-hand sides b_k (B, nb, R) without the coupling terms."""
        B, R = hess_vals.shape[0], RX.shape[2]
        dev, dt = hess_vals.device, hess_vals.dtype
        nx, nb = self.nx, self.nb
        mp = self.maps[k]
        D = torch.zeros((B, nb * nb), dtype=dt, device=dev)
        D[:, mp["w_pos"]] = hess_vals[:, mp["w_idx"]]
        D[:, mp["w_pos_t"]] = hess_vals[:, mp["w_idx"]]
        D[:, mp["c_pos"]] = jac_vals[:, mp["c_idx"]]
        D[:, mp["c_pos_t"]] = jac_vals[:, mp["c_idx"]]
        D = D.view(B, nb, nb)
        nv, ne = mp["n_var"], mp["n_eq"]
        if mp["n_ine"]:
            JI = torch.zeros((B, self.mIk * nx), dtype=dt, device=dev)
            JI[:, mp["i_pos"]] = jac_vals[:, mp["i_idx"]]
            JI = JI.view(B, self.mIk, nx)
            sg = torch.zeros((B, self.mIk), dtype=dt, device=dev)
            sg[:, :mp["n_ine"]] = sigma_I[:, mp["ine"]]
            D[:, :nx, :nx] += torch.einsum("bin,bi,bik->bnk", JI, sg, JI)
        idx = torch.arange(nb, device=dev)
        diag = torch.zeros((B, nb), dtype=dt, device=dev)
        diag[:, :nv] = delta[:, None]
        diag[:, nv:nx] = 1.0             # padding variable slots
        diag[:, nx:nx + ne] = -delta_c
        diag[:, nx + ne:] = 1.0          # padding multiplier slots
        D[:, idx, idx] += diag
        b = torch.zeros((B, nb, R), dtype=dt, device=dev)
        b[:, :nv, :] = RX[:, mp["var"], :]
        b[:, nx:nx + ne, :] = RE[:, mp["eq"], :]
        return D, b

    def _coupling(self, k, jac_vals):
        """A_k (B, n_cpl, nx): the coupling rows of stage k with respect to the variable slots of stage k - 1."""
        mq = self.maps[k]
        B = jac_vals.shape[0]
        Ak = torch.zeros((B, self.mCk * self.nx), dtype=jac_vals.dtype, device=jac_vals.device)
        Ak[:, mq["a_pos"]] = jac_vals[:, mq["a_idx"]]
        return Ak.view(B, self.mCk, self.nx)[:, :mq["n_cpl"], :]

    # ------------------------------------------------------------------ reference: the same matrix, dense
    def dense_matrix(self, hess_vals, jac_vals, sigma_I, delta, delta_c, eq_rows, ine_rows, jac_colind, jac_row,
                     hess_colind, hess_row):
        """(B, n_x + m_E, n_x + m_E) dense K for small problems (test oracle of ``solve``)."""
        B = hess_vals.shape[0]
        dev, dt = hess_vals.device, hess_vals.dtype
        n, mE = self.n_x, self.mE
        jcol = torch.as_tensor(np.repeat(np.arange(n), np.diff(np.asarray(jac_colind))), device=dev)
        jrow = torch.as_tensor(np.asarray(jac_row), dtype=torch.long, device=dev)
        hcol = torch.as_tensor(np.repeat(np.arange(n), np.diff(np.asarray(hess_colind))), device=dev)
        hrow = torch.as_tensor(np.asarray(hess_row), dtype=torch.long, device=dev)
        J = torch.zeros((B, self.m, n), dtype=dt, device=dev)
        J[:, jrow, jcol] = jac_vals
        W = torch.zeros((B, n, n), dtype=dt, device=dev)
        W[:, hrow, hcol] = hess_vals
        W[:, hcol, hrow] = hess_vals
        eq_t = torch.as_tensor(np.asarray(eq_rows), dtype=torch.long, device=dev)
        in_t = torch.as_tensor(np.asarray(ine_rows), dtype=torch.long, device=dev)
        JE, JI = J[:, eq_t, :], J[:, in_t, :]
        K = torch.zeros((B, n + mE, n + mE), dtype=dt, device=dev)
        K[:, :n, :n] = W + torch.einsum("bin,bi,bik->bnk", JI, sigma_I, JI) + delta[:, None, None] * torch.eye(n, dtype=dt, device=dev)
        K[:, :n, n:] = JE.transpose(1, 2)
        K[:, n:, :n] = JE
        K[:, n:, n:] = -delta_c * torch.eye(mE, dtype=dt, device=dev)
        return K
