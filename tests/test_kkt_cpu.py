"""Stage-wise KKT solve (SURVEY.md 8(f) f2) against a dense solve of the same matrix, on the CPU:
random values in the REAL sparsity patterns of the kinodynamic OCP (layout compiler), so the row -> stage
assignment, the gather maps and the block recursion are all exercised without a GPU."""
import numpy as np
import pytest
import torch

from hippopt_b200.kino_layout import KinoLayout, KinoSettings
from hippopt_b200.kkt import StageKKT
from hippopt_b200.workloads import kino_parameters


def _setup(model, N, final, periodic=False):
    lay = KinoLayout(model, KinoSettings(horizon=N, final_state_constraint=final, periodicity_constraint=periodic))
    p = kino_parameters(lay, model, 1, np.random.default_rng(0))
    lb, ub = lay.bounds(p)
    eq = np.nonzero(lb[0] == ub[0])[0]
    ine = np.nonzero(lb[0] != ub[0])[0]
    kkt = StageKKT(lay.n_x, lay.m, N, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine,
                   linalg="torch")  # LAPACK block algebra: this test is about the structure, on the CPU
    return lay, kkt, eq, ine


@pytest.mark.parametrize("N,final,periodic", [(2, False, False), (4, False, False), (3, True, False), (3, False, True),
                                              (4, True, True), (2, True, True)])
def test_stage_solve_matches_dense(model, N, final, periodic):
    """periodic: the 84 periodicity rows couple knot 0 with knot N-1 (config 4): border + Schur complement for
    N > 2, ordinary stage coupling for N = 2."""
    lay, kkt, eq, ine = _setup(model, N, final, periodic)
    assert kkt.n_border == (84 if periodic and N > 2 else 0)
    B = 3
    g = torch.Generator().manual_seed(N)
    hv = torch.randn((B, lay.nnz_h), generator=g, dtype=torch.float64)
    jv = torch.randn((B, lay.nnz_j), generator=g, dtype=torch.float64)
    sig = torch.rand((B, len(ine)), generator=g, dtype=torch.float64) * 3.0
    delta = torch.tensor([40.0, 55.0, 70.0], dtype=torch.float64)  # random W is indefinite: shift it well positive
    delta_c = 1e-6
    rx = torch.randn((B, lay.n_x), generator=g, dtype=torch.float64)
    rE = torch.randn((B, len(eq)), generator=g, dtype=torch.float64)
    rE[:, kkt.dead_eq] = 0.0  # rows with an empty Jacobian are outside the Newton system
    dx, dl = kkt.solve(hv, jv, sig, delta, delta_c, rx, rE)
    K = kkt.dense_matrix(hv, jv, sig, delta, delta_c, eq, ine, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row)
    ref = torch.linalg.solve(K, torch.cat([rx, rE], dim=1))
    u = torch.cat([dx, dl], dim=1)
    scale = ref.abs().amax(dim=1, keepdim=True)
    assert ((u - ref).abs() / scale).max().item() < 1e-9
    res = torch.einsum("bij,bj->bi", K, u) - torch.cat([rx, rE], dim=1)
    assert res.abs().max().item() < 1e-8 * max(1.0, float(scale.max()))
    if final:
        assert len(kkt.dead_eq) == 24  # parameter-only descriptor rows of the final-state constraint
        assert dl[:, kkt.dead_eq].abs().max().item() == 0.0


def test_stage_structure(model):
    lay, kkt, eq, ine = _setup(model, 5, False)
    assert [len(e) for e in kkt.eq_stage_rows] == [114, 142, 142, 142, 142]
    assert [len(i) for i in kkt.ine_stage_rows] == [82, 132, 132, 132, 132]
    assert [len(c) for c in kkt.cpl_local] == [0, 87, 87, 87, 87]  # 81 linear defects + 6 momentum rows
    assert kkt.nb == 195 + 142


def test_default_block_algebra_has_no_cpu_fallback(model):
    """linalg="hb" (the default) is the CUDA kernels of this library: CPU tensors are refused, not rerouted."""
    lay = KinoLayout(model, KinoSettings(horizon=2))
    p = kino_parameters(lay, model, 1, np.random.default_rng(0))
    lb, ub = lay.bounds(p)
    eq, ine = np.nonzero(lb[0] == ub[0])[0], np.nonzero(lb[0] != ub[0])[0]
    kkt = StageKKT(lay.n_x, lay.m, 2, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine)
    z = lambda *s: torch.zeros(s, dtype=torch.float64)
    with pytest.raises(ValueError, match="CUDA"):
        kkt.solve(z(1, lay.nnz_h), z(1, lay.nnz_j), z(1, len(ine)), z(1), 1e-8, z(1, lay.n_x), z(1, len(eq)))


def test_border_limit(model):
    """More far-coupling rows than the border is allowed to hold are refused at construction."""
    lay = KinoLayout(model, KinoSettings(horizon=3, periodicity_constraint=True))
    p = kino_parameters(lay, model, 1, np.random.default_rng(0))
    lb, ub = lay.bounds(p)
    eq = np.nonzero(lb[0] == ub[0])[0]
    ine = np.nonzero(lb[0] != ub[0])[0]
    with pytest.raises(NotImplementedError):
        StageKKT(lay.n_x, lay.m, 3, 189, lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row, eq, ine,
                 linalg="torch", max_border=10)


def test_sparse_operators_match_dense(model):
    """The interior-point driver never forms jac_g / hess_l: its products go straight through the CCS value
    arrays (ipsolver.SparseOps).  Checked against dense algebra on the real patterns."""
    from hippopt_b200.ipsolver import SparseOps

    lay = KinoLayout(model, KinoSettings(horizon=3, final_state_constraint=True))
    ops = SparseOps(lay.n_x, lay.m, (lay.jac_colind, lay.jac_row), (lay.hess_colind, lay.hess_row), "cpu")
    g = torch.Generator().manual_seed(5)
    B = 2
    jv = torch.randn((B, lay.nnz_j), generator=g, dtype=torch.float64)
    hv = torch.randn((B, lay.nnz_h), generator=g, dtype=torch.float64)
    x = torch.randn((B, lay.n_x), generator=g, dtype=torch.float64)
    lam = torch.randn((B, lay.m), generator=g, dtype=torch.float64)
    J, W = ops.dense_jac(jv), ops.dense_hess(hv)
    assert torch.allclose(ops.J_mul(jv, x), torch.einsum("bmn,bn->bm", J, x), rtol=1e-12, atol=1e-12)
    assert torch.allclose(ops.Jt_mul(jv, lam), torch.einsum("bmn,bm->bn", J, lam), rtol=1e-12, atol=1e-12)
    assert torch.allclose(ops.W_quad(hv, x), torch.einsum("bn,bnk,bk->b", x, W, x), rtol=1e-12, atol=1e-12)
    assert torch.equal(W, W.transpose(1, 2))


def _emulate_assemble(hdr, tab, hv, jv, sig, delta, delta_c, RX, RE, prev):
    """numpy restatement of csrc/kkt_assemble.cu for ONE instance: what hb_kkt_assemble_stage builds from a stage table."""
    nb, nx, nv, ne, R, n_cpl, n_cpl_next, n_direct, n_targets, n_contrib, n_a, n_an, nb_prev = hdr
    parts = [n_direct, n_direct, n_targets, n_targets + 1, n_contrib, n_contrib, n_contrib, nv, ne, n_cpl, n_cpl + 1, n_a, n_a,
             n_an, n_an, n_an]
    assert sum(parts) == len(tab)
    o = np.cumsum([0] + parts)
    (direct_val, direct_pos, tgt_pos, tgt_ptr, tgt_sig, tgt_e1, tgt_e2, var, eq, cpl, a_ptr, a_val, a_col, an_val, an_row,
     an_col) = (tab[o[i]:o[i + 1]] for i in range(16))
    W = R + n_cpl_next
    D = np.zeros(nb * nb)
    rhs = np.zeros((nb, W))
    D[direct_pos] = np.where(direct_val >= 0, hv[np.maximum(direct_val, 0)], jv[np.maximum(~direct_val, 0)])
    rhs[:nv, :R] = RX[var]
    rhs[nx:nx + ne, :R] = RE[eq]
    rhs[an_col, R + an_row] = jv[an_val]
    for t in range(n_targets):
        q = slice(tgt_ptr[t], tgt_ptr[t + 1])
        D[tgt_pos[t]] += np.sum(sig[tgt_sig[q]] * jv[tgt_e1[q]] * jv[tgt_e2[q]])
    D = D.reshape(nb, nb)
    i = np.arange(nb)
    D[i, i] += np.where(i < nv, delta, np.where(i < nx, 1.0, np.where(i < nx + ne, -delta_c, 1.0)))
    if n_cpl and prev is not None:
        assert prev.shape == (nb_prev, R + n_cpl)
        for r in range(n_cpl):
            q = slice(a_ptr[r], a_ptr[r + 1])
            acc = jv[a_val[q]] @ prev[a_col[q], :]
            rhs[cpl[r], :R] -= acc[:R]
            D[cpl[r], cpl] -= acc[R:]
    return D, rhs


@pytest.mark.parametrize("N,final", [(3, False), (3, True)])
def test_fused_stage_tables_match_the_torch_assembly(model, N, final):
    """The tables hb_kkt_assemble_stage consumes (per-stage block sizes, value entries, J_I^T Sigma J_I contribution lists,
    coupling rows) against the torch assembly of the linalg="torch" sweep, through a numpy restatement of the kernel."""
    lay, kkt, eq, ine = _setup(model, N, final)
    g = torch.Generator().manual_seed(7)
    hv = torch.randn((1, lay.nnz_h), generator=g, dtype=torch.float64)
    jv = torch.randn((1, lay.nnz_j), generator=g, dtype=torch.float64)
    sig = torch.rand((1, len(ine)), generator=g, dtype=torch.float64) * 3.0
    delta = torch.tensor([0.7], dtype=torch.float64)
    R = 2
    RX = torch.randn((1, lay.n_x, R), generator=g, dtype=torch.float64)
    RE = torch.randn((1, len(eq), R), generator=g, dtype=torch.float64)
    nx = kkt.nx
    assert kkt.stage_nb == [kkt.stage_nx[k] + len(kkt.eq_stage_rows[k]) for k in range(N)]
    assert max(kkt.stage_nb) <= kkt.nb and (not final or kkt.stage_nb[-1] > kkt.stage_nb[1])
    for k in range(N):
        hdr, tab = kkt._stage_np[k]
        hdr = list(hdr)
        hdr[4] = R
        nbk, nxk, ne = hdr[0], hdr[1], hdr[3]
        n_cpl = hdr[5]
        prev = None
        if n_cpl:
            prev = np.random.default_rng(k).standard_normal((hdr[12], R + n_cpl))
        D, rhs = _emulate_assemble(hdr, tab.astype(np.int64), hv[0].numpy(), jv[0].numpy(), sig[0].numpy(), 0.7, 1e-6,
                                   RX[0].numpy(), RE[0].numpy(), prev)
        Dt, bt = kkt._assemble(k, hv, jv, sig, delta, 1e-6, RX, RE)
        Dt, bt = Dt[0].numpy().copy(), bt[0].numpy().copy()
        idx = np.concatenate([np.arange(nxk), nx + np.arange(ne)])  # the stage's own slots inside the padded block
        if n_cpl:
            A = kkt._coupling(k, jv)[0].numpy()                       # (n_cpl, nx) on the padded slots of stage k - 1
            nx_prev = kkt.stage_nx[k - 1]
            assert np.all(A[:, nx_prev:] == 0.0)
            cp = nx + kkt.cpl_local[k]
            Dt[np.ix_(cp, cp)] -= A[:, :nx_prev] @ prev[:nx_prev, R:]
            bt[cp, :] -= A[:, :nx_prev] @ prev[:nx_prev, :R]
        assert np.allclose(D, Dt[np.ix_(idx, idx)], rtol=1e-13, atol=1e-13)
        assert np.allclose(rhs[:, :R], bt[idx], rtol=1e-13, atol=1e-13)
        if k + 1 < N:  # appended columns: A_{k+1}^T on this stage's variable rows
            An = kkt._coupling(k + 1, jv)[0].numpy()
            assert np.allclose(rhs[:nxk, R:], An[:, :nxk].T) and np.all(rhs[nxk:, R:] == 0.0)
