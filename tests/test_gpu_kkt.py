"""Row f2 (SURVEY.md 8(f)): batched LU kernels (csrc/lu.cu) and the stage-wise KKT sweep on the GPU.

Oracles: torch.linalg (LAPACK-equivalent solutions) for the LU kernels; a dense solve of the same KKT matrix
for the sweep, on values produced by the evaluation kernels."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


@pytest.mark.parametrize("n,r,B", [(1, 1, 3), (16, 5, 4), (17, 33, 5), (337, 88, 6), (400, 1, 2), (768, 3, 1)])
def test_lu_kernels_match_lapack(built_library, n, r, B):
    from hippopt_b200.kkt import lu_factor, lu_solve

    g = torch.Generator().manual_seed(n)
    A = torch.randn((B, n, n), generator=g, dtype=torch.float64).to(dev())
    rhs = torch.randn((B, n, r), generator=g, dtype=torch.float64).to(dev())
    F, piv, info = lu_factor(A.clone())
    assert int(info.abs().max()) == 0
    X = lu_solve(F, piv, rhs)
    ref = torch.linalg.solve(A, rhs)
    res = (torch.bmm(A, X) - rhs).abs().max().item()
    scale = ref.abs().max().item()
    assert (X - ref).abs().max().item() <= 1e-9 * scale * max(1.0, float(torch.linalg.cond(A).max()) * 1e-4)
    assert res <= 1e-10 * max(1.0, scale) * n
    # same factors, second solve with one right-hand side
    x1 = lu_solve(F, piv, rhs[:, :, :1])
    assert torch.equal(x1, X[:, :, :1])


def test_lu_pivots_like_partial_pivoting(built_library):
    """A matrix whose leading entry is zero needs the interchange; a singular one is reported in info."""
    from hippopt_b200.kkt import lu_factor, lu_solve

    A = torch.tensor([[[0.0, 2.0, 1.0], [1.0, 1.0, 0.0], [4.0, 0.0, 3.0]]], dtype=torch.float64, device=dev())
    b = torch.tensor([[[1.0], [2.0], [3.0]]], dtype=torch.float64, device=dev())
    F, piv, info = lu_factor(A.clone())
    assert int(info[0]) == 0 and int(piv[0, 0]) == 2  # largest entry of column 0 is in row 2
    assert torch.allclose(torch.bmm(A, lu_solve(F, piv, b)), b, atol=1e-14)
    S = torch.zeros((2, 20, 20), dtype=torch.float64, device=dev())
    S[0] = torch.eye(20, dtype=torch.float64)
    S[1] = torch.eye(20, dtype=torch.float64)
    S[1, 7, 7] = 0.0
    _, _, info = lu_factor(S)
    assert info.tolist() == [0, 8]
    with pytest.raises(ValueError):
        lu_factor(torch.zeros((2, 3, 3), dtype=torch.float64))  # CPU tensor: no fallback


@pytest.mark.parametrize("periodic", [False, True])
def test_stage_sweep_on_evaluated_values(model, built_library, periodic):
    """periodic = BASELINE config 4's structure: the periodicity rows are a border of the block-tridiagonal
    matrix (one sweep with 1 + 84 right-hand sides, then an 84 x 84 Schur complement)."""
    from hippopt_b200.evaluator import ALL, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.kkt import StageKKT
    from hippopt_b200.workloads import kino_batch

    N, B = 4, 5
    ev = KinoEvaluator(model, KinoSettings(horizon=N, final_state_constraint=True, periodicity_constraint=periodic))
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=3, noise=0.05)
    lb, ub = ev.bounds(p)
    d = dev()
    out = ev.eval(ALL, *(torch.tensor(a, device=d) for a in (x, p, lam, np.ones(B))))
    g = torch.Generator().manual_seed(1)
    hv, jv = out["hess"].clone(), out["jac"].clone()
    sols = {}
    for linalg in ("hb", "torch"):  # hb: one assembly kernel per stage; torch: the torch assembly and torch.linalg
        kkt, eq, ine = StageKKT.for_evaluator(ev, lb[0], ub[0], device=d, linalg=linalg)
        if linalg == "hb":
            sig = (torch.rand((B, len(ine)), generator=g, dtype=torch.float64) * 10.0).to(d)
            delta = torch.full((B,), 1e-2, dtype=torch.float64, device=d)
            rx = torch.randn((B, ev.n_x), generator=g, dtype=torch.float64).to(d)
            rE = torch.randn((B, len(eq)), generator=g, dtype=torch.float64).to(d)
            rE[:, torch.as_tensor(kkt.dead_eq, device=d)] = 0.0
        sols[linalg] = torch.cat(kkt.solve(hv, jv, sig, delta, 1e-9, rx, rE, chunk=2), dim=1)  # 3 chunks
        assert (kkt._stage_dev is not None) == (linalg == "hb")  # hb ran the fused sweep: its stage tables are uploaded
    jc, jr = ev.jac_sparsity()
    hc, hr = ev.hess_sparsity()
    K = kkt.dense_matrix(hv, jv, sig, delta, 1e-9, eq, ine, jc, jr, hc, hr)
    ref = torch.linalg.solve(K, torch.cat([rx, rE], dim=1))
    scale = ref.abs().amax(dim=1, keepdim=True)
    for name, u in sols.items():
        assert ((u - ref).abs() / scale).max().item() < 1e-6, name  # cond(K) ~ 1e11: the residual is the sharp check
        res = torch.einsum("bij,bj->bi", K, u) - torch.cat([rx, rE], dim=1)
        assert (res.abs() / scale).max().item() < 1e-12, name
    # several right-hand sides at once (limited-memory mode), fused path: column c solves K u = rhs[:, :, c]
    kkt, eq, ine = StageKKT.for_evaluator(ev, lb[0], ub[0], device=d, linalg="hb")
    RXm = torch.randn((B, ev.n_x, 3), generator=g, dtype=torch.float64).to(d)
    REm = torch.randn((B, len(eq), 3), generator=g, dtype=torch.float64).to(d)
    REm[:, torch.as_tensor(kkt.dead_eq, device=d), :] = 0.0
    dxm, dlm = kkt.solve(hv, jv, sig, delta, 1e-9, RXm, REm)
    um = torch.cat([dxm, dlm], dim=1)
    rm = torch.cat([RXm, REm], dim=1)
    resm = torch.bmm(K, um) - rm
    assert (resm.abs().amax(dim=(1, 2)) / um.abs().amax(dim=(1, 2))).max().item() < 1e-12
    # and the sweep is reproducible bit for bit
    dx2, dl2 = kkt.solve(hv, jv, sig, delta, 1e-9, RXm, REm)
    assert torch.equal(dx2, dxm) and torch.equal(dl2, dlm)


@pytest.mark.parametrize("periodic", [False, True])
def test_stage_sweep_at_the_production_chunk(model, built_library, periodic):
    """The default chunk of StageKKT.solve (2 x SM count instances) on 2 sms + 3 instances: one full chunk, whose
    stage blocks the MB = 2 factor kernel takes, then a ragged chunk of 3 on the MB = 1 kernel.  Every instance's
    residual against the dense matrix, and a dense solve on both sides of the chunk boundary and at the ends."""
    import ctypes

    from hippopt_b200.evaluator import ALL, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.kkt import StageKKT
    from hippopt_b200.workloads import kino_batch

    d = dev()
    sms = torch.cuda.get_device_properties(d).multi_processor_count
    chunk = 2 * sms
    N, B = 4, chunk + 3
    ev = KinoEvaluator(model, KinoSettings(horizon=N, final_state_constraint=True, periodicity_constraint=periodic))
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=4, noise=0.05)
    lb, ub = ev.bounds(p)
    out = ev.eval(ALL, *(torch.tensor(a, device=d) for a in (x, p, lam, np.ones(B))))
    hv, jv = out["hess"].clone(), out["jac"].clone()
    kkt, eq, ine = StageKKT.for_evaluator(ev, lb[0], ub[0], device=d, linalg="hb")
    plan = (ctypes.c_int32 * 4)()
    for batch, mb in ((chunk, 2), (3, 1)):
        assert built_library.hb_debug_lu_plan(kkt.nb, batch, 1, sms, plan) == 0 and plan[1] == mb, (kkt.nb, batch)
    g = torch.Generator().manual_seed(2)
    sig = (torch.rand((B, len(ine)), generator=g, dtype=torch.float64) * 10.0).to(d)
    delta = torch.full((B,), 1e-2, dtype=torch.float64, device=d)
    rx = torch.randn((B, ev.n_x), generator=g, dtype=torch.float64).to(d)
    rE = torch.randn((B, len(eq)), generator=g, dtype=torch.float64).to(d)
    rE[:, torch.as_tensor(kkt.dead_eq, device=d)] = 0.0
    u = torch.cat(kkt.solve(hv, jv, sig, delta, 1e-9, rx, rE), dim=1)  # default chunk
    assert kkt._stage_dev is not None  # the fused sweep ran (its stage tables are on the device)
    rhs = torch.cat([rx, rE], dim=1)
    jc, jr = ev.jac_sparsity()
    hc, hr = ev.hess_sparsity()
    dense_check = {0, chunk - 1, chunk, B - 1}
    for s in range(0, B, 32):
        sl = slice(s, min(s + 32, B))
        K = kkt.dense_matrix(hv[sl], jv[sl], sig[sl], delta[sl], 1e-9, eq, ine, jc, jr, hc, hr)
        scale = u[sl].abs().amax(dim=1, keepdim=True)
        res = torch.einsum("bij,bj->bi", K, u[sl]) - rhs[sl]
        worst = (res.abs() / scale).amax(dim=1)
        assert worst.max().item() < 1e-12, (s + int(worst.argmax()), worst.max().item())
        for i in sorted(dense_check & set(range(sl.start, sl.stop))):
            ref = torch.linalg.solve(K[i - s], rhs[i])
            err = ((u[i] - ref).abs().max() / ref.abs().max()).item()
            assert err < 1e-6, (i, err)  # cond(K) ~ 1e11: the residual is the sharp check
        del K
