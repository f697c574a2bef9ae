"""The general smooth-step terrain (``terrain="tilted_steps"``, kernel terrain 2, the ramp's terrain) on the GPU: the
surface and frame jets against sympy / mpmath, `kino_contact_kernel<2>` and `pose_contact_kernel<2>` against the
long-double oracle with no entry masked, terrain 2 on the stairs against terrain 1, determinism, the hb_save / hb_load
round trip, the ramp plan set-up (`initial_guess.ramp_step_guess`) and the B200Solver driving both templates."""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch

import tilted_oracle as to

pytestmark = pytest.mark.gpu

RTOL = 1e-10
# ramp_step_guess: all 16 instances below have their three keyframe poses converged (measured on an NVIDIA B200 at
# 1000 W; DESIGN.md section 9.1)
RAMP_MIN_KEYFRAMES_OK = 16


def dev():
    return torch.device("cuda:0")


def run(ev, x, p, lam, sigma):
    from hippopt_b200.evaluator import ALL

    t = [torch.tensor(np.ascontiguousarray(a), device=dev()) for a in (x, p, lam, sigma)]
    out = ev.eval(ALL, *t)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def tilted(K):
    return dict(terrain="tilted_steps", n_terrain_params=10 * K)


# ------------------------------------------------------------------------------------------------ surface and frame
def bidx(i, j):
    return (i + j) * (i + j + 1) // 2 + j


def jet_index(N):
    return [(d - j, j) for d in range(N + 1) for j in range(d + 1)]


_SYM = {}


def symbolic_surface():
    """order-4 normalised derivatives of one tilted step's exp(-g^20) pi + oz, lambdified for mpmath"""
    if _SYM:
        return _SYM["surface"]
    import sympy as sp

    x, y, l, w, H, ox, oy, oz, yaw, nx, ny, nz = sp.symbols("x y l w H ox oy oz yaw nx ny nz", real=True)
    c, s = sp.cos(yaw), sp.sin(yaw)
    xt = c * (x - ox) + s * (y - oy)
    yt = c * (y - oy) - s * (x - ox)
    g = (2 * xt / l) ** 10 + (2 * yt / w) ** 10
    T = sp.exp(-g ** 20) * (H - nx / nz * xt - ny / nz * yt) + oz
    out = []
    for i, j in jet_index(4):
        e = T
        if i:
            e = sp.diff(e, x, i)
        if j:
            e = sp.diff(e, y, j)
        out.append(e / (math.factorial(i) * math.factorial(j)))
    _SYM["surface"] = sp.lambdify((x, y, l, w, H, ox, oy, oz, yaw, nx, ny, nz), out, modules="mpmath", cse=True)
    return _SYM["surface"]


def reference(tp, K, xyz, dps=40):
    """[n, 195] 40-digit values of hb_debug_tilted_terrain's outputs (rounded to float64); the frame from the surface
    derivatives through the symbolic frame of tests/test_gpu_smooth_terrain.py"""
    import mpmath

    import test_gpu_smooth_terrain as sm

    surface = symbolic_surface()
    sym = sm._symbolic()
    frame, fk = sym["frame"], sym["frame_keys"]
    f = math.factorial
    out_all = np.zeros((len(xyz), sm.N_OUT))
    with mpmath.workdps(dps):
        mp = mpmath.mpf
        for p in range(len(xyz)):
            x, y, z = (mp(float(v)) for v in xyz[p])
            Tn = [mp(0)] * 15
            for s in range(K):
                c = surface(x, y, *(mp(float(v)) for v in tp[p, 10 * s:10 * s + 10]))
                Tn = [a + b for a, b in zip(Tn, c)]
            raw = {ij: Tn[q] * f(ij[0]) * f(ij[1]) for q, ij in enumerate(jet_index(4))}
            fr = frame(*(raw[ij] for ij in jet_index(4)[1:]))
            out = list(Tn)

            def tj(cf):
                return [cf[(0, 0)], cf[(1, 0)], cf[(0, 1)], mp(0), cf[(2, 0)], cf[(1, 1)], mp(0), cf[(0, 2)], mp(0),
                        mp(0)]

            o2 = jet_index(2)
            h = tj({ij: -Tn[bidx(*ij)] for ij in o2})
            h[0] += z
            h[3] = mp(1)
            out += h
            out += tj({(i, j): -raw[(i + 1, j)] / (f(i) * f(j)) for i, j in o2})
            out += tj({(i, j): -raw[(i, j + 1)] / (f(i) * f(j)) for i, j in o2})
            for name in ("n", "xh", "yh"):
                for a in range(3):
                    out += tj({(i, j): fr[fk[(name, a, (i, j))]] / (f(i) * f(j)) for i, j in o2})
            for a in range(3):
                out += tj({(i, j): fr[fk[("n", a, (i + 1, j))]] / (f(i) * f(j)) for i, j in o2})
                out += tj({(i, j): fr[fk[("n", a, (i, j + 1))]] / (f(i) * f(j)) for i, j in o2})
            out_all[p] = [float(v) for v in out]
    return out_all


def debug_tilted(tp, K, xyz):
    from hippopt_b200 import _capi

    n = len(xyz)
    t = torch.tensor(np.ascontiguousarray(tp), device=dev())
    pts = torch.tensor(np.ascontiguousarray(xyz), device=dev())
    out = torch.zeros((n, 195), dtype=torch.float64, device=dev())
    _capi.check(_capi.lib().hb_debug_tilted_terrain(t.data_ptr(), K, pts.data_ptr(), n, out.data_ptr(), None),
                "hb_debug_tilted_terrain")
    torch.cuda.synchronize()
    return out.cpu().numpy()


STEP_A = [0.9, 0.6, 0.1, 0.3, -0.1, 0.02, 0.4, -0.2, 0.1, 0.97]   # rotated, raised, tilted
STEP_B = [1.2, 0.8, 0.05, 0.1, 0.1, -0.03, -1.1, 0.15, -0.25, 0.95]  # overlaps A
STEP_C = [0.5, 0.4, 0.08, 0.35, 0.0, 0.01, 2.5, 0.3, 0.0, 0.95]      # steep tilt, inside A and B


def step_point(q, xt, yt, z=0.05):
    """world (x, y, z) of step coordinates (x_t, y_t)"""
    c, s = math.cos(q[6]), math.sin(q[6])
    return [q[3] + c * xt - s * yt, q[4] + s * xt + c * yt, z]


def surface_points():
    """edges, corners, the cut-off band and deep inside of each step, for K = 1, 2, 3 overlapping steps"""
    pts = []
    for q in (STEP_A, STEP_B, STEP_C):
        l, w = q[0], q[1]
        for u in (0.0, 0.3, 0.49, 0.5, 0.51, 0.53):
            pts.append(step_point(q, u * l, 0.1 * w))
            pts.append(step_point(q, -0.2 * l, -u * w))
        for a, b in ((0.5, 0.5), (0.49, -0.5), (-0.51, 0.49), (-0.5, -0.5)):
            pts.append(step_point(q, a * l, b * w))
        pts.append(step_point(q, 0.5 * l * 1.42 ** 0.1 * 0.999, 0.0))  # just inside the cut-off
        pts.append(step_point(q, 0.5 * l * 1.42 ** 0.1 * 1.001, 0.0))  # just beyond it
    return np.array(pts)


def check_jets(got, ref):
    """per point and per 10- / 15-coefficient block: |got - ref| <= 1e-9 max(1, max |ref| of the block)"""
    blocks = [(0, 15)] + [(15 + 10 * a, 25 + 10 * a) for a in range(18)]
    assert np.isfinite(got).all()
    for a, b in blocks:
        scale = np.maximum(1.0, np.abs(ref[:, a:b]).max(axis=1, keepdims=True))
        err = np.abs(got[:, a:b] - ref[:, a:b]) / scale
        assert err.max() <= 1e-9, (a, b, err.max(), np.unravel_index(err.argmax(), err.shape))


@pytest.mark.parametrize("K", [1, 2, 3])
def test_tilted_surface_and_frame_against_symbolic_reference(built_library, K):
    steps = np.concatenate([STEP_A, STEP_B, STEP_C][:K])
    xyz = surface_points()
    tp = np.tile(steps, (len(xyz), 1))
    check_jets(debug_tilted(tp, K, xyz), reference(tp, K, xyz))


def test_wide_step_frame_equals_the_plane(built_library):
    """A step far wider than the points' spread is its tilted plane: the terrain normal is the step's normal turned by
    the yaw, the frame is the plane's and every derivative of n vanishes."""
    rng = np.random.default_rng(3)
    ns = np.array([0.2, -0.1, 1.0])
    ns /= np.linalg.norm(ns)
    yaw = 0.3
    q = [1e3, 1e3, 0.1, 0.0, 0.0, 0.05, yaw, ns[0], ns[1], ns[2]]
    n = np.array([math.cos(yaw) * ns[0] - math.sin(yaw) * ns[1], math.sin(yaw) * ns[0] + math.cos(yaw) * ns[1], ns[2]])
    xyz = np.concatenate([rng.uniform(-1.0, 1.0, (16, 2)), rng.uniform(-0.2, 0.2, (16, 1))], axis=1)
    out = debug_tilted(np.tile(q, (16, 1)), 1, xyz)
    F = lambda a: out[:, 15 + 10 * a:25 + 10 * a]  # noqa: E731  TFrame field a
    yv = np.cross(n, [1.0, 0.0, 0.0])
    xv = np.cross(yv, n)
    xv /= np.linalg.norm(xv)
    yv = np.cross(n, xv)
    for a in range(3):
        assert np.abs(F(3 + a)[:, 0] - n[a]).max() < 1e-14
        assert np.abs(F(6 + a)[:, 0] - xv[a]).max() < 1e-14
        assert np.abs(F(9 + a)[:, 0] - yv[a]).max() < 1e-14
        assert np.abs(F(3 + a)[:, 1:]).max() < 1e-14
    for a in range(12, 18):
        assert np.abs(F(a)).max() < 1e-14
    # h = z - (plane + oz)
    xt = math.cos(yaw) * xyz[:, 0] + math.sin(yaw) * xyz[:, 1]
    yt = -math.sin(yaw) * xyz[:, 0] + math.cos(yaw) * xyz[:, 1]
    plane = 0.1 - ns[0] / ns[2] * xt - ns[1] / ns[2] * yt + 0.05
    assert np.abs(F(0)[:, 0] - (xyz[:, 2] - plane)).max() < 1e-14


def test_debug_entry_rejects_bad_arguments(built_library):
    from hippopt_b200 import _capi

    t = torch.zeros(10, dtype=torch.float64, device=dev())
    assert _capi.lib().hb_debug_tilted_terrain(t.data_ptr(), 0, t.data_ptr(), 1, t.data_ptr(), None) != 0
    assert _capi.lib().hb_debug_tilted_terrain(None, 1, t.data_ptr(), 1, t.data_ptr(), None) != 0


# ------------------------------------------------------------------------------------------------ contact kernels
def kino_inputs(ev, model, K, B, seed, noise):
    """kino_batch on K sampled tilted steps, with the contact points of some knots written onto step edges and corners"""
    from hippopt_b200.kino_layout import NZ, P
    from hippopt_b200.workloads import kino_batch

    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=seed, noise=noise)
    rng = np.random.default_rng(seed)
    po = ev.layout.po
    for b in range(B):
        for k in range(ev.layout.N):
            if (b + k) % 2:
                continue
            for i in range(8):
                s = rng.integers(K)
                q = p[b, po.terrain + 10 * s:po.terrain + 10 * s + 10]
                u = rng.choice([0.5, -0.5, 0.495, 0.505])
                v = rng.uniform(-0.5, 0.5) if i % 2 else rng.choice([0.5, -0.5])
                pt = step_point(q, u * q[0], v * q[1], z=rng.uniform(-0.05, 0.15))
                x[b, NZ * k + 15 * i + P:NZ * k + 15 * i + P + 3] = pt
    return x, p, lam, sigma


def check_kino(model, ev, K, x, p, lam, sigma, **st):
    from oracle import parity

    nlp, _ = to.kino_build(model, K, horizon=ev.layout.N, **st)
    assert np.array_equal(ev.jac_sparsity()[1], nlp.jac_structure()[1])
    assert np.array_equal(ev.hess_sparsity()[1], nlp.hess_structure()[1])
    out = run(ev, x, p, lam, sigma)
    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(out[k]).all() and np.isfinite(r).all(), k
    worst = parity.check_all(out, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2], x, rtol=RTOL)
    print("worst relative errors:", {k: f"{v:.2e}" for k, v in worst.items()})


@pytest.mark.parametrize("N,K,fin,per,noise", [(3, 1, True, False, 0.05), (3, 2, False, False, 0.15),
                                               (4, 3, True, True, 0.05), (4, 1, False, True, 0.15)])
def test_kino_contact_kernel_on_tilted_steps_against_oracle(model, built_library, N, K, fin, per, noise):
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings

    st = dict(final_state_constraint=fin, periodicity_constraint=per)
    ev = KinoEvaluator(model, KinoSettings(horizon=N, **tilted(K), **st))
    x, p, lam, sigma = kino_inputs(ev, model, K, 3, seed=60 + N + K, noise=noise)
    sigma = np.array([1.0, 0.3, 2.0])
    check_kino(model, ev, K, x, p, lam, sigma, **st)


def test_kino_contact_kernel_on_tilted_steps_at_horizon_50(model, built_library):
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings

    ev = KinoEvaluator(model, KinoSettings(horizon=50, final_state_constraint=True, **tilted(2)))
    x, p, lam, sigma = kino_inputs(ev, model, 2, 1, seed=71, noise=0.05)
    check_kino(model, ev, 2, x, p, lam, sigma, final_state_constraint=True)


def pose_inputs(ev, model, K, B, seed):
    from hippopt_b200.workloads import pose_batch, tilted_steps_sample

    rng = np.random.default_rng(seed)
    x, p, lam, sigma = pose_batch(ev.layout, model, B, seed=seed, noise=0.05)
    po = ev.layout.po
    p[:, po.terrain:] = tilted_steps_sample(K, B, rng)
    for b in range(B):
        for i in range(8):
            s = rng.integers(K)
            q = p[b, po.terrain + 10 * s:po.terrain + 10 * s + 10]
            if b % 3 == 0:
                continue
            u = rng.choice([0.5, -0.5, 0.49]) if b % 3 == 1 else rng.uniform(-0.4, 0.4)
            x[b, 6 * i:6 * i + 3] = step_point(q, u * q[0], rng.uniform(-0.5, 0.5) * q[1], z=rng.uniform(-0.05, 0.15))
    return x, p, lam, np.linspace(0.3, 2.0, B)


@pytest.mark.parametrize("K", [1, 2, 3])
def test_pose_contact_kernel_on_tilted_steps_against_oracle(model, built_library, K):
    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.pose_layout import PoseSettings
    from oracle import parity

    ev = PoseEvaluator(model, PoseSettings(**tilted(K)))
    x, p, lam, sigma = pose_inputs(ev, model, K, 7, seed=80 + K)
    out = run(ev, x, p, lam, sigma)
    nlp, _ = to.pose_build(model, K)
    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble)
    for k, r in ref.items():
        assert np.isfinite(out[k]).all() and np.isfinite(r).all(), k
    parity.check_all(out, ref, nlp.jac_structure()[:2], nlp.hess_structure()[:2], x, rtol=RTOL)


def test_tilted_steps_on_the_stairs_match_the_stairs_terrain(model, built_library):
    """Terrain 2 with the stairs written as two flat, axis-aligned steps at z = 0 against terrain 1 (kinodynamic and
    pose finder, all five outputs)."""
    from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.pose_layout import PoseSettings
    from hippopt_b200.workloads import kino_batch, pose_batch
    from oracle import parity

    stairs = dict(terrain="smooth_steps", n_terrain_params=10)
    e1 = KinoEvaluator(model, KinoSettings(horizon=4, final_state_constraint=True, **stairs))
    e2 = KinoEvaluator(model, KinoSettings(horizon=4, final_state_constraint=True, **tilted(2)))
    x, p, lam, sigma = kino_batch(e1.layout, model, 5, seed=90, noise=0.1)
    p2 = np.concatenate([p[:, :e1.layout.po.terrain], to.stairs_as_tilted(p[:, e1.layout.po.terrain:])], axis=1)
    a, b = run(e1, x, p, lam, sigma), run(e2, x, p2, lam, sigma)
    parity.check_all(b, a, e1.jac_sparsity(), e1.hess_sparsity(), x, rtol=RTOL)
    q1 = PoseEvaluator(model, PoseSettings(**stairs))
    q2 = PoseEvaluator(model, PoseSettings(**tilted(2)))
    x, p, lam, sigma = pose_batch(q1.layout, model, 6, seed=91)
    from hippopt_b200.initial_guess import stairs_terrain

    p[:, q1.layout.po.terrain:] = stairs_terrain(np.linspace(0.05, 0.15, 6))
    x[:, 0:48:6] = np.linspace(0.0, 0.9, 8)  # point x across the ground, both edges and both treads
    p2 = np.concatenate([p[:, :q1.layout.po.terrain], to.stairs_as_tilted(p[:, q1.layout.po.terrain:])], axis=1)
    a, b = run(q1, x, p, lam, sigma), run(q2, x, p2, lam, sigma)
    parity.check_all(b, a, q1.jac_sparsity(), q1.hess_sparsity(), x, rtol=RTOL)


def test_tilted_outputs_are_bit_identical_across_batch_order_and_size(model, built_library):
    from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.pose_layout import PoseSettings

    ev = KinoEvaluator(model, KinoSettings(horizon=5, **tilted(2)))
    x, p, lam, sigma = kino_inputs(ev, model, 2, 37, seed=5, noise=0.05)
    pev = PoseEvaluator(model, PoseSettings(**tilted(3)))
    for e, (x, p, lam, sigma) in ((ev, (x, p, lam, sigma)), (pev, pose_inputs(pev, model, 3, 530, seed=6))):
        B = x.shape[0]
        out = run(e, x, p, lam, sigma)
        perm = np.random.default_rng(4).permutation(B)
        permuted = run(e, x[perm], p[perm], lam[perm], sigma[perm])
        part = run(e, x[:7], p[:7], lam[:7], sigma[:7])
        for k in out:
            assert np.isfinite(out[k]).all(), k
            assert np.array_equal(permuted[k], out[k][perm]), k
            assert np.array_equal(part[k], out[k][:7]), k


def test_save_load_round_trip_of_a_tilted_handle(model, built_library, tmp_path):
    """hb_save of a terrain-2 handle, hb_load of the file: hb_eval_host gives bit-identical outputs on both handles."""
    from hippopt_b200 import _capi
    from hippopt_b200.evaluator import ALL, HostPipeline, KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings

    ev = KinoEvaluator(model, KinoSettings(horizon=4, final_state_constraint=True, **tilted(3)))
    x, p, lam, sigma = kino_inputs(ev, model, 3, 4, seed=9, noise=0.05)
    path = str(tmp_path / "tilted.bin")
    ev.save(path)
    loaded = copy.copy(ev)  # same dimensions and layout, its own handle (released by its close / __del__)
    loaded._h = ctypes.c_void_p()
    _capi.check(_capi.lib().hb_load(path.encode(), ctypes.byref(loaded._h)), "hb_load")
    outs = []
    try:
        for e in (ev, loaded):
            pipe = HostPipeline(e, 4, ALL)
            pipe.set_parameters(torch.from_numpy(np.ascontiguousarray(p)))
            o = pipe.run(*(torch.from_numpy(np.ascontiguousarray(a)) for a in (x, lam, sigma)))
            outs.append({k: v.numpy().copy() for k, v in o.items()})
    finally:
        loaded.close()
    for k in outs[0]:
        assert np.isfinite(outs[0][k]).all() and np.array_equal(outs[0][k], outs[1][k]), k


def test_create_rejects_a_terrain_block_that_is_not_whole_steps(model, built_library):
    from hippopt_b200 import _capi
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings

    lay_ok = KinoEvaluator(model, KinoSettings(horizon=3, **tilted(1))).layout
    from hippopt_b200.kino_layout import KinoLayout

    lay = KinoLayout(model, KinoSettings(horizon=3, **tilted(1)))
    lay.po.n_p = lay.n_p = lay_ok.n_p - 3  # 7 terrain parameters
    with pytest.raises(_capi.EvaluationError):
        KinoEvaluator(model, KinoSettings(horizon=3, **tilted(1)), layout=lay)


# ------------------------------------------------------------------------------------------------ ramp plans
def test_ramp_step_guess(model, built_library):
    """Keyframe poses on ramps with slopes in U(0.05, 0.2): the contact corners sit on or above the terrain, the
    corners on the slope lie on it and the guess is finite."""
    from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
    from hippopt_b200.initial_guess import ramp_step_guess, ramp_terrain
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.pose_layout import PoseSettings

    B = 16
    s = np.random.default_rng(8).uniform(0.05, 0.2, B)
    ev = KinoEvaluator(model, KinoSettings(horizon=50, final_state_constraint=True, **tilted(1)))
    gs = ramp_step_guess(model, PoseEvaluator(model, PoseSettings(**tilted(1))), ev, s, mass_normalised=True)
    n_ok = int(gs.ok.sum())
    print(f"ramp keyframes: {n_ok} of {B} instances with all three keyframe poses converged")
    assert n_ok >= RAMP_MIN_KEYFRAMES_OK
    assert torch.isfinite(gs.x0).all() and np.isfinite(gs.parameters).all()
    tp = gs.parameters[:, ev.layout.po.terrain:]
    assert np.array_equal(tp, ramp_terrain(s))
    key = gs.keyframes.cpu().numpy()
    ok = gs.ok.cpu().numpy()
    for kf in range(3):
        for i in range(8):
            pt = key[kf, ok, 9 * i:9 * i + 3]
            on_slope = (i < 4 and kf >= 1) or (i >= 4 and kf == 2)
            h = np.array([_ramp_h(pt[j], tp[ok][j]) for j in range(len(pt))])
            assert (h >= -1e-6).all(), (kf, i)
            if on_slope:
                assert np.abs(h).max() < 1e-3, (kf, i)
            else:
                assert np.abs(pt[:, 2]).max() < 1e-3, (kf, i)


def _ramp_h(pt, q):
    l, w, H, ox, oy, oz, yaw, nx, ny, nz = q
    xt, yt = pt[0] - ox, pt[1] - oy
    g = min((2 * xt / l) ** 10 + (2 * yt / w) ** 10, 10.0)
    return pt[2] - math.exp(-g ** 20) * (H - nx / nz * xt - ny / nz * yt) - oz


def test_b200_solver_drives_both_templates_on_tilted_steps(model, built_library):
    """B200Solver with explicit settings on the new terrain: the pose finder on a ramp (feet on the flat ground in front
    of it) solves to the evaluator's own cost; the kinodynamic template on two tilted steps builds and iterates."""
    from hippopt_b200.evaluator import F, KinoEvaluator, PoseEvaluator
    from hippopt_b200.initial_guess import pose_problem, ramp_terrain
    from hippopt_b200.ipsolver import OptiFailure
    from hippopt_b200.kino_layout import KinoSettings
    from hippopt_b200.plugin import B200Solver
    from hippopt_b200.pose_layout import PoseSettings
    from hippopt_b200.workloads import kino_batch

    B = 2
    pev = PoseEvaluator(model, PoseSettings(**tilted(1)))
    zero = np.zeros(B)
    x, p = pose_problem(pev.layout, model, np.stack([zero, zero + 0.1, zero], 1), np.stack([zero, zero - 0.1, zero], 1))
    p[:, pev.layout.po.terrain:] = ramp_terrain(np.array([0.1, 0.2]))
    s = B200Solver(model=model, batch=B, evaluator=pev, kkt="dense", options_solver={"tol": 1e-8, "max_iter": 300})
    s.generate_optimization_objects({"x": x, "p": p})
    s.solve()
    assert bool(s._last_output.success.all())
    vec = s.get_solution_vectors()
    f = pev.eval(F, torch.tensor(vec["x"], device=dev()), torch.tensor(p, device=dev()))["f"].cpu().numpy()
    assert s.get_cost_value() == pytest.approx(f, rel=1e-12)

    st = KinoSettings(horizon=3, **tilted(2))
    ev = KinoEvaluator(model, st)
    x, p, _, _ = kino_batch(ev.layout, model, B, seed=13)
    ks = B200Solver(model=model, settings=st, batch=B, options_solver={"max_iter": 3})
    ks.generate_optimization_objects({"x": x, "p": p})
    try:
        ks.solve()
    except OptiFailure:
        pass
    assert ks._evaluator().layout.kernel_terrain == 2 and ks._evaluator().n_p == ev.n_p
