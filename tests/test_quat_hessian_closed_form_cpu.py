"""Closed forms of the base-quaternion columns of the kinematics Hessian (hippopt_b200/csrc/kino_kin.cu, "quaternion
columns"), restated with numpy and checked against the oracle's Hessian of the Lagrangian on the CPU.

A quaternion direction q_a rotates the whole tree about the base origin (alpha = g_a) and adds u_a to the base angular
velocity.  The kernel does not walk the tree for it: the kinematic rows are either rotation invariant (feet distance)
or a world-fixed multiplier dotted with a vector X that rotates with the tree, so the tangents of the root totals
n0 = dPhi/d(rotation) and w0 = dPhi/d omega_0 follow from a handful of root quantities, and the velocity rows follow
from the covariance of the momentum map."""
import numpy as np
import pytest

from oracle import kinodynamic as kd


def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def quat_rot(q):
    v, w = q[:3], q[3]
    S = skew(v)
    return np.eye(3) + 2.0 * w * S + 2.0 * S @ S


def omega_map(a, b):
    """right-trivialised angular velocity map Omega(a, b) = 2(-b_w a_v + a_w b_v - b_v x a_v)"""
    return 2.0 * (a[3] * b[:3] - b[3] * a[:3] - np.cross(b[:3], a[:3]))


def quat_maps(q, qd):
    """g_a, u_a, w_a for a = 0..3 (kino_kin.cu quat_map); complex inputs give complex-step derivatives"""
    r = np.sqrt(q @ q)
    qh = q / r
    g, u, w = [], [], []
    for a in range(4):
        t = (np.eye(4)[a] - qh * qh[a]) / r
        g.append(omega_map(qh, t))
        u.append(omega_map(t, qd))
        w.append(omega_map(qh, np.eye(4)[a]))
    return np.array(g), np.array(u), np.array(w)


def quat_map_curvature(q, qd):
    """dg_a/dq_b, du_a/dq_b, dw_a/dq_b as [a][b][3], by complex step (exact to rounding)"""
    h = 1e-30
    out = np.zeros((3, 4, 4, 3))
    for b in range(4):
        qc = q.astype(complex)
        qc[b] += 1j * h
        for i, m in enumerate(quat_maps(qc, qd.astype(complex))):
            out[i, :, b] = m.imag / h
    return out


def knot_state(model, z, desc, fq):
    """the primal quantities of one knot, as the kernel stages them (positions relative to the base origin)"""
    q, qd, vb, s, sd = z[kd.Q:kd.Q + 4], z[kd.QD:kd.QD + 4], z[kd.VB:kd.VB + 3], z[kd.S:kd.S + 23], z[kd.SD:kd.SD + 23]
    qh = q / np.linalg.norm(q)
    nb = model.n_bodies
    R = [quat_rot(qh)] + [None] * (nb - 1)
    o, w, v, ax = [np.zeros(3)] * nb, [omega_map(qh, qd)] + [None] * (nb - 1), [vb] + [None] * (nb - 1), [None] * nb
    for l in range(1, nb):
        p = int(model.parent[l])
        a = model.joint_axis[l]
        Rl = model.joint_rot[l] @ (np.eye(3) + np.sin(s[l - 1]) * skew(a) + (1 - np.cos(s[l - 1])) * skew(a) @ skew(a))
        R[l] = R[p] @ Rl
        rho = R[p] @ model.joint_xyz[l]
        o[l] = o[p] + rho
        ax[l] = R[l] @ a
        w[l] = w[p] + sd[l - 1] * ax[l]
        v[l] = v[p] + np.cross(w[p], rho)
    M = model.total_mass()
    st = dict(qh=qh, q=q, qd=qd, omega0=w[0], o=o, ax=ax, M=M)
    P, Pd, H, J = np.zeros(3), np.zeros(3), np.zeros(3), np.zeros((3, 3))
    for l in range(nb):
        m = model.mass[l]
        d = R[l] @ model.com[l]
        Iw = R[l] @ model.inertia[l] @ R[l].T
        c, cd = o[l] + d, v[l] + np.cross(w[l], d)
        P, Pd = P + m * c, Pd + m * cd
        H = H + m * np.cross(c, cd) + Iw @ w[l]
        J = J + Iw + m * ((c @ c) * np.eye(3) - np.outer(c, c))
    st["P"], st["hang"] = P, H - np.cross(P, Pd) / M
    st["xc"] = P / M
    st["Ic"] = J - ((P @ P) * np.eye(3) - np.outer(P, P)) / M  # locked inertia about the CoM
    pts = []
    for i in range(8):
        body, Rf, tf = model.frames["l_sole" if i < 4 else "r_sole"]
        pts.append(o[body] + R[body] @ (Rf @ desc[i] + tf))
    st["r_pt"] = np.array(pts)
    cb, cR, _ = model.frames["chest"]
    st["G"] = R[cb] @ cR @ quat_rot(fq).T

    def sub_momentum(j):
        """d hang / d s_dot_j: the sub-tree of body j + 1 turns about its joint"""
        A, piv = ax[j + 1], o[j + 1]
        Ps, Ms, Js = np.zeros(3), 0.0, np.zeros((3, 3))
        for l in range(nb):
            if model.subtree_mask()[j + 1, l]:
                m = model.mass[l]
                d = R[l] @ model.com[l]
                c = o[l] + d
                Ps, Ms = Ps + m * c, Ms + m
                Js = Js + R[l] @ model.inertia[l] @ R[l].T + m * ((c @ c) * np.eye(3) - np.outer(c, c))
        pv = np.cross(A, Ps - Ms * piv)
        return Js @ A - np.cross(Ps, np.cross(A, piv)) - np.cross(P, pv) / M

    st["dh_dsd"] = np.array([sub_momentum(j) for j in range(23)])
    return st


def quaternion_columns(st, lam_fk, lam_c, lam_m, lam_u, mass_p, sigma, w_frame, w_bq, bq_ref, k1):
    """rows vb3 qd4 sd23 q4 of the four q columns, as the kernel's closed forms compute them"""
    g, u, wq = quat_maps(st["q"], st["qd"])
    curv = quat_map_curvature(st["q"], st["qd"])
    hb = -lam_m / mass_p
    Ic, om, hang, xc, G = st["Ic"], st["omega0"], st["hang"], st["xc"], st["G"]
    w0 = Ic @ hb
    phi = np.trace(G)
    mG = np.array([G[1, 2] - G[2, 1], G[2, 0] - G[0, 2], G[0, 1] - G[1, 0]])
    cw = 2.0 * sigma * w_frame if k1 else 0.0
    kappa = cw * (phi - 3.0)
    n0 = (sum(np.cross(r, -l) for r, l in zip(st["r_pt"], lam_fk)) + np.cross(xc, -lam_c) + np.cross(hang, hb)
          - np.cross(om, w0) + kappa * mG)
    K = np.einsum("i,abi->ab", n0, curv[0]) + np.einsum("i,abi->ab", w0, curv[1])  # K[a][b]
    Kd = np.einsum("i,abi->ab", w0, curv[2])
    out = np.zeros((34, 4))
    for a in range(4):
        al, ua = g[a], u[a]
        tw0 = np.cross(al, w0) - Ic @ np.cross(al, hb)
        th = np.cross(al, hang) - Ic @ np.cross(al, om) + Ic @ ua
        tn0 = (sum(np.cross(np.cross(al, r), -l) for r, l in zip(st["r_pt"], lam_fk)) + np.cross(np.cross(al, xc), -lam_c)
               + np.cross(th, hb) - np.cross(ua, w0) - np.cross(om, tw0)
               + cw * mG * (al @ mG) + kappa * (G @ al - phi * al))
        for b in range(4):
            out[3 + b, a] = tw0 @ wq[b] + Kd[b, a]
            out[30 + b, a] = tn0 @ g[b] + tw0 @ u[b] + K[b, a]
        if k1:
            out[30 + a, a] += 2.0 * sigma * w_bq * (bq_ref @ bq_ref) + 2.0 * lam_u
        for j in range(23):  # covariance of the momentum map: d/dq_a (lam_m . dh/dsd_j / mass_p)
            out[7 + j, a] = hb @ np.cross(al, st["dh_dsd"][j])
    return out


@pytest.mark.parametrize("k", [0, 2])
def test_quaternion_columns_match_the_oracle(model, k):
    N = 3
    cfg = kd.Settings(horizon=N)
    nlp, lay = kd.build(model, cfg)
    rng = np.random.default_rng(5 + k)
    X = rng.normal(0, 0.3, (1, nlp.n_x))
    P = rng.uniform(0.5, 1.5, (1, nlp.n_p))
    lam_all = rng.normal(0, 1, (1, nlp.m))
    lam = np.zeros_like(lam_all)
    kin = ("p_kinematics_consistency", "com_kinematics_consistency", "centroidal_momentum_kinematics_consistency",
           "minimum_feet_distance", "unitary_quaternion")
    rows = {}
    for name, off, n in nlp.constraint_names:
        if name.endswith(f"[{k}]") and any(t in name for t in kin):
            lam[0, off:off + n] = lam_all[0, off:off + n]
            rows[name] = lam[0, off:off + n]
    sigma = 0.7
    Hd = nlp.dense_hess(X, P, lam, sigma)[0]

    z = X[0, kd.NZ * k:kd.NZ * (k + 1)]
    Pw = np.concatenate([X[0], P[0]])
    desc = np.array([Pw[lay.desc(k, i)] for i in range(8)])
    st = knot_state(model, z, desc, Pw[lay.ref(k, "fq")])
    k1 = k >= 1
    fk = np.zeros((8, 3))
    lam_c = lam_m = np.zeros(3)
    lam_u = 0.0
    for name, v in rows.items():
        if "p_kinematics_consistency" in name:
            side, idx = ("left", 0) if ".left[" in name else ("right", 4)
            fk[idx + int(name.split(side + "[")[1][0])] = v
        elif name.startswith("com_kinematics"):
            lam_c = v
        elif name.startswith("centroidal_momentum_kinematics"):
            lam_m = v
        elif name.startswith("unitary"):
            lam_u = v[0]
    got = quaternion_columns(st, fk, lam_c, lam_m, lam_u, Pw[lay.mass], sigma, cfg.desired_frame_quaternion_cost_multiplier,
                             cfg.base_quaternion_cost_multiplier, Pw[lay.ref(k, "bq")], k1)
    base = kd.NZ * k
    cols = base + kd.Q + np.arange(4)
    rws = np.concatenate([base + kd.VB + np.arange(3), base + kd.QD + np.arange(4), base + kd.SD + np.arange(23),
                          base + kd.Q + np.arange(4)])
    want = Hd[np.ix_(rws, cols)]
    for blk in (slice(0, 3), slice(3, 7), slice(7, 30), slice(30, 34)):  # vb, qd, sd, q rows, each at its own scale
        scale = max(np.abs(want[blk]).max(), 1.0)
        assert np.abs(got[blk] - want[blk]).max() <= 1e-12 * scale
    assert np.abs(want[7:]).min() > 0.0
