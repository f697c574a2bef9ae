"""Closed forms of the least-squares cost rows of the contact kernel (hippopt_b200/csrc/kino_contact.cu,
"least-squares cost rows"), restated with numpy and checked against the row-by-row assembly of the 31 rows.

The 31 rows are linear residuals r = c^T z - ref with cost w r^2 (3 centroid rows, 4 foot-yaw rows, 24 force-ratio
rows), so the gradient is 2 w r c and the Hessian 2 sigma w c c^T.  The kernel sums them per variable and per local
Hessian entry, each lane owning a fixed set of entries taken from a host-built table (hb_kino_create, next to the
per-point table hc_pt).  This test builds that table from the layout's hc_index the way the host does, evaluates the
kernel's slot formulas and compares them with the rows assembled one by one."""
import itertools

import numpy as np
import pytest

from hippopt_b200.kino_layout import KinoLayout, KinoSettings
from hippopt_b200.robot_model import synthetic_ergocub

# kino_const.cuh: offsets inside one knot of z and of the knot's references
Z_P, Z_F, NZ, NCV = 6, 9, 189, 129
R_RATIO_L, R_YAW_L, R_RATIO_R, R_YAW_R, R_CW, R_CC, R_COUNT = 0, 4, 5, 9, 11, 14, 55


# every ordered triple of distinct points of one foot as (bottom-right, top-right, top-left): the yaw rows, the
# kernel's sign table and the host's per-lane table all follow the triple, and the layout is built with it
YAW_TRIPLES = list(itertools.permutations(range(4), 3))
_layouts = {}


def layout_for(yaw):
    if yaw not in _layouts:
        _layouts[yaw] = KinoLayout(synthetic_ergocub(), KinoSettings(horizon=4, yaw_points=yaw))
    return _layouts[yaw]


@pytest.fixture(scope="module")
def layout():
    return layout_for(KinoSettings().yaw_points)


def rows(z, ref, yaw, w_centroid, w_yaw, w_ratio):
    """the 31 rows as (variables, coefficients, weight, residual), in the kernel's row order"""
    out = []
    for c in range(3):
        var = [15 * i + Z_P + c for i in range(8)]
        out.append((var, [-0.125] * 8, w_centroid * ref[R_CW + c], ref[R_CC + c] - 0.125 * sum(z[v] for v in var)))
    for foot in range(2):
        for side in range(2):
            ang = ref[R_YAW_L if foot == 0 else R_YAW_R] + (np.pi / 2 if side else 0.0)
            sn, cs = np.sin(ang), np.cos(ang)
            pa, pb = (15 * (4 * foot + yaw[side + s]) + Z_P for s in range(2))
            var, cf = [pa, pa + 1, pb, pb + 1], [sn, -cs, -sn, cs]
            out.append((var, cf, 0.5 * w_yaw, sum(a * z[v] for v, a in zip(var, cf))))
    for foot in range(2):
        for i in range(4):
            for c in range(3):
                alpha = ref[(R_RATIO_L if foot == 0 else R_RATIO_R) + i]
                var = [15 * (4 * foot + j) + Z_F + c for j in range(4)]
                cf = [(1.0 if j == i else 0.0) - alpha for j in range(4)]
                out.append((var, cf, w_ratio, sum(a * z[v] for v, a in zip(var, cf))))
    return out


def assemble_rows(rs, hc_index, n_hc, sg):
    grad, hess = np.zeros(NZ), np.zeros(n_hc)
    for var, cf, w, r in rs:
        for v, a in zip(var, cf):
            grad[v] += 2.0 * w * r * a
        for a in range(len(var)):
            for b in range(a, len(var)):
                hess[hc_index[var[a], var[b]]] += 2.0 * sg * w * cf[a] * cf[b]
    return grad, hess


def host_table(hc_index, yaw):
    """api.cu, hb_kino_create: 8 local entries per lane (7 used), -1 where the lane has no entry"""
    P, F = Z_P, Z_F
    tab = -np.ones((32, 8), dtype=np.int64)
    entry = lambda pi, ci, pj, cj: hc_index[15 * pi + ci, 15 * pj + cj]
    for lane in range(32):
        for u in range(4):
            t = lane + 32 * u
            c, q = t // 36, t % 36
            a = q & 7
            if t < 108:
                tab[lane, u] = entry(a, P + c, (a + (q >> 3)) & 7, P + c)
        foot, i, j = lane >> 4, (lane >> 2) & 3, lane & 3
        on_row = any(i in (yaw[s], yaw[s + 1]) and j in (yaw[s], yaw[s + 1]) for s in range(2))
        if on_row:
            tab[lane, 4] = entry(4 * foot + i, P, 4 * foot + j, P + 1)
        for u in (5, 6):
            t = lane + 32 * (u - 5)
            foot, c, q = t // 30, (t // 10) % 3, t % 10
            a = q & 3
            if t < 60:
                tab[lane, u] = entry(4 * foot + a, F + c, 4 * foot + ((a + (q >> 2)) & 3), F + c)
    return tab


def closed_form(z, ref, yaw, w_centroid, w_yaw, w_ratio, sg, tab, n_hc):
    """the kernel's per-lane formulas: residuals on lanes 0..30, gradient of p_c / f_c of point v // 3 on lane v < 24,
    Hessian slots 0..6 of every lane"""
    rs = rows(z, ref, yaw, w_centroid, w_yaw, w_ratio)
    w = np.array([x[2] for x in rs] + [0.0])
    r = np.array([x[3] for x in rs] + [0.0])
    ang = [ref[R_YAW_L if f == 0 else R_YAW_R] + (np.pi / 2 if s else 0.0) for f in range(2) for s in range(2)]
    ysn, ycs = np.sin(ang), np.cos(ang)
    wy = 0.5 * w_yaw

    def ysgn(pt, side):
        q = pt & 3
        return 1.0 if q == yaw[side] else (-1.0 if q == yaw[side + 1] else 0.0)

    def alpha(foot):
        return ref[(R_RATIO_R if foot else R_RATIO_L):][:4]

    grad = np.zeros(NZ)
    for lane in range(24):
        pt, c = lane // 3, lane % 3
        foot = pt >> 2
        gp = 2.0 * w[c] * r[c] * -0.125
        if c < 2:
            for s in range(2):
                kk = ysn[2 * foot + s] if c == 0 else -ycs[2 * foot + s]
                gp += 2.0 * wy * r[3 + 2 * foot + s] * (ysgn(pt, s) * kk)
        grad[15 * pt + Z_P + c] += gp
        al = alpha(foot)
        grad[15 * pt + Z_F + c] += sum(2.0 * w_ratio * r[7 + 12 * foot + 3 * i + c] * ((i == (pt & 3)) - al[i])
                                       for i in range(4))
    hess = np.zeros(n_hc)
    tw = 2.0 * sg
    for lane in range(32):
        hv = np.zeros(7)
        for u in range(4):
            t = lane + 32 * u
            c, q = t // 36, t % 36
            a, a2 = q & 7, ((q & 7) + (q >> 3)) & 7
            i, j = min(a, a2), max(a, a2)
            foot = i >> 2
            v = tw * w[c & 3] * -0.125 * -0.125
            if c < 2 and foot == j >> 2:
                for s in range(2):
                    kk = ysn[2 * foot + s] if c == 0 else -ycs[2 * foot + s]
                    v += tw * wy * (ysgn(i, s) * kk) * (ysgn(j, s) * kk)
            hv[u] = v
        foot, i, j = lane >> 4, (lane >> 2) & 3, lane & 3
        hv[4] = sum(tw * wy * (ysgn(i, s) * ysn[2 * foot + s]) * (ysgn(j, s) * -ycs[2 * foot + s]) for s in range(2))
        for u in (5, 6):
            t = lane + 32 * (u - 5)
            foot, q = (t // 30) & 1, t % 10
            a, a2 = q & 3, ((q & 3) + (q >> 2)) & 3
            i, j = min(a, a2), max(a, a2)
            al = alpha(foot)
            hv[u] = sum(tw * w_ratio * ((m == i) - al[m]) * ((m == j) - al[m]) for m in range(4))
        for u in range(7):
            if tab[lane, u] >= 0:
                hess[tab[lane, u]] += hv[u]
    return grad, hess


def test_table_entries_are_distinct_and_cover_the_rows(layout):
    check_table(layout)


@pytest.mark.parametrize("yaw", YAW_TRIPLES)
def test_table_entries_for_every_yaw_triple(yaw):
    check_table(layout_for(yaw))


def check_table(layout):
    yaw = layout.st.yaw_points
    tab = host_table(layout.hc_index, yaw)
    used = tab[tab >= 0]
    assert len(used) == len(set(used.tolist())), "two lanes share a Hessian entry: the kernel would race"
    assert (tab[:, 7] < 0).all()
    touched = set()
    for var, cf, _, _ in rows(np.zeros(NZ), np.zeros(R_COUNT), yaw, 1.0, 1.0, 1.0):
        for a in range(len(var)):
            for b in range(a, len(var)):
                touched.add(int(layout.hc_index[var[a], var[b]]))
    assert -1 not in touched
    assert touched == set(used.tolist())


@pytest.mark.parametrize("seed", range(6))
def test_closed_form_matches_rows(layout, seed):
    check_closed_form(layout, seed)


@pytest.mark.parametrize("yaw", YAW_TRIPLES)
def test_closed_form_matches_rows_for_every_yaw_triple(yaw):
    for seed in (100, 101):
        check_closed_form(layout_for(yaw), seed)


def check_closed_form(layout, seed):
    rng = np.random.default_rng(seed)
    yaw = layout.st.yaw_points
    n_hc = layout.n_hc
    z = rng.normal(size=NZ)
    ref = rng.normal(size=R_COUNT)
    ref[[R_YAW_L, R_YAW_R]] = rng.uniform(-np.pi, np.pi, size=2)
    ref[R_RATIO_L:R_RATIO_L + 4] = rng.dirichlet(np.ones(4))
    ref[R_RATIO_R:R_RATIO_R + 4] = rng.dirichlet(np.ones(4))
    w_centroid, w_yaw, w_ratio = rng.uniform(0.1, 3000.0, size=3)
    sg = rng.uniform(0.01, 10.0)
    ref_g, ref_h = assemble_rows(rows(z, ref, yaw, w_centroid, w_yaw, w_ratio), layout.hc_index, n_hc, sg)
    tab = host_table(layout.hc_index, yaw)
    got_g, got_h = closed_form(z, ref, yaw, w_centroid, w_yaw, w_ratio, sg, tab, n_hc)
    np.testing.assert_allclose(got_g, ref_g, rtol=1e-14, atol=1e-14 * np.abs(ref_g).max())
    np.testing.assert_allclose(got_h, ref_h, rtol=1e-14, atol=1e-14 * np.abs(ref_h).max())
