"""The smooth-step terrain of the contact kernel (hippopt_b200/csrc/kino_smooth.cuh) where it is hard: on the edges,
corners and cut-off of both steps, where they overlap, deep inside and far away.

Two levels:
  * the surface jet T(x, y) (order 4) and the frame jets (TFrame) through `hb_debug_smooth_terrain`, against sympy's
    symbolic derivatives evaluated with mpmath at 40 digits, with a running error bound S of the kernel's own operation
    sequence as the tolerance;
  * the whole contact kernel (all five NLP outputs) with its contact points written onto those places, against the
    long-double oracle at 1e-10 in the parity metric, with no entry masked.

Surface: T = sum_s height_s exp(-g_s^20), g_s = (2 (x - ox_s) / l_s)^10 + (2 (y - oy_s) / w_s)^10, h = z - T."""
import math

import numpy as np
import pytest

EPS = 2.0 ** -52
TOL = 64.0  # |got - ref| <= TOL * EPS * S
G_BAND = (0.5, 0.8, 0.9, 0.95, 1.0, 1.05, 1.1, 1.2, 1.3)
CUTOFF = 1.42  # kino_smooth.cuh skips a step beyond g0 = 1.42, where exp(-g^20) < 2^-1075

# (l, w, height, ox, oy) x 2
PARAM_SETS = {
    "stairs": np.array([0.9, 0.8, 0.1, 0.675, 0.0, 0.405, 0.8, 0.1, 0.9, 0.0]),  # the workload's stairs
    "distinct": np.array([0.9, 0.8, 0.12, 0.675, 0.05, 0.5, 0.6, 0.07, 0.95, -0.08]),  # every parameter differs
    "steep": np.array([0.2, 0.1, 0.15, 0.0, 0.0, 0.2, 0.1, 0.15, 0.12, 0.04]),  # ill-conditioned tangent frame
    "zero_negative": np.array([0.9, 0.8, 0.0, 0.675, 0.0, 0.405, 0.6, -0.08, 0.9, 0.1]),
}

FIELDS = ["h", "gx", "gy", "n0", "n1", "n2", "xh0", "xh1", "xh2", "yh0", "yh1", "yh2",
          "Dn0x", "Dn0y", "Dn1x", "Dn1y", "Dn2x", "Dn2y"]
N_OUT = 15 + 10 * len(FIELDS)


def bidx(i, j):
    return (i + j) * (i + j + 1) // 2 + j


def jet_index(N):
    """(i, j) of every coefficient of an order-N bivariate jet, in storage order."""
    return [(o - j, j) for o in range(N + 1) for j in range(o + 1)]


# ------------------------------------------------------------------------------------------------------------------
# points
# ------------------------------------------------------------------------------------------------------------------
def step_g(tp, x, y):
    """(g, X^10, Y^10) of both steps, [2, n] each, in float64 (for the categories only)."""
    out = []
    for s in range(2):
        l, w, _, ox, oy = tp[..., 5 * s], tp[..., 5 * s + 1], tp[..., 5 * s + 2], tp[..., 5 * s + 3], tp[..., 5 * s + 4]
        gx, gy = (2 * (x - ox) / l) ** 10, (2 * (y - oy) / w) ** 10
        out.append((gx + gy, gx, gy))
    return tuple(np.stack([o[k] for o in out]) for k in range(3))


def categories(tp, x, y):
    """Boolean [n] per category, from the points and parameters alone."""
    g, gx, gy = step_g(tp, x, y)
    band = (g > 0.85) & (g < 1.15)
    return {
        "both_in_band": band.all(axis=0),
        "x_edge": (band & (gy < 1e-3)).any(axis=0),
        "y_edge": (band & (gx < 1e-3)).any(axis=0),
        "corner": (band & (np.minimum(gx, gy) > 0.1)).any(axis=0),
        "overlap": (g < 1.0).all(axis=0),
        "cutoff": (np.abs(g / CUTOFF - 1.0) < 1e-6).any(axis=0),
        "subnormal_exp": ((g > 1.385) & (g < 1.395)).any(axis=0),  # fp64 exp(-g^20) is subnormal there
        "interior": (g < 1e-3).any(axis=0),
        "far": (g > 1e6).all(axis=0),
    }


def _on_step(tp, s, X, Y):
    l, w, _, ox, oy = tp[5 * s:5 * s + 5]
    return ox + 0.5 * l * np.asarray(X), oy + 0.5 * w * np.asarray(Y)


def _band_curve_crossings(tp, per_set):
    """Points where both steps are in their band: step 2's band curves g2 in {0.9, 1, 1.1}, sampled densely, kept where
    g1 is in (0.9, 1.1)."""
    pts = []
    for g2 in (0.9, 1.0, 1.1):
        r = g2 ** 0.1
        t = np.linspace(-r, r, 20001)
        o = np.maximum(g2 - t ** 10, 0.0) ** 0.1
        for X, Y in ((t, o), (t, -o), (o, t), (-o, t)):
            x, y = _on_step(tp, 1, X, Y)
            g1 = step_g(tp, x, y)[0][0]
            pts += [(a, b) for a, b in zip(x[(g1 > 0.9) & (g1 < 1.1)], y[(g1 > 0.9) & (g1 < 1.1)])]
    pts = np.array(pts).reshape(-1, 2)
    if len(pts) > per_set:
        pts = pts[np.linspace(0, len(pts) - 1, per_set).astype(int)]
    return pts


def terrain_points(seed=0, n_random=120):
    """(tp [n, 10], xyz [n, 3], set name [n]) over the four parameter sets."""
    rng = np.random.default_rng(seed)
    TP, XY, NAME = [], [], []
    for name, tp in PARAM_SETS.items():
        xy = []
        for s in range(2):
            def add(X, Y):
                xy.append(np.stack(np.broadcast_arrays(*_on_step(tp, s, X, Y)), axis=-1).reshape(-1, 2))

            sg = np.array([1.0, -1.0])
            for g in G_BAND:
                for yo in (0.0, 0.3):  # x-edges, with and without a small y part
                    add(sg * (g - yo ** 10) ** 0.1, yo)
                    add(yo, sg * (g - yo ** 10) ** 0.1)  # y-edges
                for a in (0.5, 0.25):  # corners
                    X, Y = np.meshgrid(sg * (a * g) ** 0.1, sg * ((1 - a) * g) ** 0.1)
                    add(X.ravel(), Y.ravel())
            for g in (CUTOFF * (1 - 1e-9), CUTOFF * (1 + 1e-9), 1.39):
                add(sg * g ** 0.1, 0.0)
                add(sg * (g / 2) ** 0.1, sg * (g / 2) ** 0.1)
            add(np.array([0.0, 0.3, -0.5]), np.array([0.0, -0.2, 0.4]))  # interior
            g = rng.uniform(0.85, 1.15, n_random)  # random points in the band
            a = rng.uniform(0.0, 1.0, n_random)
            add(rng.choice(sg, n_random) * (a * g) ** 0.1, rng.choice(sg, n_random) * ((1 - a) * g) ** 0.1)
        xy.append(_band_curve_crossings(tp, 24))
        lo = min(tp[3] - tp[0], tp[8] - tp[5])
        hi = max(tp[3] + tp[0], tp[8] + tp[5])
        xy.append(np.array([[lo - 3.0, 0.0], [hi + 3.0, 0.1], [0.5 * (lo + hi), 3.0], [lo - 2.0, -3.0]]))  # far
        # overlap: the middle of the intersection of the two footprints
        cx = 0.5 * (max(tp[3] - tp[0] / 2, tp[8] - tp[5] / 2) + min(tp[3] + tp[0] / 2, tp[8] + tp[5] / 2))
        cy = 0.5 * (max(tp[4] - tp[1] / 2, tp[9] - tp[6] / 2) + min(tp[4] + tp[1] / 2, tp[9] + tp[6] / 2))
        xy.append(np.array([[cx, cy], [cx + 0.01 * tp[5], cy - 0.01 * tp[6]]]))
        xy = np.concatenate(xy)
        TP.append(np.repeat(tp[None], len(xy), axis=0))
        XY.append(xy)
        NAME += [name] * len(xy)
    XY = np.concatenate(XY)
    z = 0.01 + rng.uniform(-0.02, 0.02, len(XY))
    return np.concatenate(TP), np.concatenate([XY, z[:, None]], axis=1), np.array(NAME)


# ------------------------------------------------------------------------------------------------------------------
# symbolic reference (sympy derivatives, mpmath values)
# ------------------------------------------------------------------------------------------------------------------
_SYM = {}


def _symbolic():
    if _SYM:
        return _SYM
    import sympy as sp

    x, y, l, w, H, ox, oy = sp.symbols("x y l w height ox oy", real=True)
    T = H * sp.exp(-((2 * (x - ox) / l) ** 10 + (2 * (y - oy) / w) ** 10) ** 20)
    surf = []
    for i, j in jet_index(4):
        e = T
        if i:
            e = sp.diff(e, x, i)
        if j:
            e = sp.diff(e, y, j)
        surf.append(e / (math.factorial(i) * math.factorial(j)))
    _SYM["surface"] = sp.lambdify((x, y, l, w, H, ox, oy), surf, modules="mpmath", cse=True)

    # the frame as a function of the derivatives t_ij of an abstract T(x, y): n = grad h / |grad h| with
    # grad h = (-T_x, -T_y, 1), y0 = n x e_x, x0 = y0 x n, xh = x0 / |x0|, yh = n x xh  (Terrain.orientation)
    t = {ij: sp.Symbol(f"t{ij[0]}{ij[1]}") for ij in jet_index(4)[1:]}

    def D(e, axis):  # total derivative in x (axis 0) or y (axis 1)
        return sum(sp.diff(e, s) * t[(i + 1, j) if axis == 0 else (i, j + 1)] for (i, j), s in t.items() if i + j < 4)

    def cross(a, b):
        return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]

    gx, gy = -t[(1, 0)], -t[(0, 1)]
    nr = sp.sqrt(gx ** 2 + gy ** 2 + 1)
    n = [gx / nr, gy / nr, 1 / nr]
    x0 = cross(cross(n, [1, 0, 0]), n)
    xn = sp.sqrt(sum(c ** 2 for c in x0))
    xh = [c / xn for c in x0]
    yh = cross(n, xh)

    def derivs(e, order):
        d = {(0, 0): e}
        for i, j in jet_index(order)[1:]:
            d[(i, j)] = D(d[(i - 1, j)], 0) if i > 0 else D(d[(i, j - 1)], 1)
        return d

    exprs, keys = [], []
    for name, comps, order in (("n", n, 3), ("xh", xh, 2), ("yh", yh, 2)):
        for a, c in enumerate(comps):
            for ij, e in derivs(c, order).items():
                exprs.append(e)
                keys.append((name, a, ij))
    _SYM["frame"] = sp.lambdify(list(t.values()), exprs, modules="mpmath", cse=True)
    _SYM["frame_keys"] = {k: q for q, k in enumerate(keys)}
    return _SYM


def reference(tp, xyz, dps=40):
    """[n, N_OUT] exact values of hb_debug_smooth_terrain's outputs, as (hi, lo) float64 pairs: hi + lo is the
    40-digit value to 2^-106 relative."""
    import mpmath

    sym = _symbolic()
    surface, frame, fk = sym["surface"], sym["frame"], sym["frame_keys"]
    f = math.factorial
    hi = np.zeros((len(xyz), N_OUT))
    lo = np.zeros((len(xyz), N_OUT))
    with mpmath.workdps(dps):
        mp = mpmath.mpf
        for p in range(len(xyz)):
            x, y, z = (mp(float(v)) for v in xyz[p])
            Tn = [mp(0)] * 15
            for s in range(2):
                c = surface(x, y, *(mp(float(v)) for v in tp[p, 5 * s:5 * s + 5]))
                Tn = [a + b for a, b in zip(Tn, c)]
            raw = {ij: Tn[q] * f(ij[0]) * f(ij[1]) for q, ij in enumerate(jet_index(4))}
            fr = frame(*(raw[ij] for ij in jet_index(4)[1:]))
            out = list(Tn)

            def tj(c):  # bivariate order-2 coefficients {(i, j): v} -> the 10 trivariate coefficients
                return [c[(0, 0)], c[(1, 0)], c[(0, 1)], mp(0), c[(2, 0)], c[(1, 1)], mp(0), c[(0, 2)], mp(0), mp(0)]

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
            for q, v in enumerate(out):
                hi[p, q] = float(v)
                lo[p, q] = float(v - mp(hi[p, q]))
    return hi, lo


# ------------------------------------------------------------------------------------------------------------------
# running error bound of the kernel's operation sequence
# ------------------------------------------------------------------------------------------------------------------
U = 2.0 ** -53
LAM = 2.0 ** -1022  # in units of u: u * 2^-1022 = 2^-1075 is the absolute error of an operation in underflow


class R:
    """A float64 value and a bound e on its rounding error in units of u = 2^-53 (Higham's running error analysis:
    every operation adds |result| for its own rounding, products and quotients also LAM for gradual underflow; errors
    of the operands propagate through the operation's partial derivatives).  Products keep the second-order term
    u e_a e_b: where two steps' gradients cancel exactly, n_x and n_y are nothing but rounding and x0[1] = -n_x n_y
    is their product."""

    __slots__ = ("v", "e")

    def __init__(self, v, e):
        self.v, self.e = v, e

    @staticmethod
    def of(c, exact=True):
        c = np.float64(c)
        return R(c, np.float64(0.0) if exact else abs(c))

    def __add__(a, b):
        b = b if isinstance(b, R) else R.of(b)
        v = a.v + b.v
        return R(v, a.e + b.e + abs(v))

    __radd__ = __add__

    def __sub__(a, b):
        b = b if isinstance(b, R) else R.of(b)
        v = a.v - b.v
        return R(v, a.e + b.e + abs(v))

    def __neg__(a):
        return R(-a.v, a.e)

    def __mul__(a, b):
        b = b if isinstance(b, R) else R.of(b)
        v = a.v * b.v
        return R(v, (abs(a.v) + U * a.e) * b.e + abs(b.v) * a.e + abs(v) + LAM)

    __rmul__ = __mul__

    def __truediv__(a, b):
        b = b if isinstance(b, R) else R.of(b)
        v = a.v / b.v
        return R(v, (a.e + abs(v) * b.e) / abs(b.v) + abs(v) + LAM)


def r_sqrt(a):
    v = np.sqrt(a.v)
    return R(v, a.e / (2 * v) + abs(v))


def r_exp(a):
    v = np.exp(a.v)
    return R(v, abs(v) * a.e + 2 * abs(v) + LAM)  # CUDA's exp: at most 1 ulp


def j_const(N, c):
    return [R.of(c)] + [R.of(0.0) for _ in range(1, (N + 1) * (N + 2) // 2)]


def j_mul(a, b, N):
    r = j_const(N, 0.0)
    for i1 in range(N + 1):
        for j1 in range(N + 1 - i1):
            for i2 in range(N + 1 - i1 - j1):
                for j2 in range(N + 1 - i1 - j1 - i2):
                    k = bidx(i1 + i2, j1 + j2)
                    r[k] = r[k] + a[bidx(i1, j1)] * b[bidx(i2, j2)]
    return r


def j_compose(a, f, N):
    d = [R.of(0.0)] + list(a[1:])
    r = j_const(N, 0.0)
    r[0] = f[N]
    for k in range(N - 1, -1, -1):
        r = j_mul(r, d, N)
        r[0] = r[0] + f[k]
    return r


def j_invsqrt(a, N):
    s = a[0]
    f0 = R.of(1.0) / r_sqrt(s)
    inv = R.of(1.0) / s
    f1 = (-0.5 * f0) * inv
    f2 = (-0.75 * f1) * inv
    f3 = (R.of(-(5.0 / 6.0), exact=False) * f2) * inv
    f4 = (-0.875 * f3) * inv
    return j_compose(a, [f0, f1, f2, f3, f4], N)


def j_d(a, N, axis):
    r = j_const(N - 1, 0.0)
    for i, j in jet_index(N - 1):
        r[bidx(i, j)] = float(i + 1 if axis == 0 else j + 1) * a[bidx(i + 1, j) if axis == 0 else bidx(i, j + 1)]
    return r


def j_add(a, b):
    return [p + q for p, q in zip(a, b)]


def j_sub(a, b):
    return [p - q for p, q in zip(a, b)]


def j_neg(a):
    return [-p for p in a]


def j_trunc(a, M):
    return list(a[:(M + 1) * (M + 2) // 2])


def bound_surface(tp, x, y):
    """The operations of smooth_steps_surface; a step beyond the cut-off contributes below 2^-1075 (LAM)."""
    T = j_const(4, 0.0)
    for s in range(2):
        l, w, height, ox, oy = (R.of(tp[:, 5 * s + k]) for k in range(5))
        dX, dY = R.of(2.0) / l, R.of(2.0) / w
        X0, Y0 = dX * (R.of(x) - ox), dY * (R.of(y) - oy)
        X2 = X0 * X0
        X4 = X2 * X2
        X6 = X4 * X2
        Y2 = Y0 * Y0
        Y4 = Y2 * Y2
        Y6 = Y4 * Y2
        g = j_const(4, 0.0)
        g[0] = X6 * X4 + Y6 * Y4
        g[bidx(1, 0)] = R.of(10.0) * X6 * X2 * X0 * dX
        g[bidx(2, 0)] = R.of(45.0) * X6 * X2 * dX * dX
        g[bidx(3, 0)] = R.of(120.0) * X6 * X0 * dX * dX * dX
        g[bidx(4, 0)] = R.of(210.0) * X6 * dX * dX * dX * dX
        g[bidx(0, 1)] = R.of(10.0) * Y6 * Y2 * Y0 * dY
        g[bidx(0, 2)] = R.of(45.0) * Y6 * Y2 * dY * dY
        g[bidx(0, 3)] = R.of(120.0) * Y6 * Y0 * dY * dY * dY
        g[bidx(0, 4)] = R.of(210.0) * Y6 * dY * dY * dY * dY
        keep = g[0].v <= CUTOFF
        g0 = g[0]
        with np.errstate(all="ignore"):
            g2 = g0 * g0
            g4 = g2 * g2
            g8 = g4 * g4
            g16 = g8 * g8
            fp = [g16 * g4, R.of(20.0) * g16 * g2 * g0, R.of(190.0) * g16 * g2, R.of(1140.0) * g16 * g0,
                  R.of(4845.0) * g16]
            G = j_compose(g, fp, 4)
            e0 = r_exp(-G[0])
            fe = [e0, e0, e0 / 2.0, e0 / 6.0, e0 / 24.0]
            E = j_compose(j_neg(G), fe, 4)
            C = [height * c for c in E]
        C = [R(np.where(keep, c.v, 0.0), np.where(keep, c.e, LAM)) for c in C]
        T = j_add(T, C)
    return T


def tj_from(b):
    z = R.of(0.0)
    return [b[0], b[1], b[2], z, b[3], b[4], z, b[5], z, z]


def bound(tp, xyz):
    """[n, N_OUT] float64 values and running error bounds S (in units of eps = 2^-52) of the kernel's outputs."""
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    T = bound_surface(tp, x, y)
    gx3, gy3 = j_neg(j_d(T, 4, 0)), j_neg(j_d(T, 4, 1))
    s = j_add(j_mul(gx3, gx3, 3), j_mul(gy3, gy3, 3))
    s[0] = s[0] + 1.0
    inv3 = j_invsqrt(s, 3)
    n3 = [j_mul(gx3, inv3, 3), j_mul(gy3, inv3, 3), inv3]
    n2 = [j_trunc(c, 2) for c in n3]
    x0 = [j_add(j_mul(n2[2], n2[2], 2), j_mul(n2[1], n2[1], 2)), j_neg(j_mul(n2[0], n2[1], 2)),
          j_neg(j_mul(n2[0], n2[2], 2))]
    xi = j_invsqrt(j_add(j_add(j_mul(x0[0], x0[0], 2), j_mul(x0[1], x0[1], 2)), j_mul(x0[2], x0[2], 2)), 2)
    xh = [j_mul(c, xi, 2) for c in x0]
    yh = [j_sub(j_mul(n2[1], xh[2], 2), j_mul(n2[2], xh[1], 2)), j_sub(j_mul(n2[2], xh[0], 2), j_mul(n2[0], xh[2], 2)),
          j_sub(j_mul(n2[0], xh[1], 2), j_mul(n2[1], xh[0], 2))]
    h = tj_from(j_neg(j_trunc(T, 2)))
    h[0] = h[0] + R.of(z)
    h[3] = R.of(1.0)
    out = list(T) + h + tj_from(j_trunc(gx3, 2)) + tj_from(j_trunc(gy3, 2))
    for c in n2 + xh + yh:
        out += tj_from(c)
    for a in range(3):
        out += tj_from(j_d(n3[a], 3, 0)) + tj_from(j_d(n3[a], 3, 1))
    n = len(x)
    V = np.stack([np.broadcast_to(r.v, (n,)) for r in out], axis=1)
    S = np.stack([np.broadcast_to(r.e, (n,)) for r in out], axis=1) / 2.0  # units of u -> units of eps
    return V, S


def field_of_column():
    return ["T"] * 15 + [f for f in FIELDS for _ in range(10)]


def ratios(got, hi, lo, S):
    """|got - ref| / (eps S), elementwise."""
    with np.errstate(divide="ignore", invalid="ignore"):
        d = np.abs((got - hi) - lo)
        r = d / (EPS * S)
    return np.where(d == 0.0, 0.0, r)


def report(r, names=None):
    cols = np.array(field_of_column())
    worst = {}
    for f in ["T"] + FIELDS:
        rf = r[:, cols == f]
        worst[f] = float(rf.max())
    print("worst |got - ref| / (eps S) per field:", {k: f"{v:.3g}" for k, v in worst.items()})
    if names is not None:
        for nm in PARAM_SETS:
            print(f"  {nm}: worst {float(r[names == nm].max()):.3g}")
    return worst


@pytest.fixture(scope="module")
def terrain_case():
    tp, xyz, names = terrain_points()
    hi, lo = reference(tp, xyz)
    V, S = bound(tp, xyz)
    return tp, xyz, names, hi, lo, V, S


def test_point_plan_covers_every_category(terrain_case):
    """Each category is populated in every parameter set (far and overlap apart, which depend on the set)."""
    tp, xyz, names = terrain_case[:3]
    cat = categories(tp, xyz[:, 0], xyz[:, 1])
    print("points:", len(xyz), {k: int(v.sum()) for k, v in cat.items()})
    for k, v in cat.items():
        assert v.sum() > 0, k
        for nm in PARAM_SETS:
            assert v[names == nm].any(), (k, nm)
    assert len(xyz) >= 2000
    assert np.isfinite(terrain_case[3]).all()


def test_error_bound_holds_for_a_float64_evaluation(terrain_case):
    """The bound is a bound: a float64 evaluation of the kernel's own operation sequence (numpy, without FMA; beyond the
    cut-off a step is dropped, as in the kernel) stays within TOL eps S of the symbolic reference everywhere."""
    tp, xyz, names, hi, lo, V, S = terrain_case
    assert np.isfinite(V).all() and np.isfinite(S).all() and (S >= 0).all()
    r = ratios(V, hi, lo, S)
    worst = report(r, names)
    assert max(worst.values()) <= TOL


@pytest.mark.gpu
def test_kernel_surface_and_frame_against_symbolic_reference(terrain_case, built_library):
    import torch

    from hippopt_b200 import _capi

    tp, xyz, names, hi, lo, V, S = terrain_case
    dev = torch.device("cuda:0")
    TP, P = (torch.tensor(np.ascontiguousarray(a), device=dev) for a in (tp, xyz))
    out = torch.full((len(xyz), N_OUT), float("nan"), dtype=torch.float64, device=dev)
    _capi.check(built_library.hb_debug_smooth_terrain(TP.data_ptr(), P.data_ptr(), len(xyz), out.data_ptr(), None),
                "hb_debug_smooth_terrain")
    torch.cuda.synchronize()
    assert _capi.H["HB_SMOOTH_TERRAIN_OUT"] == N_OUT
    got = out.cpu().numpy()
    assert np.isfinite(got).all()
    r = ratios(got, hi, lo, S)
    report(r, names)
    cat = categories(tp, xyz[:, 0], xyz[:, 1])
    print("worst per category:", {k: f"{float(r[v].max()):.3g}" for k, v in cat.items()})
    cols = np.array(field_of_column())
    bad = np.argwhere(r > TOL)
    assert len(bad) == 0, (f"{len(bad)} coefficients beyond {TOL} eps S; first: point {bad[0][0]} "
                           f"({names[bad[0][0]]}, xyz {xyz[bad[0][0]]}) field {cols[bad[0][1]]} col {bad[0][1]}: "
                           f"got {got[tuple(bad[0])]:.17g} ref {hi[tuple(bad[0])]:.17g} S {S[tuple(bad[0])]:.3g}")


# ------------------------------------------------------------------------------------------------------------------
# the whole contact kernel at those points
# ------------------------------------------------------------------------------------------------------------------
def _entry_errors(got, ref, jp, hp, x):
    """Per-entry errors of oracle/parity.py's metric (the same floors as its check_* functions)."""
    from oracle import parity

    ref = {k: np.asarray(v, dtype=np.float64) for k, v in ref.items()}
    m = ref["g"].shape[1]
    jrow = np.asarray(jp[1])
    Sj = parity.jac_row_scale(ref["jac"], jrow, m)
    xs = np.maximum(1.0, np.abs(x).max(axis=1, keepdims=True))
    Sh, col = parity.hess_var_scale(ref["hess"], hp[0], hp[1])
    with np.errstate(all="ignore"):
        return {
            "grad_f": parity._rel(got["grad_f"], ref["grad_f"], np.abs(ref["grad_f"]).max(axis=1, keepdims=True)),
            "g": parity._rel(got["g"], ref["g"], Sj * xs),
            "jac": parity._rel(got["jac"], ref["jac"], Sj[:, jrow]),
            "hess": parity._rel(got["hess"], ref["hess"], np.sqrt(Sh[:, col] * Sh[:, np.asarray(hp[1])])),
        }


@pytest.mark.gpu
def test_contact_kernel_at_the_terrain_edges_against_long_double_oracle(model, built_library, terrain_case):
    import torch

    from hippopt_b200.evaluator import ALL, KinoEvaluator
    from hippopt_b200.kino_layout import NPT, NZ, P, KinoSettings
    from hippopt_b200.workloads import kino_batch
    from oracle import expressions as ex
    from oracle import kinodynamic as kd
    from oracle import parity

    N, B = 4, 8
    ev = KinoEvaluator(model, KinoSettings(horizon=N, terrain="smooth_steps", n_terrain_params=10,
                                           final_state_constraint=True))
    lay = ev.layout
    x, p, lam, _ = kino_batch(lay, model, B, seed=91, noise=0.05)
    sigma = np.linspace(0.25, 3.0, B)
    tp_all, xyz_all, names = terrain_case[:3]
    rng = np.random.default_rng(5)
    sets = list(PARAM_SETS)
    pos = np.zeros((B, N, NPT, 2))
    for b in range(B):
        nm = sets[b % len(sets)]
        p[b, lay.po.terrain:lay.po.terrain + 10] = PARAM_SETS[nm]
        idx = np.flatnonzero(names == nm)
        cat = categories(tp_all[idx], xyz_all[idx, 0], xyz_all[idx, 1])
        # one point of every category the set has, the rest from its band, each point once
        pick = [int(idx[rng.choice(np.flatnonzero(v))]) for v in cat.values() if v.any()]
        band = idx[(step_g(tp_all[idx], xyz_all[idx, 0], xyz_all[idx, 1])[0] < 1.2).any(axis=0)]
        rest = [int(i) for i in rng.permutation(band) if int(i) not in pick]
        pick = (pick + rest)[:N * NPT]
        pos[b] = xyz_all[pick, :2].reshape(N, NPT, 2)
    tp = p[:, lay.po.terrain:lay.po.terrain + 10]
    for k in range(N):
        for i in range(NPT):
            c = NZ * k + 15 * i + P
            x[:, c:c + 2] = pos[:, k, i]
            with np.errstate(all="ignore"):
                g = step_g(tp, pos[:, k, i, 0], pos[:, k, i, 1])[0]
                T = sum(np.where(g[s] <= CUTOFF, tp[:, 5 * s + 2] * np.exp(-np.minimum(g[s], CUTOFF) ** 20), 0.0)
                        for s in range(2))
            x[:, c + 2] = T + rng.uniform(-0.02, 0.02, B)
    TPb = np.repeat(tp[:, None], N * NPT, axis=1).reshape(-1, 10)
    cat = categories(TPb, pos[..., 0].ravel(), pos[..., 1].ravel())
    print("contact points per category:", {k: int(v.sum()) for k, v in cat.items()})
    for k, v in cat.items():
        assert v.any(), f"no contact point in category {k}"

    nlp, _ = kd.build(model, kd.Settings(horizon=N, terrain=ex.TwoSmoothSteps(), terrain_params=10,
                                         final_state_constraint=True))
    jp, hp = nlp.jac_structure()[:2], nlp.hess_structure()[:2]
    assert np.array_equal(ev.jac_sparsity()[1], jp[1]) and np.array_equal(ev.hess_sparsity()[1], hp[1])
    t = [torch.tensor(np.ascontiguousarray(a), device="cuda:0") for a in (x, p, lam, sigma)]
    out = ev.eval(ALL, *t)
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy().copy() for k, v in out.items()}
    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble)
    for k, v in ref.items():
        assert np.isfinite(v).all(), f"long-double reference not finite in {k}"
        assert np.isfinite(got[k]).all(), k
    worst = parity.check_all(got, ref, jp, hp, x, rtol=parity.RTOL)
    print("worst relative error per output:", {k: f"{v:.2e}" for k, v in worst.items()})

    # per category: the entries that depend on a point's position (its columns of jac_g / grad_f / hess_l, the rows
    # of g with an entry in those columns)
    err = _entry_errors(got, ref, jp, hp, x)
    jcol = np.repeat(np.arange(len(jp[0]) - 1), np.diff(jp[0]))
    hcol = np.repeat(np.arange(len(hp[0]) - 1), np.diff(hp[0]))
    hrow, jrow = np.asarray(hp[1]), np.asarray(jp[1])
    per_cat = {}
    for name, v in cat.items():
        worst_c = {"grad_f": 0.0, "g": 0.0, "jac": 0.0, "hess": 0.0}
        for q in np.flatnonzero(v):
            b, r = divmod(q, N * NPT)
            k, i = divmod(r, NPT)
            cols = NZ * k + 15 * i + P + np.arange(3)
            je = np.isin(jcol, cols)
            he = np.isin(hcol, cols) | np.isin(hrow, cols)
            rows = np.unique(jrow[je])
            worst_c["grad_f"] = max(worst_c["grad_f"], float(err["grad_f"][b, cols].max()))
            worst_c["jac"] = max(worst_c["jac"], float(err["jac"][b, je].max()))
            worst_c["hess"] = max(worst_c["hess"], float(err["hess"][b, he].max()))
            worst_c["g"] = max(worst_c["g"], float(err["g"][b, rows].max()))
        per_cat[name] = worst_c
        print(f"  {name:14s}", {k2: f"{v2:.2e}" for k2, v2 in worst_c.items()})
