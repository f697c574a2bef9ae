"""Layout compiler for the humanoid kinodynamic multiple-shooting NLP.

Reproduces, without CasADi, the orderings the reference's graph construction fixes:

* decision vector ``x`` = ``opti.variable`` creation order = depth-first dataclass field order of
  the horizon-expanded ``Variables`` (`/root/reference/src/hippopt/base/opti_solver.py:303-310`,
  `turnkey_planners/humanoid_kinodynamic/variables.py:121-301`; SURVEY.md Appendix B.1),
* parameter vector ``p`` likewise (Appendix B.2),
* constraint rows ``g`` in ``subject_to`` call order, i.e. FAMILY-major / knot-minor
  (`turnkey_planners/humanoid_kinodynamic/planner.py:124-176`,
  `base/multiple_shooting_solver.py:703-742, 807-824`; Appendix B.3),
* the structural CCS patterns of ``jac_g`` and the upper-triangular ``hess_l`` (what CasADi derives by
  dependency propagation [ext]); here from per-family structural rules.

and emits the scatter maps the CUDA kernels (csrc/kinodynamic.cu) use: every kernel produces its
values in a fixed *kernel-local* order per knot, and ``map[k][e]`` is the CCS slot of local entry
``e`` of knot ``k`` (``-1``: the entry does not exist at this knot).

Local Jacobian orders (``z`` = the 189 variables of column-knot k):
  contact kernel (JC): see :meth:`KinoLayout._enumerate_jc`;  kinematics kernel (JK): `_enumerate_jk`.
Local Hessian orders: contact kernel (HC) routes (var_i, var_j) pairs of its 129 variables through
the lookup table ``hc_index``;  kinematics kernel (HK): direction-major ``j * 57 + i`` (27 directions
(q, s) x 57 rows (vb, qd, sd, q, s)), plus 27 velocity-diagonal entries (HK2).
"""
from __future__ import annotations

import dataclasses

import numpy as np

from .robot_model import RobotModel

NZ = 189
NJ = 23
NPT = 8
V, FD, P, F, U = 0, 3, 6, 9, 12
VB, QD, PB, Q, SD, S, COM, H = 120, 123, 127, 130, 134, 157, 180, 183
# contact-kernel variable set for the Hessian lookup: 8 x 15 point vars, com(3), h(6)
NCV = 129

SKEW_PAIRS = [(0, 1), (0, 2), (1, 0), (1, 2), (2, 0), (2, 1)]


# terrain name -> kernel terrain (HB_KI_TERRAIN).  "smooth_steps": the two axis-aligned flat steps of the stairs, ten
# parameters (l, w, height, ox, oy) x 2; "tilted_steps": K >= 1 general steps (yaw, origin height, tilted top), 10 K
# parameters (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) per step.  The terrain parameters close p.
TERRAINS = {"planar": 0, "smooth_steps": 1, "tilted_steps": 2}


def kernel_terrain(terrain: str, n_terrain_params: int) -> int:
    """The kernel terrain of a terrain name, after checking that the parameter count fits it."""
    if terrain not in TERRAINS:
        raise ValueError(f"terrain must be one of {sorted(TERRAINS)}, not {terrain!r}")
    n = n_terrain_params
    if terrain == "planar" and n != 0:
        raise ValueError("the planar terrain takes no terrain parameters")
    if terrain == "smooth_steps" and n != 10:
        raise ValueError("the smooth steps take 10 terrain parameters")
    if terrain == "tilted_steps" and (n < 10 or n % 10 != 0):
        raise ValueError(f"tilted_steps takes 10 parameters per step (a positive multiple of 10), not {n}")
    return TERRAINS[terrain]


@dataclasses.dataclass
class KinoSettings:
    """Numeric settings; defaults = `main_single_step_flat_ground.py:54-104` (BASELINE config 3)."""

    horizon: int = 30
    terrain: str = "planar"  # one of TERRAINS
    n_terrain_params: int = 0
    final_state_constraint: bool = False
    periodicity_constraint: bool = False
    foot_frames: tuple = ("l_sole", "r_sole")
    frame_quaternion_cost_frame: str = "chest"
    joint_regularization_cost_weights: np.ndarray = dataclasses.field(
        default_factory=lambda: np.concatenate([0.1 * np.ones(3), 10.0 * np.ones(8), np.ones(12)])
    )
    com_linear_velocity_cost_weights: tuple = (10.0, 0.1, 1.0)
    contacts_centroid_cost_multiplier: float = 100.0
    com_linear_velocity_cost_multiplier: float = 1.0
    desired_frame_quaternion_cost_multiplier: float = 90.0
    base_quaternion_cost_multiplier: float = 50.0
    base_quaternion_velocity_cost_multiplier: float = 0.001
    joint_regularization_cost_multiplier: float = 0.1
    force_regularization_cost_multiplier: float = 10.0
    foot_yaw_regularization_cost_multiplier: float = 2000.0
    swing_foot_height_cost_multiplier: float = 1000.0
    contact_velocity_control_cost_multiplier: float = 5.0
    contact_force_control_cost_multiplier: float = 0.0001
    yaw_points: tuple = (2, 3, 0)  # bottom-right, top-right, top-left of rectangular_foot()


class ParamOffsets:
    """Offsets inside p (Appendix B.2)."""

    def __init__(self, N: int, n_terrain: int = 0):
        o = 0
        self.desc0 = o
        o += 24 * N
        self.mass, self.plm, self.pld = o, o + 1, o + 2
        o += 3
        self.init = o
        o += 105
        self.final = o
        o += 105
        self.dt = o
        o += 1
        self.gravity = o
        o += 6
        self.kt, self.k_bs, self.eps, self.mu = o, o + 1, o + 2, o + 3
        o += 4
        self.max_u = o
        o += 3
        self.max_fd = o
        o += 3
        self.max_L, self.min_com_h, self.min_feet_d, self.max_feet_h = o, o + 1, o + 2, o + 3
        o += 4
        self.max_s, self.min_s, self.max_sd, self.min_sd = o, o + NJ, o + 2 * NJ, o + 3 * NJ
        o += 4 * NJ
        self.refs0 = o
        o += 55 * N
        self.terrain = o
        o += n_terrain
        self.n_p = o

    # initial/final state sub-offsets
    @staticmethod
    def st_pt(i, what):
        return 9 * i + {"p": 0, "f": 3, "desc": 6}[what]

    ST_PB, ST_Q, ST_S, ST_COM = 72, 75, 79, 102
    # references sub-offsets
    R_RATIO_L, R_YAW_L, R_RATIO_R, R_YAW_R, R_SWING = 0, 4, 5, 9, 10
    R_CW, R_CC, R_COMV, R_FQ, R_BQ, R_BQV, R_JR = 11, 14, 17, 20, 24, 28, 32


# linear-dynamics state scalars in family emission order: (state offset, rate offset, length)
def linear_states():
    out = []
    for i in range(NPT):
        out.append((15 * i + F, 15 * i + FD, 3))
        out.append((15 * i + P, 15 * i + V, 3))
    out += [(PB, VB, 3), (Q, QD, 4), (S, SD, NJ), (COM, H, 3)]
    return out


def count_rows(horizon: int, final_state: bool, periodicity: bool) -> int:
    """m of the kinodynamic OCP from its constraint families alone (no robot model needed): template matching."""
    lay = KinoLayout.__new__(KinoLayout)
    lay.N = horizon
    lay.st = KinoSettings(horizon=horizon, final_state_constraint=final_state, periodicity_constraint=periodicity)
    lay._families()
    return lay.m


class KinoLayout:
    def __init__(self, model: RobotModel, settings: KinoSettings):
        self.model = model
        self.st = settings
        self.kernel_terrain = kernel_terrain(settings.terrain, settings.n_terrain_params)
        N = self.N = settings.horizon
        self.knot_size = NZ  # variables per knot (stage size of the KKT sweep)
        self.n_x = NZ * N + 6
        self.po = ParamOffsets(N, settings.n_terrain_params)
        self.n_p = self.po.n_p
        self.h_init = NZ * N
        self.smooth = settings.terrain != "planar"
        self._families()
        self._patterns()

    # ------------------------------------------------------------------ rows
    def _families(self):
        N = self.N
        self.fam: dict[str, tuple[int, int, int, int]] = {}
        m = 0

        def add(name, rows, k0, k1):
            nonlocal m
            self.fam[name] = (m, rows, k0, k1)
            m += rows * (k1 - k0 + 1)

        for i in range(NPT):
            add(f"pt{i}.f_ic", 3, 0, 0)
            add(f"pt{i}.f_dyn", 3, 1, N - 1)
            add(f"pt{i}.p_ic", 3, 0, 0)
            add(f"pt{i}.p_dyn", 3, 1, N - 1)
            add(f"pt{i}.planar", 3, 0, N - 1)
            add(f"pt{i}.dcc", 1, 0, N - 1)
            add(f"pt{i}.height", 1, 1, N - 1)
            add(f"pt{i}.normal", 1, 1, N - 1)
            add(f"pt{i}.friction", 1, 1, N - 1)
            add(f"pt{i}.u_bounds", 3, 0, N - 1)
            add(f"pt{i}.fd_bounds", 3, 0, N - 1)
            add(f"pt{i}.fk", 3, 1, N - 1)
        for name, n in (("pb", 3), ("q", 4), ("s", NJ), ("com", 3)):
            add(f"{name}_ic", n, 0, 0)
            add(f"{name}_dyn", n, 1, N - 1)
        if not self.st.periodicity_constraint:
            add("h_ic", 6, 0, 0)
        add("h_dyn", 6, 1, N - 1)
        add("unit_quat", 1, 1, N - 1)
        add("com_kin", 3, 1, N - 1)
        add("mom_kin", 3, 0, N - 1)
        add("L_bounds", 3, 0, N - 1)
        add("com_height", 1, 1, N - 1)
        add("feet_dist", 1, 1, N - 1)
        add("s_bounds", NJ, 1, N - 1)
        add("sd_bounds", NJ, 0, N - 1)
        if self.st.final_state_constraint:
            add("final", 105, N - 1, N - 1)
        add("feet_relh", 1, 1, N - 1)
        if self.st.periodicity_constraint:
            add("periodicity", 84, 0, 0)
        self.m = m

    def row(self, name: str, k: int, r: int = 0) -> int:
        """Global g index of local row r of family ``name`` at knot k, or -1 if absent."""
        if name not in self.fam:
            return -1
        base, rows, k0, k1 = self.fam[name]
        if k < k0 or k > k1:
            return -1
        return base + (k - k0) * rows + r

    def row_base(self, name: str) -> tuple[int, int, int]:
        """(offset of knot 0's virtual slot, rows per knot, first knot) for the device tables."""
        if name not in self.fam:
            return (-1, 0, 1 << 30)
        base, rows, k0, k1 = self.fam[name]
        return (base - k0 * rows, rows, k0)

    # final-state rows: alphabetical leaf order (optimization_object.py:305-306)
    def final_rows(self):
        """List of (local row, x offset inside the last knot or -1 for parameter-only rows)."""
        out = []
        r = 0
        for c in range(3):
            out.append((r, COM + c))
            r += 1
        for i in range(NPT):
            for c in range(3):
                out.append((r, -1))  # descriptor.position_in_foot_frame: parameter-only row
                r += 1
            for c in range(3):
                out.append((r, 15 * i + F + c))
                r += 1
            for c in range(3):
                out.append((r, 15 * i + P + c))
                r += 1
        for off, n in ((PB, 3), (Q, 4), (S, NJ)):
            for c in range(n):
                out.append((r, off + c))
                r += 1
        assert r == 105
        return out

    def periodicity_vars(self):
        out = []
        for i in range(NPT):
            out += [15 * i + U + c for c in range(3)] + [15 * i + FD + c for c in range(3)]
        out += [H + c for c in range(6)] + [VB + c for c in range(3)] + [QD + c for c in range(4)]
        out += [SD + c for c in range(NJ)]
        assert len(out) == 84
        return out

    # ------------------------------------------------------------------ bounds (host side)
    def simple_bound_rows(self, include_equalities: bool = False):
        """Rows of g that are a bare decision variable, g_i = x_j -- the rows CasADi's nlpsol option
        ``detect_simple_bounds`` (set by every main of the reference, e.g. main_single_step_flat_ground.py:106) turns
        into lbx / ubx and removes from g [ext].  Returns (rows, x index of each row).

        Planar terrain: control bounds u_v, joint position / velocity bounds, point height p_z, normal force f_z, CoM
        height (SURVEY.md 8(a): 720 + 667 + 690 + 232 + 232 + 29 = 2 570 of the 8 142 rows of config 3); on the smooth
        terrain the height / normal-force / CoM-height rows are nonlinear and stay general.  Rows with a parametric
        gain (f_dot * mass, h_ang * mass) are not bare variables and stay general.  ``include_equalities`` adds the
        initial-condition rows x_j = parameter (lbx = ubx), which CasADi detects as well [ext] but IPOPT then treats
        as fixed variables unless fixed_variable_treatment = relax_bounds."""
        rows, cols = [], []

        def add(name, k, xoff):
            r0 = self.row(name, k)
            if r0 >= 0:
                for c, off in enumerate(xoff):
                    rows.append(r0 + c)
                    cols.append(NZ * k + off)

        for k in range(self.N):
            for i in range(NPT):
                add(f"pt{i}.u_bounds", k, [15 * i + U + c for c in range(3)])
                if not self.smooth:
                    add(f"pt{i}.height", k, [15 * i + P + 2])
                    add(f"pt{i}.normal", k, [15 * i + F + 2])
                if include_equalities and k == 0:
                    add(f"pt{i}.f_ic", 0, [15 * i + F + c for c in range(3)])
                    add(f"pt{i}.p_ic", 0, [15 * i + P + c for c in range(3)])
            if not self.smooth:
                add("com_height", k, [COM + 2])
            add("s_bounds", k, [S + j for j in range(NJ)])
            add("sd_bounds", k, [SD + j for j in range(NJ)])
            if include_equalities and k == 0:
                for name, off, n in (("pb_ic", PB, 3), ("q_ic", Q, 4), ("s_ic", S, NJ), ("com_ic", COM, 3)):
                    add(name, 0, [off + c for c in range(n)])
        order = np.argsort(rows)
        return np.asarray(rows, dtype=np.int64)[order], np.asarray(cols, dtype=np.int64)[order]

    def bounds(self, p: np.ndarray):
        """(lbg, ubg) for parameter vectors p of shape (B, n_p) -- canonical forms of the
        reference's constraints as CasADi Opti derives them [ext] (see oracle/kinodynamic.py)."""
        p = np.atleast_2d(p)
        B = p.shape[0]
        po = self.po
        N = self.N
        lb = np.zeros((B, self.m))
        ub = np.zeros((B, self.m))
        inf = np.inf

        def setrows(name, k, lo, hi):
            r0 = self.row(name, k)
            if r0 < 0:
                return
            n = self.fam[name][1]
            lb[:, r0:r0 + n] = lo
            ub[:, r0:r0 + n] = hi

        for i in range(NPT):
            v = p[:, po.init + po.st_pt(i, "f"):po.init + po.st_pt(i, "f") + 3]
            setrows(f"pt{i}.f_ic", 0, v, v)
            v = p[:, po.init + po.st_pt(i, "p"):po.init + po.st_pt(i, "p") + 3]
            setrows(f"pt{i}.p_ic", 0, v, v)
            mu = p[:, po.max_u:po.max_u + 3]
            mf = p[:, po.max_fd:po.max_fd + 3]
            for k in range(N):
                setrows(f"pt{i}.dcc", k, 0.0, inf)
                setrows(f"pt{i}.height", k, 0.0, inf)
                setrows(f"pt{i}.normal", k, 0.0, inf)
                setrows(f"pt{i}.friction", k, 0.0, inf)
                setrows(f"pt{i}.u_bounds", k, -mu, mu)
                setrows(f"pt{i}.fd_bounds", k, -mf, mf)
        for name, off, n in (("pb", po.ST_PB, 3), ("q", po.ST_Q, 4), ("s", po.ST_S, NJ), ("com", po.ST_COM, 3)):
            v = p[:, po.init + off:po.init + off + n]
            setrows(f"{name}_ic", 0, v, v)
        for k in range(N):
            setrows("unit_quat", k, 1.0, 1.0)
            setrows("L_bounds", k, -p[:, [po.max_L]], p[:, [po.max_L]])
            setrows("com_height", k, p[:, [po.min_com_h]], inf)
            setrows("feet_dist", k, p[:, [po.min_feet_d]], inf)
            setrows("s_bounds", k, p[:, po.min_s:po.min_s + NJ], p[:, po.max_s:po.max_s + NJ])
            setrows("sd_bounds", k, p[:, po.min_sd:po.min_sd + NJ], p[:, po.max_sd:po.max_sd + NJ])
            setrows("feet_relh", k, -p[:, [po.max_feet_h]], p[:, [po.max_feet_h]])
        if self.st.final_state_constraint:
            fin = np.zeros((B, 105))
            r = 0
            fin[:, 0:3] = p[:, po.final + po.ST_COM:po.final + po.ST_COM + 3]
            r = 3
            for i in range(NPT):
                for what in ("desc", "f", "p"):
                    o = po.final + po.st_pt(i, what)
                    fin[:, r:r + 3] = p[:, o:o + 3]
                    r += 3
            for off, n in ((po.ST_PB, 3), (po.ST_Q, 4), (po.ST_S, NJ)):
                fin[:, r:r + n] = p[:, po.final + off:po.final + off + n]
                r += n
            setrows("final", N - 1, fin, fin)
        return lb, ub

    # ------------------------------------------------------------------ local Jacobian orders
    def _enumerate_jc(self, k: int):
        """Contact-kernel local Jacobian entries of column-knot k: list of (row, col) (or (-1,-1))."""
        N = self.N
        e: list[tuple[int, int]] = []
        xk = NZ * k

        def put(r, c):
            e.append((r, c) if r >= 0 and c >= 0 else (-1, -1))

        names = []
        for i in range(NPT):
            names += [f"pt{i}.f", f"pt{i}.p"]
        names += ["pb", "q", "s", "com"]
        # C1: linear dynamics: per state scalar [next-side state, next-side rate, prev-side state, prev-side rate]
        for (name, (so, ro, n)) in zip(names, linear_states()):
            for c in range(n):
                put(self.row(name + "_dyn", k, c), xk + so + c)
                put(self.row(name + "_dyn", k, c), xk + ro + c)
                put(self.row(name + "_dyn", k + 1, c), xk + so + c)
                put(self.row(name + "_dyn", k + 1, c), xk + ro + c)
        # C2: initial conditions (k = 0)
        for (name, (so, ro, n)) in zip(names, linear_states()):
            for c in range(n):
                put(self.row(name + "_ic", k, c), xk + so + c)
        for c in range(6):
            put(self.row("h_ic", k, c), xk + H + c)
        for c in range(6):
            put(self.row("h_ic", k, c), self.h_init + c)
        # C3: final state (k = N-1) and periodicity (k = 0: +1, k = N-1: -1)
        for (r, off) in self.final_rows():
            if off >= 0:
                put(self.row("final", k, r), xk + off)
        for r, off in enumerate(self.periodicity_vars()):
            if k == 0:
                put(self.row("periodicity", 0, r), xk + off)
            elif k == N - 1:
                put(self.row("periodicity", 0, r), xk + off)
            else:
                put(-1, -1)
        # C4: centroidal momentum dynamics, two sides (row-knot k, then row-knot k+1)
        for rk in (k, k + 1):
            for c in range(6):
                put(self.row("h_dyn", rk, c), xk + H + c)
            for i in range(NPT):
                for c in range(3):
                    put(self.row("h_dyn", rk, c), xk + 15 * i + F + c)
            for i in range(NPT):
                for (a, b) in SKEW_PAIRS:
                    put(self.row("h_dyn", rk, 3 + a), xk + 15 * i + P + b)
            for i in range(NPT):
                for (a, b) in SKEW_PAIRS:
                    put(self.row("h_dyn", rk, 3 + a), xk + 15 * i + F + b)
            for (a, b) in SKEW_PAIRS:
                put(self.row("h_dyn", rk, 3 + a), xk + COM + b)
        # C5: per-point path rows
        for i in range(NPT):
            o = xk + 15 * i
            pl = f"pt{i}.planar"
            if not self.smooth:
                for c in range(3):
                    put(self.row(pl, k, c), o + V + c)
                for c in range(3):
                    put(self.row(pl, k, c), o + U + c)
                put(self.row(pl, k, 0), o + P + 2)
                put(self.row(pl, k, 1), o + P + 2)
                for off in (V + 2, FD + 2, P + 2, F + 2):
                    put(self.row(f"pt{i}.dcc", k), o + off)
                put(self.row(f"pt{i}.height", k), o + P + 2)
                put(self.row(f"pt{i}.normal", k), o + F + 2)
                for c in range(3):
                    put(self.row(f"pt{i}.friction", k), o + F + c)
            else:
                for c in range(3):
                    put(self.row(pl, k, c), o + V + c)
                for c in range(3):
                    for d in range(3):
                        put(self.row(pl, k, c), o + U + d)
                for c in range(3):
                    for d in range(3):
                        put(self.row(pl, k, c), o + P + d)
                for blk in (V, FD, P, F):
                    for d in range(3):
                        put(self.row(f"pt{i}.dcc", k), o + blk + d)
                for d in range(3):
                    put(self.row(f"pt{i}.height", k), o + P + d)
                # n and R_t depend on (x, y) only: grad h = (-T_x, -T_y, 1)
                for name in ("normal", "friction"):
                    for d in range(2):
                        put(self.row(f"pt{i}.{name}", k), o + P + d)
                    for d in range(3):
                        put(self.row(f"pt{i}.{name}", k), o + F + d)
            for c in range(3):
                put(self.row(f"pt{i}.u_bounds", k, c), o + U + c)
            for c in range(3):
                put(self.row(f"pt{i}.fd_bounds", k, c), o + FD + c)
            for c in range(3):
                put(self.row(f"pt{i}.fk", k, c), o + P + c)
            for c in range(3):
                put(self.row(f"pt{i}.fk", k, c), xk + PB + c)
        # C6: robot rows with constant / trivial entries
        for c in range(3):
            put(self.row("com_kin", k, c), xk + COM + c)
        for c in range(3):
            put(self.row("com_kin", k, c), xk + PB + c)
        for c in range(3):
            put(self.row("mom_kin", k, c), xk + H + 3 + c)
        for c in range(3):
            put(self.row("L_bounds", k, c), xk + H + 3 + c)
        if not self.smooth:
            put(self.row("com_height", k), xk + COM + 2)
        else:
            for d in range(3):
                put(self.row("com_height", k), xk + COM + d)
        for c in range(NJ):
            put(self.row("s_bounds", k, c), xk + S + c)
        for c in range(NJ):
            put(self.row("sd_bounds", k, c), xk + SD + c)
        for i in range(NPT):
            put(self.row("feet_relh", k), xk + 15 * i + P + 2)
        return e

    def leg_joints(self, foot: int) -> list[int]:
        body = self.model.frames[self.st.foot_frames[foot]][0]
        return [b - 1 for b in self.model.chain_to_root(body)]

    def chest_joints(self) -> list[int]:
        body = self.model.frames[self.st.frame_quaternion_cost_frame][0]
        return [b - 1 for b in self.model.chain_to_root(body)]

    def _enumerate_jk(self, k: int):
        """Kinematics-kernel local Jacobian entries of column-knot k."""
        e: list[tuple[int, int]] = []
        xk = NZ * k

        def put(r, c):
            e.append((r, c) if r >= 0 else (-1, -1))

        for c in range(4):
            put(self.row("unit_quat", k), xk + Q + c)
        # FK rows: per point, per row: q(4) then every joint (23); non-chain joints are absent
        for i in range(NPT):
            chain = set(self.leg_joints(0 if i < 4 else 1))
            for a in range(3):
                r = self.row(f"pt{i}.fk", k, a)
                for c in range(4):
                    put(r, xk + Q + c)
                for j in range(NJ):
                    put(r if j in chain else -1, xk + S + j)
        for a in range(3):
            r = self.row("com_kin", k, a)
            for c in range(4):
                put(r, xk + Q + c)
            for j in range(NJ):
                put(r, xk + S + j)
        for a in range(3):
            r = self.row("mom_kin", k, a)
            for off, n in ((VB, 3), (QD, 4), (Q, 4), (SD, NJ), (S, NJ)):
                for c in range(n):
                    put(r, xk + off + c)
        legs = set(self.leg_joints(0)) | set(self.leg_joints(1))
        r = self.row("feet_dist", k)
        for j in range(NJ):
            put(r if j in legs else -1, xk + S + j)
        return e

    # ------------------------------------------------------------------ local Hessian orders
    @staticmethod
    def cv_to_z(v: int) -> int:
        """contact-kernel variable id (0..128) -> offset inside the knot."""
        if v < 120:
            return v
        if v < 123:
            return COM + (v - 120)
        return H + (v - 123)

    def _hc_pairs(self, first: bool = False):
        """Structural (i <= j in contact-var ids) pairs of the contact-kernel Hessian block.
        ``first``: knot 0, where every expression added with ``apply_to_first_elements=False``
        (swing, control and force regularisations, friction, yaw, centroid) is absent."""
        pairs = set()

        def add(a, b):
            pairs.add((min(a, b), max(a, b)))

        yp = self.st.yaw_points
        for i in range(NPT):
            o = 15 * i
            if not self.smooth:
                add(o + P + 2, o + P + 2)  # planar tanh'', swing, centroid
                add(o + P + 2, o + U + 0)
                add(o + P + 2, o + U + 1)
                add(o + P + 2, o + F + 2)  # dcc
                add(o + V + 2, o + F + 2)
                add(o + FD + 2, o + P + 2)
                if not first:
                    add(o + V + 0, o + V + 0)  # swing heuristic
                    add(o + V + 1, o + V + 1)
            else:
                # smooth terrain: h = z - T(x, y); n, R_t depend on (x, y) only, so the coefficient of
                # u_z (= n) and d L / d v_z carry no z dependence
                for a in range(3):
                    for b in range(3):
                        add(o + P + a, o + P + b)
                        add(o + P + a, o + F + b)
                        add(o + P + a, o + FD + b)
                        add(o + V + a, o + F + b)
                        if not (a == 2 and b == 2):
                            add(o + P + a, o + U + b)
                            add(o + P + a, o + V + b)
                        if not first:  # friction cone, swing heuristic
                            add(o + V + a, o + V + b)
                            add(o + F + a, o + F + b)
            for c in range(3):
                if not first:
                    add(o + U + c, o + U + c)
                    add(o + FD + c, o + FD + c)
                    add(o + F + c, o + F + c)  # friction + force ratio
            for (a, b) in SKEW_PAIRS:  # centroidal momentum dynamics: (p - x) x f
                add(o + P + a, o + F + b)
                add(120 + a, o + F + b)
        for foot in range(0 if not first else 2, 2):
            base = 4 * foot
            for i in range(4):
                for j in range(i, 4):
                    for c in range(3):
                        add(15 * (base + i) + F + c, 15 * (base + j) + F + c)  # force ratio
            # yaw task: 0.5 (fwd^2 + side^2); fwd couples (p0, p1)_xy, side couples (p1, p2)_xy
            p0, p1, p2 = (15 * (base + y) + P for y in yp)
            for (a, b) in ((p0, p1), (p1, p2)):
                vs = [a, a + 1, b, b + 1]
                for u in vs:
                    for w in vs:
                        add(u, w)
        for i in range(NPT if not first else 0):  # contacts centroid cost: all points, per component
            for j in range(i, NPT):
                for c in range(3):
                    add(15 * i + P + c, 15 * j + P + c)
        for c in range(3):
            add(123 + c, 123 + c)  # com velocity cost on h[0:3]
        if self.smooth and not first:  # minimum com height: h(com) = com_z - T(com_x, com_y)
            add(120, 120)
            add(120, 121)
            add(121, 121)
        return sorted(pairs)

    # ------------------------------------------------------------------ patterns + maps
    def _patterns(self):
        N = self.N
        jc = [self._enumerate_jc(k) for k in range(N)]
        jk = [self._enumerate_jk(k) for k in range(N)]
        self.n_jc, self.n_jk = len(jc[0]), len(jk[0])
        rows, cols = [], []
        for lst in (jc, jk):
            for k in range(N):
                for (r, c) in lst[k]:
                    if r >= 0:
                        rows.append(r)
                        cols.append(c)
        rows = np.asarray(rows, dtype=np.int64)
        cols = np.asarray(cols, dtype=np.int64)
        key = cols * self.m + rows
        keys = np.unique(key)
        if len(keys) != len(key):
            raise AssertionError("duplicate local Jacobian entries")
        self.jac_row = (keys % self.m).astype(np.int64)
        self.jac_col = (keys // self.m).astype(np.int64)
        self.jac_colind = np.zeros(self.n_x + 1, dtype=np.int64)
        np.add.at(self.jac_colind, self.jac_col + 1, 1)
        self.jac_colind = np.cumsum(self.jac_colind)
        self.nnz_j = len(keys)

        def jmap(lst, n):
            out = -np.ones((N, n), dtype=np.int32)
            for k in range(N):
                rc = np.asarray(lst[k], dtype=np.int64)
                ok = rc[:, 0] >= 0
                out[k, ok] = np.searchsorted(keys, rc[ok, 1] * self.m + rc[ok, 0])
            return out

        self.jc_map = jmap(jc, self.n_jc)
        self.jk_map = jmap(jk, self.n_jk)

        # Hessian: contact block pairs + kinematics block
        hc_pairs = self._hc_pairs()
        self.n_hc = len(hc_pairs)
        self.hc_index = -np.ones((NCV, NCV), dtype=np.int16)
        for e, (a, b) in enumerate(hc_pairs):
            self.hc_index[a, b] = e
            self.hc_index[b, a] = e
        # kinematics block: directions (q 0..3, s 0..22), rows (vb, qd, sd, q, s)
        dir_off = [Q + c for c in range(4)] + [S + c for c in range(NJ)]
        row_off = ([VB + c for c in range(3)] + [QD + c for c in range(4)] + [SD + c for c in range(NJ)]
                   + [Q + c for c in range(4)] + [S + c for c in range(NJ)])
        self.hk_dirs, self.hk_rows = dir_off, row_off
        hk_local = []
        for j, cj in enumerate(dir_off):
            for i, ci in enumerate(row_off):
                if i < 30:  # velocity rows (vb, qd, sd) only ever meet (q, s) in this lane
                    hk_local.append((min(ci, cj), max(ci, cj)))
                else:  # (q, s) x (q, s): the mirrored pair is produced by the other lane
                    hk_local.append((ci, cj) if ci <= cj else (-1, -1))
        hk2_local = [(QD + c, QD + c) for c in range(4)] + [(SD + c, SD + c) for c in range(NJ)]
        hc_first = set(self._hc_pairs(first=True))

        def hc_present(k, pair):
            return k > 0 or pair in hc_first

        def hk2_present(k, e):
            return k > 0 or e < 4  # joint regularisation (sd diagonal) skips the first knot

        ent = []
        for k in range(N):
            xk = NZ * k
            for (a, b) in hc_pairs:
                if not hc_present(k, (a, b)):
                    continue
                za, zb = self.cv_to_z(a), self.cv_to_z(b)
                r, c = (za, zb) if za <= zb else (zb, za)
                ent.append((xk + c) * self.n_x + xk + r)
            for (r, c) in hk_local:
                if r >= 0:
                    ent.append((xk + c) * self.n_x + xk + r)
            for e, (r, c) in enumerate(hk2_local):
                if hk2_present(k, e):
                    ent.append((xk + c) * self.n_x + xk + r)
        hkeys = np.unique(np.asarray(ent, dtype=np.int64))
        if len(hkeys) != len(ent):
            raise AssertionError("duplicate local Hessian entries")
        self.hess_row = hkeys % self.n_x
        self.hess_col = hkeys // self.n_x
        self.hess_colind = np.zeros(self.n_x + 1, dtype=np.int64)
        np.add.at(self.hess_colind, self.hess_col + 1, 1)
        self.hess_colind = np.cumsum(self.hess_colind)
        self.nnz_h = len(hkeys)
        self.hc_map = -np.ones((N, self.n_hc), dtype=np.int32)
        self.hk_map = -np.ones((N, len(hk_local)), dtype=np.int32)
        self.hk2_map = -np.ones((N, len(hk2_local)), dtype=np.int32)
        for k in range(N):
            xk = NZ * k
            for e, (a, b) in enumerate(hc_pairs):
                if not hc_present(k, (a, b)):
                    continue
                za, zb = self.cv_to_z(a), self.cv_to_z(b)
                r, c = (za, zb) if za <= zb else (zb, za)
                self.hc_map[k, e] = np.searchsorted(hkeys, (xk + c) * self.n_x + xk + r)
            for e, (r, c) in enumerate(hk_local):
                if r >= 0:
                    self.hk_map[k, e] = np.searchsorted(hkeys, (xk + c) * self.n_x + xk + r)
            for e, (r, c) in enumerate(hk2_local):
                if hk2_present(k, e):
                    self.hk2_map[k, e] = np.searchsorted(hkeys, (xk + c) * self.n_x + xk + r)

    def kernel_bytes_per_knot(self) -> dict:
        """Algorithmic bytes per knot-eval of each kernel (f+J+H): its inputs (the knot of x, the knot's
        parameters, the multipliers of the rows it owns, sigma) plus every output value it writes."""
        N = self.N
        jk = float((self.jk_map >= 0).sum()) / N
        jc = float((self.jc_map >= 0).sum()) / N
        hk = float((self.hk_map >= 0).sum() + (self.hk2_map >= 0).sum()) / N
        hc = float((self.hc_map >= 0).sum()) / N
        kin_rows = sum(self.fam[n][1] * (self.fam[n][3] - self.fam[n][2] + 1) for n in self.fam
                       if n.endswith(".fk") or n in ("unit_quat", "com_kin", "mom_kin", "feet_dist")) / N
        con_rows = self.m / N - kin_rows
        kin = 8.0 * ((NZ + 79 + kin_rows + 1) + (1 + 57 + kin_rows + jk + hk))
        con = 8.0 * ((2 * NZ + 79 + con_rows + 1) + (1 + 132 + con_rows + jc + hc))
        return {"kinematics": kin, "contact": con}

    # per-knot counts, for the roofline arithmetic (DESIGN.md)
    def algorithmic_bytes_per_knot(self, with_hessian: bool = True) -> float:
        """SURVEY.md 8(d): 8 (n_xk + n_pk + m_k + 1) + 8 (1 + n_xk + m_k + nnzJ_k [+ nnzH_k])."""
        N = self.N
        n_xk, n_pk = NZ, 79
        m_k = self.m / N
        j_k = self.nnz_j / N
        h_k = self.nnz_h / N if with_hessian else 0.0
        return 8.0 * (n_xk + n_pk + m_k + 1) + 8.0 * (1 + n_xk + m_k + j_k + h_k)
