"""Layout compiler for the humanoid pose finder (BASELINE config 2).

Static-pose NLP of `/root/reference/src/hippopt/turnkey_planners/humanoid_pose_finder/planner.py:
303-413, 444-788` with the defaults of `planner.py:79-92` (CoM / point positions as costs, hands
skipped): x (81), p (202), g (89) orderings of SURVEY.md Appendix B.4 and the CCS patterns of jac_g /
upper-triangular hess_l.  PlanarTerrain by default; ``terrain="smooth_steps"`` poses the same problem on
the two smooth steps of the stairs (BASELINE config 5) with their ten parameters (l, w, height, ox, oy) x 2
appended to p (p = 212), as the kinodynamic layout does.

The device kernels work on a *virtual knot* in the kinodynamic 189-variable layout
(`kino_layout`): ``zmap[i]`` is the x offset of virtual variable i or -1.  The kinematics kernel keeps
its local Jacobian / Hessian orders (kino_layout.KinoLayout._enumerate_jk, direction-major Hessian),
the pose contact kernel (csrc/pose_contact.cu) uses :meth:`PoseLayout._enumerate_jp`.
"""
from __future__ import annotations

import dataclasses

import numpy as np

from .kino_layout import COM, F, H, NCV, NJ, NPT, NZ, P, PB, Q, QD, S, SD, SKEW_PAIRS, VB, kernel_terrain
from .robot_model import RobotModel

XPB, XQ, XS, XCOM, NX = 48, 51, 55, 78, 81


@dataclasses.dataclass
class PoseSettings:
    """`humanoid_pose_finder/main.py:75-98`."""

    terrain: str = "planar"  # one of kino_layout.TERRAINS
    n_terrain_params: int = 0
    foot_frames: tuple = ("l_sole", "r_sole")
    frame_quaternion_cost_frame: str = "chest"
    joint_regularization_cost_weights: np.ndarray = dataclasses.field(
        default_factory=lambda: np.concatenate([0.1 * np.ones(3), 10.0 * np.ones(8), np.ones(12)])
    )
    base_quaternion_cost_multiplier: float = 50.0
    desired_frame_quaternion_cost_multiplier: float = 100.0
    joint_regularization_cost_multiplier: float = 0.1
    force_regularization_cost_multiplier: float = 0.2
    com_regularization_cost_multiplier: float = 10.0
    average_force_regularization_cost_multiplier: float = 10.0
    point_position_regularization_cost_multiplier: float = 100.0


class PoseParamOffsets:
    def __init__(self, n_terrain: int = 0):
        o = 0
        self.desc0 = o
        o += 24
        self.mass, self.plm, self.pld = o, o + 1, o + 2
        o += 3
        self.gravity = o
        o += 6
        self.ref = o  # references.state: per point (p, f, descriptor), pb, q, s, com
        o += 105
        self.ref_fq = o
        o += 4
        self.ref_lhand, self.ref_rhand = o, o + 3
        o += 6
        self.eps, self.mu = o, o + 1
        o += 2
        self.max_s, self.min_s = o, o + NJ
        o += 2 * NJ
        self.lhand_in_frame, self.rhand_in_frame = o, o + 3
        o += 6
        self.terrain = o
        o += n_terrain
        self.n_p = o

    ST_PB, ST_Q, ST_S, ST_COM = 72, 75, 79, 102


class PoseLayout:
    def __init__(self, model: RobotModel, settings: PoseSettings | None = None):
        self.model = model
        self.st = settings or PoseSettings()
        self.N = 1
        self.n_x = NX
        self.kernel_terrain = kernel_terrain(self.st.terrain, self.st.n_terrain_params)
        self.smooth = self.st.terrain != "planar"
        self.po = PoseParamOffsets(self.st.n_terrain_params)
        self.n_p = self.po.n_p
        zmap = -np.ones(NZ, dtype=np.int32)
        for i in range(NPT):
            zmap[15 * i + P:15 * i + P + 3] = np.arange(6 * i, 6 * i + 3)
            zmap[15 * i + F:15 * i + F + 3] = np.arange(6 * i + 3, 6 * i + 6)
        zmap[PB:PB + 3] = np.arange(XPB, XPB + 3)
        zmap[Q:Q + 4] = np.arange(XQ, XQ + 4)
        zmap[S:S + NJ] = np.arange(XS, XS + NJ)
        zmap[COM:COM + 3] = np.arange(XCOM, XCOM + 3)
        self.zmap = zmap
        # rows in subject_to order (planner.py:379-393, 444-521)
        self.fam: dict[str, tuple[int, int, int, int]] = {}
        m = 0
        for i in range(NPT):
            for name, rows in (("complementarity", 1), ("height", 1), ("normal", 1), ("friction", 1), ("fk", 3)):
                self.fam[f"pt{i}.{name}"] = (m, rows, 0, 0)
                m += rows
        for name, rows in (("unit_quat", 1), ("com_kin", 3), ("balance", 6), ("s_bounds", NJ)):
            self.fam[name] = (m, rows, 0, 0)
            m += rows
        self.m = m
        self._patterns()

    def row(self, name, r=0):
        return self.fam[name][0] + r

    def leg_joints(self, foot):
        body = self.model.frames[self.st.foot_frames[foot]][0]
        return [b - 1 for b in self.model.chain_to_root(body)]

    def bounds(self, p):
        p = np.atleast_2d(p)
        B = p.shape[0]
        lb = np.zeros((B, self.m))
        ub = np.zeros((B, self.m))
        for i in range(NPT):
            for name in ("complementarity", "height", "normal", "friction"):
                ub[:, self.row(f"pt{i}.{name}")] = np.inf
        lb[:, self.row("unit_quat")] = ub[:, self.row("unit_quat")] = 1.0
        r0 = self.row("s_bounds")
        lb[:, r0:r0 + NJ] = p[:, self.po.min_s:self.po.min_s + NJ]
        ub[:, r0:r0 + NJ] = p[:, self.po.max_s:self.po.max_s + NJ]
        return lb, ub

    # ------------------------------------------------------------------ local orders
    def _enumerate_jp(self):
        """Pose contact kernel: (row, x column) per local Jacobian entry.  Per point 13 entries on the planar
        terrain, 25 on the smooth steps, where h = z - T(x, y) and n, R_t depend on (x, y) only."""
        e = []
        z = self.zmap
        for i in range(NPT):
            o = 15 * i
            if not self.smooth:
                e.append((self.row(f"pt{i}.complementarity"), z[o + P + 2]))
                e.append((self.row(f"pt{i}.complementarity"), z[o + F + 2]))
                e.append((self.row(f"pt{i}.height"), z[o + P + 2]))
                e.append((self.row(f"pt{i}.normal"), z[o + F + 2]))
                for c in range(3):
                    e.append((self.row(f"pt{i}.friction"), z[o + F + c]))
            else:
                for blk in (P, F):
                    for d in range(3):
                        e.append((self.row(f"pt{i}.complementarity"), z[o + blk + d]))
                for d in range(3):
                    e.append((self.row(f"pt{i}.height"), z[o + P + d]))
                for name in ("normal", "friction"):
                    for d in range(2):
                        e.append((self.row(f"pt{i}.{name}"), z[o + P + d]))
                    for d in range(3):
                        e.append((self.row(f"pt{i}.{name}"), z[o + F + d]))
            for c in range(3):
                e.append((self.row(f"pt{i}.fk", c), z[o + P + c]))
            for c in range(3):
                e.append((self.row(f"pt{i}.fk", c), z[PB + c]))
        for c in range(3):
            e.append((self.row("com_kin", c), z[COM + c]))
        for c in range(3):
            e.append((self.row("com_kin", c), z[PB + c]))
        for i in range(NPT):
            for c in range(3):
                e.append((self.row("balance", c), z[15 * i + F + c]))
        for blk in (P, F):
            for i in range(NPT):
                for (a, b) in SKEW_PAIRS:
                    e.append((self.row("balance", 3 + a), z[15 * i + blk + b]))
        for (a, b) in SKEW_PAIRS:
            e.append((self.row("balance", 3 + a), z[COM + b]))
        for c in range(NJ):
            e.append((self.row("s_bounds", c), z[S + c]))
        return e

    def _enumerate_jk(self):
        """Kinematics kernel local order (kino_layout.KinoLayout._enumerate_jk) with the rows that do
        not exist here (momentum, feet distance) absent."""
        e = []
        z = self.zmap
        for c in range(4):
            e.append((self.row("unit_quat"), z[Q + c]))
        for i in range(NPT):
            chain = set(self.leg_joints(0 if i < 4 else 1))
            for a in range(3):
                r = self.row(f"pt{i}.fk", a)
                for c in range(4):
                    e.append((r, z[Q + c]))
                for j in range(NJ):
                    e.append((r, z[S + j]) if j in chain else (-1, -1))
        for a in range(3):
            r = self.row("com_kin", a)
            for c in range(4):
                e.append((r, z[Q + c]))
            for j in range(NJ):
                e.append((r, z[S + j]))
        e += [(-1, -1)] * (3 * 57 + NJ)
        return e

    def _hp_pairs(self):
        pairs = set()

        def add(a, b):
            pairs.add((min(a, b), max(a, b)))

        for i in range(NPT):
            o = 15 * i
            add(o + P + 2, o + F + 2)  # relaxed complementarity
            if self.smooth:
                # h(p) n(p).f, n.f and (R_t(p)^T f)^2: every (p, p), (p, f) and (f, f) pair of the point
                for a in range(3):
                    for b in range(3):
                        add(o + P + a, o + P + b)
                        add(o + P + a, o + F + b)
                        add(o + F + a, o + F + b)
            for c in range(3):
                add(o + P + c, o + P + c)  # point position regularisation
                add(o + F + c, o + F + c)  # friction, force regularisation, average force
            for (a, b) in SKEW_PAIRS:  # static balance (p - x) x f
                add(o + P + a, o + F + b)
                add(120 + a, o + F + b)
        for foot in range(2):
            for i in range(4):
                for j in range(i, 4):
                    for c in range(3):
                        add(15 * (4 * foot + i) + F + c, 15 * (4 * foot + j) + F + c)
        for c in range(3):
            add(120 + c, 120 + c)
        return sorted(pairs)

    @staticmethod
    def cv_to_z(v):
        return v if v < 120 else (COM + v - 120 if v < 123 else H + v - 123)

    def _patterns(self):
        jp, jk = self._enumerate_jp(), self._enumerate_jk()
        self.n_jc, self.n_jk = len(jp), len(jk)
        rc = np.array([(r, c) for (r, c) in jp + jk if r >= 0], dtype=np.int64)
        key = rc[:, 1] * self.m + rc[:, 0]
        keys = np.unique(key)
        assert len(keys) == len(key), "duplicate local Jacobian entries"
        self.jac_row, self.jac_col = keys % self.m, keys // self.m
        self.jac_colind = np.concatenate([[0], np.cumsum(np.bincount(self.jac_col, minlength=self.n_x))])
        self.nnz_j = len(keys)

        def jmap(lst):
            out = -np.ones((1, len(lst)), dtype=np.int32)
            for e, (r, c) in enumerate(lst):
                if r >= 0:
                    out[0, e] = np.searchsorted(keys, c * self.m + r)
            return out

        self.jc_map, self.jk_map = jmap(jp), jmap(jk)
        # Hessian
        hp_pairs = self._hp_pairs()
        self.n_hc = len(hp_pairs)
        self.hc_index = -np.ones((NCV, NCV), dtype=np.int16)
        for e, (a, b) in enumerate(hp_pairs):
            self.hc_index[a, b] = self.hc_index[b, a] = e
        z = self.zmap
        anc = self.model.subtree_mask()  # anc[j, l]: body l in the subtree of body j
        dir_off = [Q + c for c in range(4)] + [S + c for c in range(NJ)]
        row_off = ([VB + c for c in range(3)] + [QD + c for c in range(4)] + [SD + c for c in range(NJ)]
                   + [Q + c for c in range(4)] + [S + c for c in range(NJ)])
        hk_local = []
        for j, cj in enumerate(dir_off):
            for i, ci in enumerate(row_off):
                ok = i >= 30 and ci <= cj
                if ok and i >= 34 and j >= 4:  # (s_i, s_j): only joints on one chain couple
                    bi, bj = i - 34 + 1, j - 4 + 1
                    ok = anc[bi, bj] or anc[bj, bi]
                hk_local.append((z[ci], z[cj]) if ok else (-1, -1))
        ent = []
        for (a, b) in hp_pairs:
            xa, xb = z[self.cv_to_z(a)], z[self.cv_to_z(b)]
            ent.append((min(xa, xb), max(xa, xb)))
        ent += [(r, c) for (r, c) in hk_local if r >= 0]
        ent = np.array(ent, dtype=np.int64)
        hkey = ent[:, 1] * self.n_x + ent[:, 0]
        hkeys = np.unique(hkey)
        assert len(hkeys) == len(hkey), "duplicate local Hessian entries"
        self.hess_row, self.hess_col = hkeys % self.n_x, hkeys // self.n_x
        self.hess_colind = np.concatenate([[0], np.cumsum(np.bincount(self.hess_col, minlength=self.n_x))])
        self.nnz_h = len(hkeys)
        self.hc_map = -np.ones((1, self.n_hc), dtype=np.int32)
        for e, (a, b) in enumerate(hp_pairs):
            xa, xb = z[self.cv_to_z(a)], z[self.cv_to_z(b)]
            self.hc_map[0, e] = np.searchsorted(hkeys, max(xa, xb) * self.n_x + min(xa, xb))
        self.hk_map = -np.ones((1, len(hk_local)), dtype=np.int32)
        for e, (r, c) in enumerate(hk_local):
            if r >= 0:
                self.hk_map[0, e] = np.searchsorted(hkeys, c * self.n_x + r)
        self.hk2_map = -np.ones((1, 27), dtype=np.int32)
