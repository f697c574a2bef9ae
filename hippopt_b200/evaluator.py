"""Batched NLP evaluators: thin Python owners of device buffers around the C ABI.

PyTorch is used only for device memory and streams; every number is produced by the CUDA
kernels behind ``hb_eval`` (include/hippopt_b200.h).  ``eval`` mirrors the five CasADi nlpsol
oracle functions IPOPT calls inside ``opti.solve()``
(`/root/reference/src/hippopt/base/opti_solver.py:479`): f, grad_f, g, jac_g, hess_l.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _capi
from ._capi import H
from .kino_layout import NJ, KinoLayout, KinoSettings
from .robot_model import RobotModel

F, GRAD_F, G, JAC_G, HESS_L = (H["HB_EVAL_F"], H["HB_EVAL_GRAD_F"], H["HB_EVAL_G"], H["HB_EVAL_JAC_G"],
                               H["HB_EVAL_HESS_L"])
ALL = F | GRAD_F | G | JAC_G | HESS_L


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


class _Evaluator:
    """Common part: dims, output buffer ownership, the hb_eval call."""

    def __init__(self):
        self._h = ctypes.c_void_p()
        self._bufs: dict = {}

    def _read_dims(self):
        v = [ctypes.c_int64() for _ in range(5)]
        _capi.check(_capi.lib().hb_dims(self._h, *[ctypes.byref(a) for a in v]), "hb_dims")
        self.n_x, self.n_p, self.m, self.nnz_j, self.nnz_h = (int(a.value) for a in v)

    def close(self):
        if self._h:
            _capi.lib().hb_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _out(self, name, shape, device):
        key = (name, tuple(shape), str(device))
        buf = self._bufs.get(key)
        if buf is None:
            buf = torch.empty(shape, dtype=torch.float64, device=device)
            self._bufs[key] = buf
        return buf

    def eval(self, mask: int, x: torch.Tensor, p: torch.Tensor, lam_g: torch.Tensor | None = None,
             sigma: torch.Tensor | None = None, stream: torch.cuda.Stream | None = None,
             out: dict | None = None) -> dict:
        """x: (B, n_x) cuda float64; p: (B, n_p) or (n_p,); lam_g: (B, m); sigma: (B,).
        Returns a dict with the requested outputs; ``out`` supplies caller-owned output tensors,
        otherwise internal buffers are reused between calls."""
        if not x.is_cuda or x.dtype != torch.float64 or not x.is_contiguous():
            raise ValueError("x must be a contiguous float64 CUDA tensor")
        if x.dim() != 2 or x.shape[1] != self.n_x:
            raise ValueError(f"x must have shape (B, {self.n_x})")
        B = x.shape[0]
        if not p.is_cuda or p.dtype != torch.float64 or not p.is_contiguous():
            raise ValueError("p must be a contiguous float64 CUDA tensor")
        if p.dim() == 1:
            if p.shape[0] != self.n_p:
                raise ValueError(f"p must have {self.n_p} entries")
            p_stride = 0
        else:
            if tuple(p.shape) != (B, self.n_p):
                raise ValueError(f"p must have shape ({B}, {self.n_p})")
            p_stride = self.n_p
        if mask & HESS_L:
            if lam_g is None or sigma is None:
                raise ValueError("lam_g and sigma are required for the Hessian")
            if tuple(lam_g.shape) != (B, self.m) or tuple(sigma.shape) != (B,):
                raise ValueError("lam_g must be (B, m) and sigma (B,)")
            for t in (lam_g, sigma):
                if not t.is_cuda or t.dtype != torch.float64 or not t.is_contiguous():
                    raise ValueError("lam_g / sigma must be contiguous float64 CUDA tensors")
        dev = x.device
        given = out if out is not None else {}
        out = {}
        for bit, name, shape in ((F, "f", (B,)), (GRAD_F, "grad_f", (B, self.n_x)), (G, "g", (B, self.m)),
                                 (JAC_G, "jac", (B, self.nnz_j)), (HESS_L, "hess", (B, self.nnz_h))):
            if not mask & bit:
                continue
            t = given.get(name)
            if t is None:
                t = self._out(name, shape, dev)
            elif tuple(t.shape) != shape or not t.is_cuda or t.dtype != torch.float64 or not t.is_contiguous():
                raise ValueError(f"out[{name!r}] must be a contiguous float64 CUDA tensor of shape {shape}")
            out[name] = t
        st = stream if stream is not None else torch.cuda.current_stream(dev)
        rc = _capi.lib().hb_eval(self._h, mask, _ptr(x), _ptr(p), p_stride, _ptr(lam_g), _ptr(sigma),
                                 _ptr(out.get("f")), _ptr(out.get("grad_f")), _ptr(out.get("g")),
                                 _ptr(out.get("jac")), _ptr(out.get("hess")), B, ctypes.c_void_p(st.cuda_stream))
        _capi.check(rc, "hb_eval")
        return out

    def last_launch_count(self) -> int:
        return int(_capi.lib().hb_last_launch_count(self._h))

    def set_option(self, name: str, value: int) -> None:
        """name: a HB_OPT_* constant of include/hippopt_b200.h without the prefix, e.g. "JAC_ADJOINT"."""
        _capi.check(_capi.lib().hb_set_option(self._h, H["HB_OPT_" + name], int(value)), "hb_set_option")

    def profile(self, enable: bool) -> None:
        _capi.check(_capi.lib().hb_profile_enable(self._h, int(enable)), "hb_profile_enable")

    def profile_read(self):
        """({kernel: summed ms}, number of hb_eval calls) since profile(True)."""
        ms = (ctypes.c_double * 3)()
        n = ctypes.c_int64()
        _capi.check(_capi.lib().hb_profile_read(self._h, ms, ctypes.byref(n)), "hb_profile_read")
        return {"contact": ms[0], "kinematics": ms[1], "reduce_f": ms[2]}, int(n.value)


class HostPipeline:
    """The call a CPU-side solver makes: host buffers in, host buffers out.

    IPOPT lives on the host (SURVEY.md 8(f) f1), so every evaluation needs x (and lam_g, sigma) copied
    to the device and the values copied back.  This is a thin owner of pinned host output buffers
    around ``hb_eval_host`` (include/hippopt_b200.h): the library cuts the batch into chunks pipelined
    over its own CUDA streams so that H2D copies, the kernels and D2H copies of different chunks
    overlap.  Parameters are uploaded once per solve (``set_parameters``), as they do not change
    between IPOPT iterations."""

    def __init__(self, ev: _Evaluator, batch: int, mask: int = ALL, pinned: bool = True):
        self.ev, self.B, self.mask = ev, batch, mask
        shapes = {"f": (), "grad_f": (ev.n_x,), "g": (ev.m,), "jac": (ev.nnz_j,), "hess": (ev.nnz_h,)}
        bits = {"f": F, "grad_f": GRAD_F, "g": G, "jac": JAC_G, "hess": HESS_L}
        self.names = [n for n in shapes if mask & bits[n]]
        # one pinned block in the library's slab order (f | grad_f | g | jac | hess): hb_eval_host merges copies whose
        # host and device ranges are adjacent, which they are whenever the whole batch is one chunk
        sizes = {n: batch * int(np.prod(shapes[n], dtype=np.int64)) for n in self.names}
        block = self.host_buffer((sum(sizes.values()),), pinned)
        self.host_out, o = {}, 0
        for n in self.names:
            self.host_out[n] = block[o:o + sizes[n]].view((batch, *shapes[n]))
            o += sizes[n]
        self._block = block
        self.h2d_bytes = self.d2h_bytes = 0

    @staticmethod
    def host_buffer(shape, pinned: bool = True) -> torch.Tensor:
        t = torch.empty(shape, dtype=torch.float64)
        return t.pin_memory() if pinned else t

    def set_parameters(self, p_host: torch.Tensor) -> None:
        """p_host: (B, n_p) or (n_p,) float64 host tensor; uploaded once per solve."""
        if p_host.is_cuda or p_host.dtype != torch.float64 or not p_host.is_contiguous():
            raise ValueError("p_host must be a contiguous float64 host tensor")
        if p_host.dim() == 1 and p_host.shape[0] == self.ev.n_p:
            stride, batch = 0, 0
        elif p_host.dim() == 2 and p_host.shape[1] == self.ev.n_p:
            stride, batch = self.ev.n_p, p_host.shape[0]
        else:
            raise ValueError(f"p_host must have shape (B, {self.ev.n_p}) or ({self.ev.n_p},)")
        _capi.check(_capi.lib().hb_host_set_parameters(self.ev._h, _ptr(p_host), stride, batch), "hb_host_set_parameters")

    def run(self, x_host: torch.Tensor, lam_host: torch.Tensor | None = None,
            sigma_host: torch.Tensor | None = None) -> dict:
        """x_host (B, n_x), lam_host (B, m), sigma_host (B,): float64 host tensors (pinned for full overlap).
        One blocking ``hb_eval_host`` call; returns the host output tensors."""
        ev, B = self.ev, self.B
        need_l = bool(self.mask & HESS_L)
        for name, t, shape in (("x_host", x_host, (B, ev.n_x)), ("lam_host", lam_host, (B, ev.m)),
                               ("sigma_host", sigma_host, (B,))):
            if t is None:
                if name != "x_host" and not need_l:
                    continue
                raise ValueError(f"{name} is required")
            if t.is_cuda or t.dtype != torch.float64 or not t.is_contiguous() or tuple(t.shape) != shape:
                raise ValueError(f"{name} must be a contiguous float64 host tensor of shape {shape}")
        o = self.host_out
        rc = _capi.lib().hb_eval_host(ev._h, self.mask, _ptr(x_host), _ptr(lam_host if need_l else None),
                                      _ptr(sigma_host if need_l else None), _ptr(o.get("f")), _ptr(o.get("grad_f")),
                                      _ptr(o.get("g")), _ptr(o.get("jac")), _ptr(o.get("hess")), B)
        _capi.check(rc, "hb_eval_host")
        up, down = ctypes.c_int64(), ctypes.c_int64()
        _capi.check(_capi.lib().hb_host_last_traffic(ev._h, ctypes.byref(up), ctypes.byref(down)), "hb_host_last_traffic")
        self.h2d_bytes, self.d2h_bytes = int(up.value), int(down.value)
        return self.host_out


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def bound_table(lay, seed: int = 0):
    """(lb_idx, lb_val, ub_idx, ub_val) with lbg[r] = lb_val[r] * p[lb_idx[r]] if lb_idx[r] >= 0 else lb_val[r].

    Every bound of these planners is a constant or +- one parameter (oracle/kinodynamic.py header: canonical forms of
    Opti), so the table is recovered from `layout.bounds` itself by evaluating it on two random parameter vectors --
    no second statement of the bound rules -- and verified on a third."""
    rng = np.random.default_rng(seed)
    n_p, m = lay.n_p, lay.m
    p1, p2, p3 = (rng.uniform(1.0, 2.0, (1, n_p)) * rng.choice([-1.0, 1.0], (1, n_p)) for _ in range(3))
    out = []
    for side in (0, 1):
        b1, b2, b3 = (lay.bounds(p)[side][0] for p in (p1, p2, p3))
        idx = -np.ones(m, dtype=np.int32)
        val = b1.copy()
        moving = np.nonzero(b1 != b2)[0]
        order = np.argsort(np.abs(p1[0]))
        sorted_abs = np.abs(p1[0])[order]
        for r in moving:
            j = int(np.searchsorted(sorted_abs, abs(b1[r])))
            cands = [order[q] for q in (j - 1, j, j + 1) if 0 <= q < n_p]
            hit = [c for c in cands if abs(abs(p1[0, c]) - abs(b1[r])) <= 1e-12 * abs(b1[r])]
            if len(hit) != 1:
                raise ValueError(f"bound of row {r} is not +- one parameter")
            idx[r] = hit[0]
            val[r] = b1[r] / p1[0, hit[0]]
        chk = np.where(idx >= 0, val * p3[0, np.maximum(idx, 0)], val)
        if not np.array_equal(chk, b3) or not np.array_equal(np.where(idx >= 0, val * p2[0, np.maximum(idx, 0)], val), b2):
            raise ValueError("bounds are not affine in single parameters")
        out += [idx, np.ascontiguousarray(val, dtype=np.float64)]
    return tuple(out)


class KinoEvaluator(_Evaluator):
    """Evaluator of the humanoid kinodynamic OCP
    (`/root/reference/src/hippopt/turnkey_planners/humanoid_kinodynamic/planner.py:27-176`)."""

    def __init__(self, model: RobotModel, settings: KinoSettings, layout: KinoLayout | None = None):
        super().__init__()
        self.model = model
        self.settings = settings
        self.layout = lay = layout if layout is not None else KinoLayout(model, settings)
        icfg = np.zeros(H["HB_KI_COUNT"], dtype=np.int32)
        po = lay.po
        ints = {
            "HORIZON": lay.N, "N_X": lay.n_x, "N_P": lay.n_p, "M": lay.m, "NNZ_J": lay.nnz_j, "NNZ_H": lay.nnz_h,
            "N_JC": lay.n_jc, "N_JK": lay.n_jk, "N_HC": lay.n_hc, "TERRAIN": lay.kernel_terrain,
            "HAS_FINAL": int(settings.final_state_constraint), "HAS_PERIODICITY": int(settings.periodicity_constraint),
            "H_INIT": lay.h_init, "PO_DESC0": po.desc0, "PO_MASS": po.mass, "PO_INIT": po.init, "PO_FINAL": po.final,
            "PO_DT": po.dt, "PO_GRAVITY": po.gravity, "PO_KT": po.kt, "PO_KBS": po.k_bs, "PO_EPS": po.eps,
            "PO_MU": po.mu, "PO_MAX_U": po.max_u, "PO_MAX_FD": po.max_fd, "PO_MAX_L": po.max_L,
            "PO_MIN_COM_H": po.min_com_h, "PO_MIN_FEET_D": po.min_feet_d, "PO_MAX_FEET_H": po.max_feet_h,
            "PO_MAX_S": po.max_s, "PO_MIN_S": po.min_s, "PO_MAX_SD": po.max_sd, "PO_MIN_SD": po.min_sd,
            "PO_REFS0": po.refs0, "PO_TERRAIN": po.terrain, "YAW_BR": settings.yaw_points[0],
            "YAW_TR": settings.yaw_points[1], "YAW_TL": settings.yaw_points[2], "N_BODIES": model.n_bodies,
            "FOOT_BODY_L": model.frames[settings.foot_frames[0]][0],
            "FOOT_BODY_R": model.frames[settings.foot_frames[1]][0],
            "CHEST_BODY": model.frames[settings.frame_quaternion_cost_frame][0],
            "KIND": 0, "X_STRIDE": 189, "COST_K0": 1, "JOINT_COST_KIND": 0, "PO_FQ": po.refs0 + po.R_FQ,
            "PO_BQ": po.refs0 + po.R_BQ, "PO_BQV": po.refs0 + po.R_BQV, "PO_JR": po.refs0 + po.R_JR, "REF_STRIDE": 55,
        }
        for k, v in ints.items():
            icfg[H["HB_KI_" + k]] = v
        icfg[H["HB_KI_ZMAP0"]:H["HB_KI_ZMAP0"] + 189] = np.arange(189)
        icfg[H["HB_KI_PARENT0"]:H["HB_KI_PARENT0"] + model.n_bodies] = model.parent
        pt_names = ["f_ic", "f_dyn", "p_ic", "p_dyn", "planar", "dcc", "height", "normal", "friction", "u_bounds",
                    "fd_bounds", "fk"]
        robot = {"PB_IC": "pb_ic", "PB_DYN": "pb_dyn", "Q_IC": "q_ic", "Q_DYN": "q_dyn", "S_IC": "s_ic",
                 "S_DYN": "s_dyn", "COM_IC": "com_ic", "COM_DYN": "com_dyn", "H_IC": "h_ic", "H_DYN": "h_dyn",
                 "UNIT_QUAT": "unit_quat", "COM_KIN": "com_kin", "MOM_KIN": "mom_kin", "L_BOUNDS": "L_bounds",
                 "COM_HEIGHT": "com_height", "FEET_DIST": "feet_dist", "S_BOUNDS": "s_bounds",
                 "SD_BOUNDS": "sd_bounds", "FINAL": "final", "FEET_RELH": "feet_relh", "PERIODICITY": "periodicity"}

        def put_fam(fid, name):
            base, rows, k0, k1 = lay.fam.get(name, (-1, 0, 1, 0))
            icfg[H["HB_KI_FAM0"] + 4 * fid:H["HB_KI_FAM0"] + 4 * fid + 4] = (base, rows, k0, k1)

        assert H["HB_KF_PT_COUNT"] == len(pt_names)
        for i in range(8):
            for j, nm in enumerate(pt_names):
                put_fam(i * H["HB_KF_PT_COUNT"] + j, f"pt{i}.{nm}")
        for cname, nm in robot.items():
            put_fam(H["HB_KF_" + cname], nm)

        dcfg = np.zeros(H["HB_KD_COUNT"], dtype=np.float64)
        s = settings
        dcfg[H["HB_KD_W_SWING"]] = s.swing_foot_height_cost_multiplier
        dcfg[H["HB_KD_W_U"]] = s.contact_velocity_control_cost_multiplier
        dcfg[H["HB_KD_W_FD"]] = s.contact_force_control_cost_multiplier
        dcfg[H["HB_KD_W_CENTROID"]] = s.contacts_centroid_cost_multiplier
        dcfg[H["HB_KD_W_COMVEL0"]:H["HB_KD_W_COMVEL0"] + 3] = (
            s.com_linear_velocity_cost_multiplier * np.asarray(s.com_linear_velocity_cost_weights, dtype=np.float64))
        dcfg[H["HB_KD_W_FRAME"]] = s.desired_frame_quaternion_cost_multiplier
        dcfg[H["HB_KD_W_BQ"]] = s.base_quaternion_cost_multiplier
        dcfg[H["HB_KD_W_BQV"]] = s.base_quaternion_velocity_cost_multiplier
        dcfg[H["HB_KD_W_JOINT"]] = s.joint_regularization_cost_multiplier
        dcfg[H["HB_KD_W_RATIO"]] = s.force_regularization_cost_multiplier
        dcfg[H["HB_KD_W_YAW"]] = s.foot_yaw_regularization_cost_multiplier
        dcfg[H["HB_KD_WJ0"]:H["HB_KD_WJ0"] + NJ] = s.joint_regularization_cost_weights
        _fill_model_tables(dcfg, model, s.foot_frames, s.frame_quaternion_cost_frame)
        self._create_handle(icfg, dcfg, lay)

    def _create_handle(self, icfg, dcfg, lay):
        self._keep = (icfg, dcfg, _i32(lay.jc_map), _i32(lay.jk_map), np.ascontiguousarray(lay.hc_index, dtype=np.int16),
                      _i32(lay.hc_map), _i32(lay.hk_map), _i32(lay.hk2_map))
        i32p, i16p, f64p = (ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int16),
                            ctypes.POINTER(ctypes.c_double))
        a = self._keep
        rc = _capi.lib().hb_kino_create(
            a[0].ctypes.data_as(i32p), a[1].ctypes.data_as(f64p), a[2].ctypes.data_as(i32p), a[3].ctypes.data_as(i32p),
            a[4].ctypes.data_as(i16p), a[5].ctypes.data_as(i32p), a[6].ctypes.data_as(i32p), a[7].ctypes.data_as(i32p),
            ctypes.byref(self._h))
        _capi.check(rc, "hb_kino_create")
        self._read_dims()
        assert (self.n_x, self.n_p, self.m) == (lay.n_x, lay.n_p, lay.m)
        self._attach_tables(lay)

    def _attach_tables(self, lay):
        """Patterns and the affine description of lbg / ubg go into the handle, so that hb_pattern_*, hb_bounds and a
        file written by hb_save serve callers that do not have this layout compiler."""
        li, lv, ui, uv = bound_table(lay)
        i64p, i32p, f64p = (ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_double))
        t = [np.ascontiguousarray(a, dtype=np.int64) for a in (lay.jac_colind, lay.jac_row, lay.hess_colind, lay.hess_row)]
        rc = _capi.lib().hb_kino_attach_tables(self._h, *(a.ctypes.data_as(i64p) for a in t), li.ctypes.data_as(i32p),
                                               lv.ctypes.data_as(f64p), ui.ctypes.data_as(i32p), uv.ctypes.data_as(f64p))
        _capi.check(rc, "hb_kino_attach_tables")

    def save(self, path: str) -> None:
        """Write the handle to a file a non-Python caller opens with hb_load (include/hippopt_b200.h)."""
        _capi.check(_capi.lib().hb_save(self._h, path.encode()), "hb_save")

    def cost_terms(self, x: torch.Tensor, p: torch.Tensor) -> torch.Tensor:
        """[B, N, HB_COST_TERMS] values of the named cost expressions (hb_eval_cost_terms; names: naming.py)."""
        B = x.shape[0]
        if x.shape != (B, self.n_x) or x.dtype != torch.float64 or not x.is_contiguous():
            raise ValueError(f"x must be a contiguous float64 tensor of shape (B, {self.n_x})")
        p_stride = 0 if p.dim() == 1 else self.n_p
        if p.shape[-1] != self.n_p or (p.dim() == 2 and p.shape[0] != B) or not p.is_contiguous():
            raise ValueError(f"p must be contiguous, of shape ({self.n_p},) or (B, {self.n_p})")
        out = self._out("cost_terms", (B, self.layout.N, H["HB_COST_TERMS"]), x.device)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _capi.check(_capi.lib().hb_eval_cost_terms(self._h, _ptr(x), _ptr(p), p_stride, _ptr(out), B,
                                                   ctypes.c_void_p(stream)), "hb_eval_cost_terms")
        return out

    # patterns (CasADi-style compressed-column)
    def jac_sparsity(self):
        return self.layout.jac_colind, self.layout.jac_row

    def hess_sparsity(self):
        return self.layout.hess_colind, self.layout.hess_row

    def bounds(self, p):
        return self.layout.bounds(np.asarray(p))


def _fill_model_tables(dcfg, model, foot_frames, chest_frame):
    dcfg[H["HB_KD_TOTAL_MASS"]] = model.total_mass()
    for f, fr in enumerate(foot_frames):
        _, R, t = model.frames[fr]
        dcfg[H["HB_KD_FOOT_R0"] + 9 * f:H["HB_KD_FOOT_R0"] + 9 * f + 9] = R.ravel()
        dcfg[H["HB_KD_FOOT_T0"] + 3 * f:H["HB_KD_FOOT_T0"] + 3 * f + 3] = t
    dcfg[H["HB_KD_CHEST_R0"]:H["HB_KD_CHEST_R0"] + 9] = model.frames[chest_frame][1].ravel()
    st = H["HB_KD_BODY_STRIDE"]
    for b in range(model.n_bodies):
        o = H["HB_KD_BODY0"] + st * b
        dcfg[o:o + 9] = model.joint_rot[b].ravel()
        dcfg[o + 9:o + 12] = model.joint_xyz[b]
        dcfg[o + 12:o + 15] = model.joint_axis[b]
        dcfg[o + 15] = model.mass[b]
        dcfg[o + 16:o + 19] = model.com[b]
        dcfg[o + 19:o + 28] = model.inertia[b].ravel()


class PoseEvaluator(KinoEvaluator):
    """Evaluator of the static pose finder
    (`/root/reference/src/hippopt/turnkey_planners/humanoid_pose_finder/planner.py:303-413`), the one
    reference configuration IPOPT solves with the exact Hessian.  ``PoseSettings(terrain="smooth_steps",
    n_terrain_params=10)`` poses it on the stairs, ``PoseSettings(terrain="tilted_steps", n_terrain_params=10 K)`` on K
    general smooth steps (the ramp), with the steps' parameters appended to p."""

    def __init__(self, model: RobotModel, settings=None):
        from .pose_layout import PoseLayout, PoseSettings

        _Evaluator.__init__(self)
        self.model = model
        self.settings = s = settings or PoseSettings()
        self.layout = lay = PoseLayout(model, s)
        po = lay.po
        icfg = np.zeros(H["HB_KI_COUNT"], dtype=np.int32)
        ints = {
            "HORIZON": 1, "N_X": lay.n_x, "N_P": lay.n_p, "M": lay.m, "NNZ_J": lay.nnz_j, "NNZ_H": lay.nnz_h,
            "N_JC": lay.n_jc, "N_JK": lay.n_jk, "N_HC": lay.n_hc, "TERRAIN": lay.kernel_terrain,
            "HAS_FINAL": 0, "HAS_PERIODICITY": 0, "PO_TERRAIN": po.terrain,
            "H_INIT": 0, "PO_DESC0": po.desc0, "PO_MASS": po.mass, "PO_INIT": po.ref, "PO_GRAVITY": po.gravity,
            "PO_EPS": po.eps, "PO_MU": po.mu, "PO_MAX_S": po.max_s, "PO_MIN_S": po.min_s,
            "N_BODIES": model.n_bodies, "FOOT_BODY_L": model.frames[s.foot_frames[0]][0],
            "FOOT_BODY_R": model.frames[s.foot_frames[1]][0],
            "CHEST_BODY": model.frames[s.frame_quaternion_cost_frame][0],
            "KIND": 1, "X_STRIDE": 0, "COST_K0": 0, "JOINT_COST_KIND": 1, "PO_FQ": po.ref_fq,
            "PO_BQ": po.ref + po.ST_Q, "PO_BQV": po.ref + po.ST_Q, "PO_JR": po.ref + po.ST_S, "REF_STRIDE": 0,
        }
        for k, v in ints.items():
            icfg[H["HB_KI_" + k]] = v
        icfg[H["HB_KI_ZMAP0"]:H["HB_KI_ZMAP0"] + 189] = lay.zmap
        icfg[H["HB_KI_PARENT0"]:H["HB_KI_PARENT0"] + model.n_bodies] = model.parent
        for fid in range(H["HB_KF_COUNT"]):
            icfg[H["HB_KI_FAM0"] + 4 * fid:H["HB_KI_FAM0"] + 4 * fid + 4] = (-1, 0, 1, 0)

        def put_fam(fid, name):
            icfg[H["HB_KI_FAM0"] + 4 * fid:H["HB_KI_FAM0"] + 4 * fid + 4] = lay.fam[name]

        for i in range(8):
            base = i * H["HB_KF_PT_COUNT"]
            put_fam(base + H["HB_KF_PT_DCC"], f"pt{i}.complementarity")
            put_fam(base + H["HB_KF_PT_HEIGHT"], f"pt{i}.height")
            put_fam(base + H["HB_KF_PT_NORMAL"], f"pt{i}.normal")
            put_fam(base + H["HB_KF_PT_FRICTION"], f"pt{i}.friction")
            put_fam(base + H["HB_KF_PT_FK"], f"pt{i}.fk")
        put_fam(H["HB_KF_UNIT_QUAT"], "unit_quat")
        put_fam(H["HB_KF_COM_KIN"], "com_kin")
        put_fam(H["HB_KF_H_DYN"], "balance")
        put_fam(H["HB_KF_S_BOUNDS"], "s_bounds")
        dcfg = np.zeros(H["HB_KD_COUNT"], dtype=np.float64)
        # cost-weight slots shared with the kinodynamic table (csrc/pose_contact.cu header)
        dcfg[H["HB_KD_W_CENTROID"]] = s.com_regularization_cost_multiplier
        dcfg[H["HB_KD_W_RATIO"]] = s.average_force_regularization_cost_multiplier
        dcfg[H["HB_KD_W_SWING"]] = s.point_position_regularization_cost_multiplier
        dcfg[H["HB_KD_W_FD"]] = s.force_regularization_cost_multiplier
        dcfg[H["HB_KD_W_FRAME"]] = s.desired_frame_quaternion_cost_multiplier
        dcfg[H["HB_KD_W_BQ"]] = s.base_quaternion_cost_multiplier
        dcfg[H["HB_KD_W_JOINT"]] = s.joint_regularization_cost_multiplier
        dcfg[H["HB_KD_WJ0"]:H["HB_KD_WJ0"] + NJ] = s.joint_regularization_cost_weights
        _fill_model_tables(dcfg, model, s.foot_frames, s.frame_quaternion_cost_frame)
        self._create_handle(icfg, dcfg, lay)


class ToyEvaluator(_Evaluator):
    """Mass-falling OCP of `/root/reference/test/test_multiple_shooting.py:253-353`; p = [g, x0, v0]."""

    def __init__(self, horizon: int = 100, integrator: str = "euler", dt: float = 0.01):
        super().__init__()
        kind = {"euler": 0, "trapezoid": 1}[integrator]
        _capi.check(_capi.lib().hb_toy_create(horizon, kind, dt, ctypes.byref(self._h)), "hb_toy_create")
        self.horizon, self.dt = horizon, dt
        self._read_dims()

    def _pattern(self, fn, nnz):
        colind = np.zeros(self.n_x + 1, dtype=np.int64)
        row = np.zeros(nnz, dtype=np.int64)
        i64p = ctypes.POINTER(ctypes.c_int64)
        _capi.check(fn(self._h, colind.ctypes.data_as(i64p), row.ctypes.data_as(i64p)), "hb_pattern")
        return colind, row

    def jac_sparsity(self):
        return self._pattern(_capi.lib().hb_pattern_jac, self.nnz_j)

    def hess_sparsity(self):
        return self._pattern(_capi.lib().hb_pattern_hess, self.nnz_h)

    def bounds(self, p):
        """(lbg, ubg) in the row order of the test's subject_to calls."""
        p = np.atleast_2d(np.asarray(p, dtype=np.float64))
        N = self.horizon
        B = p.shape[0]
        lb = np.zeros((B, self.m))
        ub = np.zeros((B, self.m))
        o = 2 * (N - 1)
        lb[:, o] = ub[:, o] = p[:, 1]
        lb[:, o + 1] = ub[:, o + 1] = p[:, 2]
        o += 2
        lb[:, o] = ub[:, o] = p[:, 1]
        o += N
        lb[:, o] = ub[:, o] = p[:, 2]
        o += N
        lb[:, o:o + 3 * (N - 1)] = 5.0
        ub[:, o:o + 3 * (N - 1)] = np.inf
        o += 3 * (N - 1)
        lb[:, o + 3:o + 6] = ub[:, o + 3:o + 6] = 6.0
        return lb, ub


def probe_fp64_tflops() -> float:
    v = ctypes.c_double()
    _capi.check(_capi.lib().hb_probe_fp64_tflops(ctypes.byref(v), None), "hb_probe_fp64_tflops")
    return float(v.value)
