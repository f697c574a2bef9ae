"""The solver back end behind hippopt's `OptimizationSolver` interface (SURVEY.md 8(b), row a30).

Two classes:

* `B200Solver` -- casadi-free.  The 16 methods of `OptimizationSolver`
  (`/root/reference/src/hippopt/base/optimization_solver.py:24-96`) plus `cost_function()`
  (`multiple_shooting_solver.py:906-907` calls it although it is not in the ABC) over the TEMPLATE problems this
  library evaluates (kinodynamic OCP, pose finder, toy OCP): a batch of B instances is solved on the device by
  `hippopt_b200.ipsolver.BatchedInteriorPoint`; `get_values()` / `get_cost_values()` / `get_constraint_multipliers()`
  return what `OptiSolver.solve()` stores (`base/opti_solver.py:522-537`), one entry per instance.  Expressions are
  not CasADi graphs here but handles on the template's named expressions (hippopt_b200/naming.py): `add_cost` /
  `add_constraint` switch the optional ones on, exactly the switch `ExpressionType.skip / subject_to / minimize`
  is for the reference's `final_state_expression` and `periodicity_expression` (`planner.py:417, 923`).

* `make_opti_solver(cs, hp)` -> `B200OptiSolver(hp.OptiSolver)` -- the CasADi shim: needs `casadi` and `hippopt`, so it
  is built by a factory that receives the two modules (import-guarded: `install()` raises a clear error where they are
  missing; the unit tests pass small recording stand-ins).  It overrides `solve()` only (`opti_solver.py:444-537`):
  the planners keep building their Opti graph, and at solve time the five nlpsol oracle functions are replaced by
  `cs.Callback`s that forward to `hb_eval_host` through ONE shared pipeline with an x-keyed cache (two launches per
  IPOPT iterate: f / grad_f / g / jac_g at a new x, hess_l when the multipliers arrive).

Template matching never trusts dimensions alone: `OracleBridge.verify` evaluates Opti's own f and g once at the
initial point and compares with the kernels (1e-9 relative to the vector's scale) before IPOPT is started; a problem
that does not match falls back to the stock `OptiSolver.solve()`.
"""
from __future__ import annotations

import copy
import dataclasses
import logging

import numpy as np

from . import naming

LOG = logging.getLogger("[hippopt_b200::plugin]")


# ---------------------------------------------------------------------------------------------------------------
# exceptions with the reference's texts (optimization_solver.py:13-21)
class SolutionNotAvailableException(Exception):
    def __init__(self):
        super().__init__("No solution is available. Was solve() called successfully?")


class ProblemNotRegisteredException(Exception):
    def __init__(self):
        super().__init__("No problem has been registered.")


# ---------------------------------------------------------------------------------------------------------------
# nlpsol option handling shared by both classes
# Options of CasADi's nlpsol that cannot be forwarded when the oracle functions are Callbacks [ext]:
#   expand                SX-expands the MX graph: a Callback node cannot be expanded
#   detect_simple_bounds  rewrites g / lbx / ubx from the symbolic g: done explicitly by RowReduction instead
#   cse, ...              graph transformations, meaningless for an opaque evaluator
UNFORWARDABLE_PLUGIN_OPTIONS = ("expand", "detect_simple_bounds", "cse", "common_options", "jit", "jit_options",
                                "specific_options", "verbose_init")


def split_plugin_options(options_plugin: dict) -> tuple[dict, dict]:
    """(options to forward to nlpsol, options consumed here)."""
    fwd = {k: v for k, v in (options_plugin or {}).items() if k not in UNFORWARDABLE_PLUGIN_OPTIONS}
    used = {k: v for k, v in (options_plugin or {}).items() if k in UNFORWARDABLE_PLUGIN_OPTIONS}
    return fwd, used


class RowReduction:
    """`detect_simple_bounds` made explicit: rows of g that are a bare variable become bounds on x.

    IPOPT then sees `g[general]` with `lbx / ubx`; multipliers come back on the reference's full row set:
    lam_g[general] from IPOPT's lam_g, lam_g[simple row i of x_j] = lam_x[j] (one row per variable; where several rows
    bound the same variable the multiplier goes to the row whose bound is the active one)."""

    def __init__(self, layout, enabled: bool, include_equalities: bool = False):
        m, n = layout.m, layout.n_x
        self.m, self.n = m, n
        if enabled and hasattr(layout, "simple_bound_rows"):
            self.simple, self.target = layout.simple_bound_rows(include_equalities)
        else:
            self.simple, self.target = np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
        keep = np.ones(m, dtype=bool)
        keep[self.simple] = False
        self.general = np.nonzero(keep)[0]
        self.m_reduced = len(self.general)
        new_row = -np.ones(m, dtype=np.int64)
        new_row[self.general] = np.arange(self.m_reduced)
        jrow = np.asarray(layout.jac_row)
        self.jac_keep = np.nonzero(keep[jrow])[0]                     # entries of the full CCS value array that stay
        jcol = np.repeat(np.arange(n), np.diff(np.asarray(layout.jac_colind)))
        self.jac_row = new_row[jrow[self.jac_keep]]
        counts = np.bincount(jcol[self.jac_keep], minlength=n)
        self.jac_colind = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)

    def g(self, g_full):
        return g_full[..., self.general]

    def jac(self, jac_full):
        return jac_full[..., self.jac_keep]

    def lam_full(self, lam_reduced):
        """multipliers IPOPT hands to hess_l -> the kernels' full row set (simple rows are linear: no Hessian)."""
        out = np.zeros(lam_reduced.shape[:-1] + (self.m,))
        out[..., self.general] = lam_reduced
        return out

    def bounds(self, lbg, ubg):
        """(lbg_reduced, ubg_reduced, lbx, ubx) from the full canonical bounds."""
        lbx, ubx = np.full(self.n, -np.inf), np.full(self.n, np.inf)
        np.maximum.at(lbx, self.target, lbg[self.simple])
        np.minimum.at(ubx, self.target, ubg[self.simple])
        return lbg[self.general], ubg[self.general], lbx, ubx

    def multipliers(self, lam_g_reduced, lam_x, x, lbg, ubg):
        lam = self.lam_full(np.asarray(lam_g_reduced, dtype=np.float64))
        lam_x = np.asarray(lam_x, dtype=np.float64)
        for r, j in zip(self.simple, self.target):
            # IPOPT's sign: negative on an active lower bound, positive on an active upper bound
            active_low = abs(x[j] - lbg[r]) <= abs(ubg[r] - x[j])
            if (lam_x[j] <= 0.0) == bool(active_low) or lam_x[j] == 0.0:
                lam[r] = lam_x[j]
        return lam


class OracleCache:
    """One shared evaluation pipeline for the five nlpsol oracle functions of ONE instance.

    IPOPT asks for f, grad_f, g and jac_g through separate callbacks at the same x, and for hess_l later with the
    updated multipliers [ext]; the kernels produce any subset in one pass.  The first request at a new x runs
    F|GRAD_F|G|JAC_G once and the other three return views of the cached host buffers; hess_l runs HESS_L alone.
    `host_eval(mask, x, lam, sigma) -> dict` is `HostEvaluator.__call__` below (hb_eval_host) or a test double."""

    def __init__(self, host_eval, masks):
        self.host_eval, self.masks = host_eval, masks  # masks: dict name -> bit
        self._x_key, self._first = None, None
        self.launches = {"first_order": 0, "hess": 0}
        self.calls = {k: 0 for k in ("f", "grad_f", "g", "jac", "hess")}

    def first_order(self, x: np.ndarray) -> dict:
        key = x.tobytes()
        if key != self._x_key:
            m = self.masks
            self._first = self.host_eval(m["f"] | m["grad_f"] | m["g"] | m["jac"], x, None, None)
            self._first = {k: np.array(v, copy=True) for k, v in self._first.items()}
            self._x_key = key
            self.launches["first_order"] += 1
        return self._first

    def get(self, name: str, x: np.ndarray) -> np.ndarray:
        self.calls[name] += 1
        return self.first_order(x)[name]

    def hess(self, x: np.ndarray, lam: np.ndarray, sigma: float) -> np.ndarray:
        self.calls["hess"] += 1
        self.launches["hess"] += 1
        return np.array(self.host_eval(self.masks["hess"], x, lam, np.atleast_1d(float(sigma)))["hess"], copy=True)


class HostEvaluator:
    """`hb_eval_host` for one instance with pinned buffers (two pipelines over one handle: first-order mask and
    Hessian mask); parameters are uploaded once per solve (`hb_host_set_parameters`)."""

    def __init__(self, ev):
        import torch

        from .evaluator import F, G, GRAD_F, HESS_L, JAC_G, HostPipeline

        self.ev, self.torch = ev, torch
        self.masks = {"f": F, "grad_f": GRAD_F, "g": G, "jac": JAC_G, "hess": HESS_L}
        self.first = HostPipeline(ev, 1, F | GRAD_F | G | JAC_G)
        self.second = HostPipeline(ev, 1, HESS_L)
        # x | lam_g | sigma in one pinned block: one host-to-device copy per evaluation (hb_eval_host merges adjacent ranges)
        blk = HostPipeline.host_buffer((ev.n_x + ev.m + 1,))
        self.x_host = blk[:ev.n_x].view(1, ev.n_x)
        self.lam_host = blk[ev.n_x:ev.n_x + ev.m].view(1, ev.m)
        self.sig_host = blk[ev.n_x + ev.m:]
        self._blk = blk

    def set_parameters(self, p: np.ndarray) -> None:
        self.first.set_parameters(self.torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64).ravel()))

    def __call__(self, mask, x, lam, sigma):
        self.x_host[0].copy_(self.torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64).ravel()))
        if mask & self.masks["hess"]:
            self.lam_host[0].copy_(self.torch.from_numpy(np.ascontiguousarray(lam, dtype=np.float64).ravel()))
            self.sig_host[0] = float(np.ravel(sigma)[0])
            out = self.second.run(self.x_host, self.lam_host, self.sig_host)
        else:
            out = self.first.run(self.x_host)
        return {k: v[0].numpy() if v.dim() > 1 else v.numpy() for k, v in out.items()}


# ---------------------------------------------------------------------------------------------------------------
# template matching
@dataclasses.dataclass
class TemplateMatch:
    kind: str                 # "kinodynamic" | "pose_finder" | "toy"
    horizon: int = 0
    final_state: bool = False
    periodicity: bool = False
    smooth_terrain: bool = False
    n_terrain_params: int = 0


def match_template(nx: int, np_: int, ng: int) -> TemplateMatch | None:
    """Dimensions of the baked Opti problem -> the template they belong to (SURVEY.md Appendix B), or None.
    kinodynamic: n_x = 189 N + 6, n_p = 79 N + 326 (+ terrain parameters), m from the constraint families.
    pose finder: (81, 202, 89), or (81, 212, 89) on the smooth steps, whose ten parameters are appended to p."""
    from .kino_layout import NZ, count_rows

    if nx == 81 and np_ in (202, 212) and ng == 89:   # pose finder, Appendix B.4
        n_terr = np_ - 202
        return TemplateMatch("pose_finder", smooth_terrain=n_terr > 0, n_terrain_params=n_terr)
    if nx % 9 == 0 and np_ == 3 and ng in (7 * (nx // 9) + 3, 7 * (nx // 9) + 2):  # toy OCP: 9 N variables
        return TemplateMatch("toy", horizon=nx // 9)
    if nx > 6 and (nx - 6) % NZ == 0:
        N = (nx - 6) // NZ
        base_p = 79 * N + 326
        for n_terr in (0, 10):
            if np_ != base_p + n_terr:
                continue
            for fin in (False, True):
                for per in (False, True):
                    if count_rows(N, fin, per) == ng:
                        return TemplateMatch("kinodynamic", N, fin, per, n_terr > 0, n_terr)
    return None


# ---------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass(frozen=True)
class TemplateExpression:
    """Handle on a named expression of a template problem (stands where the reference has a `cs.MX`)."""

    name: str
    kind: str  # "cost" | "constraint"

    def __str__(self):
        return self.name


class _FlatLayout:
    """Sizes and bounds of an evaluator that has no layout object of its own."""

    def __init__(self, ev):
        self.n_x, self.n_p, self.m = ev.n_x, ev.n_p, ev.m
        self.bounds = ev.bounds


class B200Solver:
    """casadi-free `OptimizationSolver` over a template problem, B instances at once (module docstring)."""

    def __init__(self, model=None, settings=None, batch: int = 1, device="cuda:0", options_solver: dict | None = None,
                 options_plugin: dict | None = None, callback_criterion=None, evaluator=None, kkt: str = "stage"):
        from .kino_layout import KinoSettings

        self._model = model
        self._settings = settings if settings is not None else KinoSettings()
        self._batch, self._device = int(batch), device
        self._options_solver = dict(options_solver or {})
        self._options_plugin, self._consumed_options = split_plugin_options(options_plugin or {})
        self._callback_criterion = callback_criterion
        self._kkt = kkt
        self._ev = evaluator
        self._problem = None
        self._objects = self._objects_structure = None
        self._guess = None
        self._cost_expressions: dict[str, TemplateExpression] = {}
        self._constraint_expressions: dict[str, TemplateExpression] = {}
        self._output_solution = self._output_cost = self._cost_values = self._constraint_values = None
        self._last_output = None

    # -- structure ---------------------------------------------------------------------------------------
    def _evaluator(self):
        if self._ev is None:
            from .evaluator import KinoEvaluator

            if self._model is None:
                raise ValueError("B200Solver needs a RobotModel (model=) or an evaluator (evaluator=)")
            self._ev = KinoEvaluator(self._model, self._settings)
        return self._ev

    def _layout(self):
        if self._ev is not None:
            if hasattr(self._ev, "layout"):
                return self._ev.layout
            return _FlatLayout(self._ev)  # templates without a field / name table (toy OCP)
        from .kino_layout import KinoLayout

        if self._model is None:
            raise ValueError("B200Solver needs a RobotModel (model=) or an evaluator (evaluator=)")
        return KinoLayout(self._model, self._settings)

    def generate_optimization_objects(self, input_structure=None, **kwargs):
        """`input_structure`: {"x": (B, n_x) or (n_x,), "p": (B, n_p) or (n_p,)} numeric arrays -- what the reference
        passes as a tree of numpy fields (optimization_solver.py:25-29), flattened along Appendix B.  Returns the
        "objects": index arrays into x / p per field group (the stand-in for Opti variables / parameters)."""
        lay = self._layout()
        if input_structure is not None and not isinstance(input_structure, dict):
            raise ValueError("The input structure is neither an optimization object nor a list.")
        self._objects_structure = copy.deepcopy(input_structure)
        self._objects = {"x": np.arange(lay.n_x), "p": np.arange(lay.n_p),
                         "constraints": naming.constraint_rows(lay), "costs": naming.cost_names(lay)}
        for name in self._objects["constraints"]:
            self._constraint_expressions[name] = TemplateExpression(name, "constraint")
        for name in self._objects["costs"]:
            self._cost_expressions[name] = TemplateExpression(name, "cost")
        if kwargs.get("fill_initial_guess", True) and input_structure is not None:
            self.set_initial_guess(input_structure)
        return self._objects

    def get_optimization_objects(self):
        return self._objects

    def get_optimization_structure(self):
        return self._objects_structure

    def register_problem(self, problem) -> None:
        self._problem = problem

    def get_problem(self):
        if self._problem is None:
            raise ProblemNotRegisteredException
        return self._problem

    def set_initial_guess(self, initial_guess) -> None:
        lay = self._layout()
        if not isinstance(initial_guess, dict) or "x" not in initial_guess or "p" not in initial_guess:
            raise ValueError("The guess must be a dict with the fields 'x' and 'p'.")
        x = np.atleast_2d(np.asarray(initial_guess["x"], dtype=np.float64))
        p = np.atleast_2d(np.asarray(initial_guess["p"], dtype=np.float64))
        if x.shape[1] != lay.n_x:
            raise ValueError(f"The guess has the field x but its dimension ({x.shape}) does not match with the "
                             f"corresponding optimization variable ({lay.n_x}).")
        if p.shape[1] != lay.n_p:
            raise ValueError(f"The guess has the field p but its dimension ({p.shape}) does not match with the "
                             f"corresponding optimization variable ({lay.n_p}).")
        self._guess = {"x": np.broadcast_to(x, (self._batch, lay.n_x)).copy(),
                       "p": np.broadcast_to(p, (self._batch, lay.n_p)).copy()}
        if "lam_g" in initial_guess:  # warm start (main_single_step_flat_ground.py:120-125: previous Output as guess)
            self._guess["lam_g"] = np.broadcast_to(np.atleast_2d(initial_guess["lam_g"]), (self._batch, lay.m)).copy()

    def get_initial_guess(self):
        return copy.deepcopy(self._guess)

    # -- expressions -------------------------------------------------------------------------------------
    _OPTIONAL = {"final_state_expression": "final_state_constraint", "periodicity_expression": "periodicity_constraint"}

    def add_cost(self, input_cost, name: str = None) -> None:
        name = str(input_cost) if name is None else name
        if name in self._cost_expressions and self._objects is None:
            raise ValueError("The cost " + name + " is already present.")
        if not isinstance(input_cost, TemplateExpression) or input_cost.kind != "cost":
            raise ValueError("Only the template's own cost expressions can be added (naming.cost_slots).")
        if self._objects is not None and name not in self._objects["costs"]:
            raise ValueError("The cost " + name + " is not an expression of this template.")
        self._cost_expressions[name] = input_cost

    def add_constraint(self, input_constraint, name: str = None) -> None:
        name = str(input_constraint) if name is None else name
        if not isinstance(input_constraint, TemplateExpression) or input_constraint.kind != "constraint":
            raise ValueError("Only the template's own constraint expressions can be added (naming.constraint_rows).")
        if name in self._OPTIONAL:
            if getattr(self._settings, self._OPTIONAL[name]):
                raise ValueError("The constraint " + name + " is already present.")
            self._settings = dataclasses.replace(self._settings, **{self._OPTIONAL[name]: True})
            self._ev = None  # other row set: new layout / handle
            if self._objects is not None:
                self.generate_optimization_objects(self._objects_structure, fill_initial_guess=False)
        elif name in self._constraint_expressions:
            raise ValueError("The constraint " + name + " is already present.")
        self._constraint_expressions[name] = input_constraint

    def cost_function(self):
        return list(self._cost_expressions.values())

    def get_cost_expressions(self):
        return self._cost_expressions

    def get_constraint_expressions(self):
        return self._constraint_expressions

    # -- solve -------------------------------------------------------------------------------------------
    def solve(self) -> None:
        import torch

        from .ipsolver import BatchedInteriorPoint

        if self._guess is None:
            raise ValueError("The following parameters are not set: ['p'] (set_initial_guess was not called)")
        ev, lay = self._evaluator(), self._layout()
        dev = torch.device(self._device)
        x0 = torch.as_tensor(self._guess["x"], device=dev)
        p = torch.as_tensor(self._guess["p"], device=dev)
        lbg, ubg = lay.bounds(self._guess["p"])
        ip = BatchedInteriorPoint(ev, kkt=self._kkt, ipopt_options=self._options_solver,
                                  callback_criterion=self._callback_criterion)
        out = ip.solve(x0, p, lbg, ubg, lam0=self._guess.get("lam_g"))  # raises OptiFailure like opti_solver.py:520
        self._last_output = out
        x = out.values.contiguous()
        pose = naming.is_pose_layout(lay)
        terms = ev.cost_terms(x, p).cpu().numpy() if (hasattr(ev, "cost_terms") and not pose) else None
        xs, lam = x.cpu().numpy(), out.constraint_multipliers.cpu().numpy()
        self._output_cost = out.cost_value.cpu().numpy()
        from . import solution

        self._output_solution = [solution.values_dict(lay, xs[b], self._guess["p"][b]) for b in range(self._batch)]
        if terms is not None:
            self._cost_values = [naming.cost_values(lay, terms[b]) for b in range(self._batch)]
        elif pose:  # the pose finder's 28 named costs, from the solution on the host
            model = self._model if self._model is not None else getattr(lay, "model", None)
            self._cost_values = [naming.pose_cost_values(lay, model, xs[b], self._guess["p"][b])
                                 for b in range(self._batch)]
        else:
            self._cost_values = [{} for _ in range(self._batch)]
        self._constraint_values = [naming.constraint_multipliers(lay, lam[b]) for b in range(self._batch)]
        self._solution_vectors = {"x": xs, "lam_g": lam, "p": self._guess["p"]}

    def get_solution_sensitivity(self, param_idx, delta: float = 0.0, delta_c: float = 0.0):
        """d x* / d p[:, param_idx] of the last solve, (B, n_x, k): the counterpart of differentiating the reference's
        `OptiSolver.to_function(...)` (opti_solver.py:597-638, main_sensitivity.py:213-247) -- one more KKT solve with a
        right-hand side per parameter (hippopt_b200/sensitivity.py)."""
        import torch

        from .sensitivity import solution_sensitivity

        if self._output_solution is None:
            raise SolutionNotAvailableException
        ev, lay = self._evaluator(), self._layout()
        dev = torch.device(self._device)
        sv = self._solution_vectors
        dx, _, _ = solution_sensitivity(ev, torch.as_tensor(sv["x"], device=dev), torch.as_tensor(sv["lam_g"], device=dev),
                                        torch.as_tensor(sv["p"], device=dev), lay.bounds, param_idx, kkt=self._kkt,
                                        delta=delta, delta_c=delta_c)
        return dx.cpu().numpy()

    def get_values(self):
        if self._output_solution is None:
            raise SolutionNotAvailableException
        return self._output_solution

    def get_cost_value(self):
        if self._output_cost is None:
            raise SolutionNotAvailableException
        return self._output_cost

    def get_cost_values(self):
        return self._cost_values

    def get_constraint_multipliers(self):
        return self._constraint_values

    def get_solution_vectors(self):
        """x / lam_g / p of the last solve: the guess of a warm-started next solve (`set_initial_guess`)."""
        if self._output_solution is None:
            raise SolutionNotAvailableException
        return self._solution_vectors


# ---------------------------------------------------------------------------------------------------------------
# CasADi side
class OracleBridge:
    """Builds the Callback-backed nlpsol for one matched template and runs it (needs the casadi module `cs`)."""

    def __init__(self, cs, layout, host_eval, masks, detect_simple_bounds: bool, include_equalities: bool = False):
        self.cs, self.layout = cs, layout
        self.cache = OracleCache(host_eval, masks)
        self.red = RowReduction(layout, detect_simple_bounds, include_equalities)
        self._callbacks = []  # keep references: CasADi does not own Python callbacks

    def _callback(self, name, n_in, sp_in, sp_out, fn):
        cs = self.cs

        class _Oracle(cs.Callback):
            def __init__(cb):
                cs.Callback.__init__(cb)
                cb.construct(name, {})

            def get_n_in(cb):
                return n_in

            def get_n_out(cb):
                return len(sp_out)

            def get_sparsity_in(cb, i):
                return sp_in[i]

            def get_sparsity_out(cb, i):
                return sp_out[i]

            def eval(cb, arg):
                vals = fn(*[np.asarray(a, dtype=np.float64).ravel() for a in arg])
                return [cs.DM(sp, np.asarray(v, dtype=np.float64).ravel()) if sp.nnz() != sp.numel()
                        else cs.DM(np.asarray(v, dtype=np.float64).reshape(sp.size1(), sp.size2()))
                        for sp, v in zip(sp_out, vals)]

        cb = _Oracle()
        self._callbacks.append(cb)
        return cb

    def build(self, options_plugin: dict, options_solver: dict, inner_solver: str = "ipopt"):
        cs, lay, red, cache = self.cs, self.layout, self.red, self.cache
        n, npar, mr = lay.n_x, lay.n_p, red.m_reduced
        dense = lambda r: cs.Sparsity.dense(r, 1)  # noqa: E731
        jac_sp = cs.Sparsity(mr, n, [int(v) for v in red.jac_colind], [int(v) for v in red.jac_row])
        hes_sp = cs.Sparsity(n, n, [int(v) for v in lay.hess_colind], [int(v) for v in lay.hess_row])
        xs, ps, one = dense(n), dense(npar), dense(1)
        f_cb = self._callback("hb_nlp_f", 2, [xs, ps], [one], lambda x, p: [cache.get("f", x)])
        g_cb = self._callback("hb_nlp_g", 2, [xs, ps], [dense(mr)], lambda x, p: [red.g(cache.get("g", x))])
        # nlpsol's oracle signatures [ext]: nlp_grad_f (x, p) -> (f, grad_f); nlp_jac_g (x, p) -> (g, jac_g);
        # nlp_hess_l (x, p, lam_f, lam_g) -> triu(hess_l)
        grad_cb = self._callback("hb_nlp_grad_f", 2, [xs, ps], [one, xs],
                                 lambda x, p: [cache.get("f", x), cache.get("grad_f", x)])
        jac_cb = self._callback("hb_nlp_jac_g", 2, [xs, ps], [dense(mr), jac_sp],
                                lambda x, p: [red.g(cache.get("g", x)), red.jac(cache.get("jac", x))])
        hess_cb = self._callback("hb_nlp_hess_l", 4, [xs, ps, one, dense(mr)], [hes_sp],
                                 lambda x, p, sig, lam: [cache.hess(x, red.lam_full(lam), float(sig[0]))])
        x_sym, p_sym = cs.MX.sym("x", n), cs.MX.sym("p", npar)
        nlp = {"x": x_sym, "p": p_sym, "f": f_cb(x_sym, p_sym), "g": g_cb(x_sym, p_sym)}
        opts, consumed = split_plugin_options(options_plugin)
        opts = dict(opts)
        opts[inner_solver] = dict(options_solver or {})
        opts.update({"grad_f": grad_cb, "jac_g": jac_cb, "hess_lag": hess_cb,
                     "calc_lam_p": False})  # d/dp of a Callback cannot be generated [ext]
        if str((options_solver or {}).get("hessian_approximation", "exact")) == "limited-memory":
            opts.pop("hess_lag")  # IPOPT's L-BFGS never asks for hess_l (main_periodic_step.py:116)
        self.options_passed = opts
        self.solver = cs.nlpsol("solver", inner_solver, nlp, opts)
        return self.solver

    def build_external(self, options_plugin: dict, options_solver: dict, inner_solver: str, library_path: str, handle):
        """The compiled alternative to the Callbacks: CasADi loads the five oracle functions from the library by name
        (`casadi.external`, the codegen ABI exported by include/hippopt_b200.h) after the problem has been bound to
        them (`hb_external_bind`); no Python runs inside IPOPT's iteration.  The external functions work on the full
        row set, so `detect_simple_bounds` is not applied in this mode (bounds stay rows of g)."""
        from . import _capi

        cs, lay = self.cs, self.layout
        _capi.check(_capi.lib().hb_external_bind(handle), "hb_external_bind")
        self.red = RowReduction(lay, False)
        ext = {n: cs.external(n, library_path) for n in ("hb_nlp_f", "hb_nlp_g", "hb_nlp_grad_f", "hb_nlp_jac_g", "hb_nlp_hess_l")}
        x_sym, p_sym = cs.MX.sym("x", lay.n_x), cs.MX.sym("p", lay.n_p)
        nlp = {"x": x_sym, "p": p_sym, "f": ext["hb_nlp_f"](x_sym, p_sym), "g": ext["hb_nlp_g"](x_sym, p_sym)}
        opts, _ = split_plugin_options(options_plugin)
        opts = dict(opts)
        opts[inner_solver] = dict(options_solver or {})
        opts.update({"grad_f": ext["hb_nlp_grad_f"], "jac_g": ext["hb_nlp_jac_g"], "hess_lag": ext["hb_nlp_hess_l"],
                     "calc_lam_p": False})
        if str((options_solver or {}).get("hessian_approximation", "exact")) == "limited-memory":
            opts.pop("hess_lag")
        self.options_passed = opts
        self._callbacks = list(ext.values())
        self.solver = cs.nlpsol("solver", inner_solver, nlp, opts)
        return self.solver

    def verify(self, x0, p, f_ref: float, g_ref: np.ndarray, rtol: float = 1e-9) -> None:
        """One evaluation of the kernels at the initial point against Opti's own f and g (same canonical form)."""
        first = self.cache.first_order(np.ascontiguousarray(x0, dtype=np.float64))
        f = float(np.ravel(first["f"])[0])
        g = np.asarray(first["g"]).ravel()
        fs = max(abs(f_ref), 1e-300)
        gs = max(float(np.abs(g_ref).max()) if g_ref.size else 0.0, 1e-300)
        if abs(f - f_ref) > rtol * fs or (g_ref.size and float(np.abs(g - g_ref).max()) > rtol * gs):
            raise TemplateMismatch(f"kernel evaluation differs from the Opti graph at the initial point: "
                                   f"f {f} vs {f_ref}, max |dg| {float(np.abs(g - g_ref).max()) if g_ref.size else 0.0}")

    def run(self, x0, p, lbg, ubg, lam_g0=None):
        red = self.red
        lbg_r, ubg_r, lbx, ubx = red.bounds(np.asarray(lbg, dtype=np.float64), np.asarray(ubg, dtype=np.float64))
        args = dict(x0=x0, p=p, lbg=lbg_r, ubg=ubg_r, lbx=lbx, ubx=ubx)
        if lam_g0 is not None:
            args["lam_g0"] = red.g(np.asarray(lam_g0, dtype=np.float64))
        sol = self.solver(**args)
        x = np.asarray(sol["x"], dtype=np.float64).ravel()
        lam = red.multipliers(np.asarray(sol["lam_g"]).ravel(), np.asarray(sol["lam_x"]).ravel(), x,
                              np.asarray(lbg, dtype=np.float64), np.asarray(ubg, dtype=np.float64))
        return x, float(np.asarray(sol["f"]).ravel()[0]), lam, self.solver.stats()


class TemplateMismatch(Exception):
    pass


def make_opti_solver(cs, hp, evaluator_factory=None):
    """-> class B200OptiSolver(hp.OptiSolver): overrides solve() (`base/opti_solver.py:444-537`).

    `evaluator_factory(match: TemplateMatch) -> (layout, host_eval, masks)`; the default builds the CUDA evaluator
    from `B200OptiSolver.robot_model` / `.kino_settings` (set by `install`)."""

    class B200OptiSolver(hp.OptiSolver):
        robot_model = None        # hippopt_b200.robot_model.RobotModel of the planner's URDF / joint list
        kino_settings = None      # hippopt_b200.kino_layout.KinoSettings mirroring the planner's Settings
        strict = False            # True: a template mismatch raises instead of falling back to the stock path
        oracle = "callback"       # "callback": cs.Callback objects (Python inside the iteration, simple bounds reduced);
        #                           "external": casadi.external on the library's codegen ABI (no Python in the loop)
        last_bridge = None        # for inspection: launches / calls per solve

        def _default_factory(self, match: TemplateMatch):
            from .evaluator import KinoEvaluator, PoseEvaluator, ToyEvaluator

            if match.kind == "kinodynamic":
                st = dataclasses.replace(self.kino_settings, horizon=match.horizon,
                                         final_state_constraint=match.final_state,
                                         periodicity_constraint=match.periodicity,
                                         terrain="smooth_steps" if match.smooth_terrain else "planar",
                                         n_terrain_params=match.n_terrain_params)
                ev = KinoEvaluator(self.robot_model, st)
            elif match.kind == "pose_finder":
                from .pose_layout import PoseSettings

                ev = PoseEvaluator(self.robot_model, PoseSettings(
                    terrain="smooth_steps" if match.smooth_terrain else "planar",
                    n_terrain_params=match.n_terrain_params))
            else:
                raise TemplateMismatch("toy OCP: construct ToyEvaluator with the problem's dt explicitly")
            host = HostEvaluator(ev)
            return ev.layout, host, host.masks

        def _match_template(self):
            opti = self._solver
            match = match_template(int(opti.nx), int(opti.np), int(opti.ng))
            if match is None:
                raise TemplateMismatch(f"no template with n_x={opti.nx}, n_p={opti.np}, m={opti.ng}")
            factory = evaluator_factory or self._default_factory
            return match, factory(match)

        def _fill_outputs(self, x, cost, lam_g):
            """The fields `solve()` populates (opti_solver.py:522-537).  Values of the named costs and the duals of
            the named constraints are evaluated with CasADi's own functions of (x, p) / lam_g -- once per solve --
            so that Opti's sign conventions for flipped inequalities apply unchanged [ext]."""
            opti = self._solver
            p = np.asarray(opti.debug.value(opti.p)).ravel()
            values = {}
            off = 0
            for var in self._variables_map:               # creation order = order inside opti.x [ext]
                n = int(var.numel())
                block = x[off:off + n]
                shape = tuple(var.shape) if hasattr(var, "shape") else (n, 1)
                # OptiSol.value() hands back numpy arrays squeezed like this [ext]: vectors 1-D, matrices 2-D
                values[var] = block.copy() if 1 in shape else block.reshape(shape, order="F")
                off += n
            for par in self._parameters_map:
                values[par] = np.asarray(opti.debug.value(par))
            self._output_cost = cost
            self._output_solution = self._generate_solution_output(variables=self._objects, input_solution=values)
            names = list(self._cost_expressions)
            if names:
                fun = cs.Function("hb_costs", [opti.x, opti.p], [self._cost_expressions[n] for n in names])
                vals = fun(x, p)
                vals = vals if isinstance(vals, (list, tuple)) else [vals]
                self._cost_values = {n: float(np.asarray(v).ravel()[0]) for n, v in zip(names, vals)}
            else:
                self._cost_values = {}
            cnames = list(self._constraint_expressions)
            if cnames:
                dfun = cs.Function("hb_duals", [opti.lam_g], [opti.dual(self._constraint_expressions[n]) for n in cnames])
                dv = dfun(lam_g)
                dv = dv if isinstance(dv, (list, tuple)) else [dv]
                self._constraint_values = {n: np.array(np.asarray(v).ravel()) for n, v in zip(cnames, dv)}
            else:
                self._constraint_values = {}

        def solve(self) -> None:
            self._cost = self._cost if self._cost is not None else cs.MX(0)
            opti = self._solver
            opti.minimize(self._cost)
            if len(self._free_parameters):
                raise ValueError("The following parameters are not set: " + str(self._free_parameters))
            try:
                match, (layout, host_eval, masks) = self._match_template()
                x0 = np.asarray(opti.debug.value(opti.x, opti.initial()), dtype=np.float64).ravel()
                p = np.asarray(opti.debug.value(opti.p), dtype=np.float64).ravel()
                lbg = np.asarray(opti.debug.value(opti.lbg), dtype=np.float64).ravel()
                ubg = np.asarray(opti.debug.value(opti.ubg), dtype=np.float64).ravel()
                if hasattr(host_eval, "set_parameters"):
                    host_eval.set_parameters(p)
                _, consumed = split_plugin_options(self._options_plugin)
                bridge = OracleBridge(cs, layout, host_eval, masks, bool(consumed.get("detect_simple_bounds", False)))
                fg = cs.Function("hb_probe", [opti.x, opti.p], [opti.f, opti.g])(x0, p)
                bridge.verify(x0, p, float(np.asarray(fg[0]).ravel()[0]), np.asarray(fg[1], dtype=np.float64).ravel())
            except TemplateMismatch as err:
                if self.strict:
                    raise
                LOG.warning("falling back to the stock OptiSolver.solve(): %s", err)
                return super().solve()
            type(self).last_bridge = self.last_bridge = bridge
            ev = getattr(host_eval, "ev", None)
            if self.oracle == "external" and ev is not None:
                from . import _capi

                bridge.build_external(self._options_plugin, self._options_solver, self._inner_solver, _capi.LIB_PATH, ev._h)
            else:
                bridge.build(self._options_plugin, self._options_solver, self._inner_solver)
            # the callback criterion needs Opti's iteration callback; the shim keeps IPOPT's own termination
            try:
                x, cost, lam_g, stats = bridge.run(x0, p, lbg, ubg)
            except Exception as err:  # noqa: BLE001 -- same catch-all as opti_solver.py:479-481
                raise hp.OptiFailure(message=err, callback_used=False)
            if not stats.get("success", False):
                raise hp.OptiFailure(message=Exception(str(stats.get("return_status", "failed"))), callback_used=False)
            self._fill_outputs(x, cost, lam_g)

    return B200OptiSolver


def install(robot_model, kino_settings, strict: bool = False):
    """Bind `hippopt.OptiSolver` to the B200 back end before a planner is constructed (both turnkey planners
    hard-code `hp.OptiSolver(...)`: humanoid_kinodynamic/planner.py:65-71, humanoid_pose_finder/planner.py:334-339)."""
    try:
        import casadi as cs
        import hippopt as hp
    except ImportError as err:  # the build container has neither: the shim is exercised with stand-ins in tests/
        raise ImportError("hippopt_b200.plugin.install needs the `casadi` and `hippopt` packages of the reference "
                          f"environment ({err}); B200Solver is the casadi-free entry point") from err
    cls = make_opti_solver(cs, hp)
    cls.robot_model, cls.kino_settings, cls.strict = robot_model, kino_settings, strict
    hp.OptiSolver = cls
    if hasattr(hp, "base") and hasattr(hp.base, "opti_solver"):
        hp.base.opti_solver.OptiSolver = cls
    return cls
