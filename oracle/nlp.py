"""oracle/nlp.py -- TEST INFRASTRUCTURE ONLY.

Container that plays the role CasADi ``Opti`` + ``nlpsol`` play for the reference
(`/root/reference/src/hippopt/base/opti_solver.py:113,123-125,446,479,563-572`): it records
``subject_to`` rows and ``minimize`` terms in call order, and exposes the five NLP oracle
functions IPOPT calls (f, grad_f, g, jac_g, hess_l) together with the structural CCS sparsity
patterns of jac_g and (upper-triangular) hess_l obtained by dependency propagation [ext: what
CasADi's ``Function.jacobian_sparsity`` does].

Rows/costs are recorded as *applications* of small expression templates (an SX graph over
template symbols plus an index array binding every template symbol to a slot of w = [x; p]),
which is only a compression of the flat graph the reference builds with ``cs.substitute``
(`base/multiple_shooting_solver.py:807-824`): values, derivatives and patterns are identical to
those of the flat graph.
"""
from __future__ import annotations

import numpy as np

from . import sx
from .sx import SX


class Template:
    """rows / bounds (or one cost expression) over ``inputs`` (template symbols)."""

    def __init__(self, name: str, inputs, rows, lb=None, ub=None):
        self.name = name
        self.inputs = list(inputs)
        self.rows = [sx._wrap(r) for r in rows]
        n = len(self.rows)
        self.lb = [sx._wrap(v) for v in (lb if lb is not None else [0.0] * n)]
        self.ub = [sx._wrap(v) for v in (ub if ub is not None else [0.0] * n)]
        assert len(self.lb) == n and len(self.ub) == n
        self._tape = None
        self._bound_tape = None
        self._pattern = None
        self._grad = None

    @property
    def tape(self) -> sx.Tape:
        if self._tape is None:
            self._tape = sx.Tape(self.rows, self.inputs)
        return self._tape

    @property
    def bound_tape(self) -> sx.Tape:
        if self._bound_tape is None:
            self._bound_tape = sx.Tape(self.lb + self.ub, self.inputs)
        return self._bound_tape

    @property
    def pattern(self):
        """rows[i] -> template input indices the row structurally depends on."""
        if self._pattern is None:
            self._pattern = sx.jac_pattern(self.rows, self.inputs)
        return self._pattern

    def lagrangian_gradient(self):
        """(lam symbols, gradient graphs of sum_r lam_r rows_r w.r.t. every template input)."""
        if self._grad is None:
            lam = [sx.sym(f"lam_{self.name}_{i}") for i in range(len(self.rows))]
            L = sx.const(0.0)
            for l, r in zip(lam, self.rows):
                L = L + l * r
            g = sx.gradient(L, self.inputs)
            tape = sx.Tape(g, self.inputs + lam)
            pat = sx.jac_pattern(g, self.inputs)
            self._grad = (lam, g, tape, pat)
        return self._grad


class NLP:
    def __init__(self, n_x: int, n_p: int):
        self.n_x, self.n_p = n_x, n_p
        self.m = 0
        self.row_apps: list[tuple[Template, np.ndarray, int]] = []
        self.cost_apps: list[tuple[Template, np.ndarray, float]] = []
        self.row_names: list[str] = []        # one per row: "<expression name>{i}"-style debugging labels
        self.constraint_names: list[tuple[str, int, int]] = []  # (reference expression name, first row, rows)
        self.cost_names: list[str] = []       # reference expression name of every cost application
        self._jac = None
        self._hess = None
        self._plans: dict = {}

    # -- recording ------------------------------------------------------------------
    def subject_to(self, template: Template, binding, name: str = "") -> int:
        binding = np.asarray(binding, dtype=np.int64)
        assert binding.shape == (len(template.inputs),)
        off = self.m
        self.row_apps.append((template, binding, off))
        self.m += len(template.rows)
        self.row_names.extend([f"{name}{{{i}}}" for i in range(len(template.rows))])
        self.constraint_names.append((name, off, len(template.rows)))
        return off

    def minimize(self, template: Template, binding, scaling: float = 1.0, name: str = "") -> None:
        binding = np.asarray(binding, dtype=np.int64)
        assert len(template.rows) == 1 and binding.shape == (len(template.inputs),)
        self.cost_apps.append((template, binding, float(scaling)))
        self.cost_names.append(name)

    # -- helpers ----------------------------------------------------------------------
    @staticmethod
    def _group(apps):
        groups: dict[int, list] = {}
        for app in apps:
            groups.setdefault(id(app[0]), []).append(app)
        return list(groups.values())

    def _w(self, X, P, dtype=np.float64):
        X = np.atleast_2d(np.asarray(X, dtype=dtype))
        P = np.atleast_2d(np.asarray(P, dtype=dtype))
        assert X.shape[1] == self.n_x and P.shape[1] == self.n_p
        if P.shape[0] == 1 and X.shape[0] > 1:
            P = np.repeat(P, X.shape[0], axis=0)
        return np.concatenate([X, P], axis=1)

    @staticmethod
    def _gather(W, apps):
        """(B, A, n_in) -> (B*A, n_in) inputs of all applications of one template."""
        idx = np.stack([a[1] for a in apps])  # (A, n_in)
        U = W[:, idx]  # (B, A, n_in)
        return U.reshape(-1, idx.shape[1]), idx

    # -- values ---------------------------------------------------------------------
    # Every eval_* takes ``dtype``, the floating type of the whole evaluation (Tape.eval): np.longdouble gives an
    # extended-precision reference, finite where the float64 tapes form 0 * inf far from a smooth step.
    def eval_g(self, X, P, dtype=np.float64):
        W = self._w(X, P, dtype)
        B = W.shape[0]
        out = np.zeros((B, self.m), dtype=dtype)
        for apps in self._group(self.row_apps):
            t = apps[0][0]
            U, idx = self._gather(W, apps)
            vals = t.tape.eval(U, dtype).reshape(B, len(apps), -1)
            for a, (_, _, off) in enumerate(apps):
                out[:, off:off + vals.shape[2]] = vals[:, a, :]
        return out

    def eval_bounds(self, P, dtype=np.float64):
        P = np.atleast_2d(np.asarray(P, dtype=dtype))
        W = np.concatenate([np.zeros((P.shape[0], self.n_x), dtype=dtype), P], axis=1)
        B = W.shape[0]
        lb = np.zeros((B, self.m), dtype=dtype)
        ub = np.zeros((B, self.m), dtype=dtype)
        for apps in self._group(self.row_apps):
            t = apps[0][0]
            n = len(t.rows)
            U, idx = self._gather(W, apps)
            vals = t.bound_tape.eval(U, dtype).reshape(B, len(apps), -1)
            for a, (_, _, off) in enumerate(apps):
                lb[:, off:off + n] = vals[:, a, :n]
                ub[:, off:off + n] = vals[:, a, n:]
        return lb, ub

    def eval_f(self, X, P, dtype=np.float64):
        W = self._w(X, P, dtype)
        B = W.shape[0]
        f = np.zeros(B, dtype=dtype)
        # accumulate in recording order, like ``self._cost += input_cost`` (opti_solver.py:556-559)
        cache = {}
        for apps in self._group(self.cost_apps):
            U, _ = self._gather(W, apps)
            vals = apps[0][0].tape.eval(U, dtype).reshape(B, len(apps))
            for a, app in enumerate(apps):
                cache[id(app)] = vals[:, a]
        for app in self.cost_apps:
            f = f + app[2] * cache[id(app)]
        return f

    def eval_cost_terms(self, X, P, dtype=np.float64):
        W = self._w(X, P, dtype)
        B = W.shape[0]
        out = np.zeros((B, len(self.cost_apps)), dtype=dtype)
        pos = {id(app): i for i, app in enumerate(self.cost_apps)}
        for apps in self._group(self.cost_apps):
            U, _ = self._gather(W, apps)
            vals = apps[0][0].tape.eval(U, dtype).reshape(B, len(apps))
            for a, app in enumerate(apps):
                out[:, pos[id(app)]] = app[2] * vals[:, a]
        return out

    def eval_grad_f(self, X, P, dtype=np.float64):
        W = self._w(X, P, dtype)
        B = W.shape[0]
        grad = np.zeros((B, self.n_x), dtype=dtype)
        for apps in self._group(self.cost_apps):
            t = apps[0][0]
            U, idx = self._gather(W, apps)
            xin = [i for i in range(len(t.inputs)) if np.all(idx[:, i] < self.n_x)]
            pat = set(t.pattern[0])
            xin = [i for i in xin if i in pat]
            if not xin:
                continue
            _, tang = t.tape.eval_fwd(U, xin, dtype)
            tang = tang.reshape(B, len(apps), len(xin))
            for a, (_, binding, scale) in enumerate(apps):
                np.add.at(grad, (slice(None), binding[xin]), scale * tang[:, a, :])
        return grad

    # -- Jacobian ---------------------------------------------------------------------
    def jac_structure(self):
        """CCS (colind, row) of jac_g plus, per application, the slot of every local entry."""
        if self._jac is not None:
            return self._jac
        rows, cols = [], []
        for (t, binding, off) in self.row_apps:
            for r, deps in enumerate(t.pattern):
                for i in deps:
                    c = int(binding[i])
                    if c < self.n_x:
                        rows.append(off + r)
                        cols.append(c)
        rows = np.asarray(rows, dtype=np.int64)
        cols = np.asarray(cols, dtype=np.int64)
        key = cols * self.m + rows
        uniq = np.unique(key)
        assert len(uniq) == len(key), "duplicate Jacobian entries"
        order = np.argsort(key, kind="stable")
        colind = np.zeros(self.n_x + 1, dtype=np.int64)
        np.add.at(colind, cols + 1, 1)
        colind = np.cumsum(colind)
        self._jac = (colind, rows[order], cols[order], uniq)
        return self._jac

    def eval_jac(self, X, P, dtype=np.float64):
        colind, row, col, keys = self.jac_structure()
        W = self._w(X, P, dtype)
        B = W.shape[0]
        vals = np.zeros((B, len(row)), dtype=dtype)
        for apps in self._group(self.row_apps):
            t = apps[0][0]
            U, idx = self._gather(W, apps)
            xin = sorted({i for deps in t.pattern for i in deps if np.all(idx[:, i] < self.n_x)})
            if not xin:
                continue
            _, tang = t.tape.eval_fwd(U, xin, dtype)
            tang = tang.reshape(B, len(apps), len(t.rows), len(xin))
            plan = self._plans.get(("jac", id(t)))
            if plan is None:  # scatter plan (application, row, direction) -> CCS slot, built once
                pos = {i: d for d, i in enumerate(xin)}
                A, R, D, S = [], [], [], []
                for a, (_, binding, off) in enumerate(apps):
                    for r, deps in enumerate(t.pattern):
                        for i in deps:
                            c = int(binding[i])
                            if c < self.n_x:
                                A.append(a)
                                R.append(r)
                                D.append(pos[i])
                                S.append(c * self.m + off + r)
                plan = (np.array(A), np.array(R), np.array(D), np.searchsorted(keys, np.array(S, dtype=np.int64)))
                self._plans[("jac", id(t))] = plan
            A, R, D, S = plan
            vals[:, S] = tang[:, A, R, D]
        return vals

    # -- Hessian of the Lagrangian ---------------------------------------------------------
    def hess_structure(self):
        if self._hess is not None:
            return self._hess
        ent = set()
        for (t, binding, _) in list(self.row_apps) + [(c[0], c[1], 0) for c in self.cost_apps]:
            _, _, _, pat = t.lagrangian_gradient()
            for i, deps in enumerate(pat):
                ci = int(binding[i])
                if ci >= self.n_x:
                    continue
                for j in deps:
                    cj = int(binding[j])
                    if cj >= self.n_x:
                        continue
                    r, c = (ci, cj) if ci <= cj else (cj, ci)
                    ent.add(c * self.n_x + r)
        keys = np.array(sorted(ent), dtype=np.int64)
        col = keys // self.n_x
        row = keys % self.n_x
        colind = np.zeros(self.n_x + 1, dtype=np.int64)
        np.add.at(colind, col + 1, 1)
        colind = np.cumsum(colind)
        self._hess = (colind, row, col, keys)
        return self._hess

    def eval_hess(self, X, P, lam, sigma=1.0, dtype=np.float64):
        colind, row, col, keys = self.hess_structure()
        W = self._w(X, P, dtype)
        B = W.shape[0]
        lam = np.atleast_2d(np.asarray(lam, dtype=dtype))
        sigma = np.broadcast_to(np.asarray(sigma, dtype=dtype), (B,))
        vals = np.zeros((B, len(keys)), dtype=dtype)

        def run(apps, lam_of_app):
            t = apps[0][0]
            lam_syms, g, tape, pat = t.lagrangian_gradient()
            U, idx = self._gather(W, apps)
            xin = sorted({j for deps in pat for j in deps if np.all(idx[:, j] < self.n_x)})
            if not xin:
                return
            L = np.stack([lam_of_app(app) for app in apps], axis=1).reshape(B * len(apps), -1)
            _, tang = tape.eval_fwd(np.concatenate([U, L], axis=1), xin, dtype)
            tang = tang.reshape(B, len(apps), len(t.inputs), len(xin))
            plan = self._plans.get(("hess", id(t)))
            if plan is None:
                pos = {j: d for d, j in enumerate(xin)}
                A, I, D, S = [], [], [], []
                for a, app in enumerate(apps):
                    binding = app[1]
                    for i, deps in enumerate(pat):
                        ci = int(binding[i])
                        if ci >= self.n_x:
                            continue
                        for j in deps:
                            cj = int(binding[j])
                            if cj >= self.n_x or ci > cj:
                                continue  # lower triangle is the mirror image
                            if ci == cj and i != j:
                                raise AssertionError("two template inputs bound to one variable")
                            A.append(a)
                            I.append(i)
                            D.append(pos[j])
                            S.append(cj * self.n_x + ci)
                plan = (np.array(A), np.array(I), np.array(D), np.searchsorted(keys, np.array(S, dtype=np.int64)))
                self._plans[("hess", id(t))] = plan
            A, I, D, S = plan
            if len(S):
                np.add.at(vals, (slice(None), S), tang[:, A, I, D])

        for apps in self._group(self.row_apps):
            n = len(apps[0][0].rows)
            run(apps, lambda app: lam[:, app[2]:app[2] + n])
        for apps in self._group(self.cost_apps):
            run(apps, lambda app: (sigma * app[2])[:, None])
        return vals

    # -- dense helpers for tests -----------------------------------------------------------
    def dense_jac(self, X, P, dtype=np.float64):
        colind, row, col, _ = self.jac_structure()
        v = self.eval_jac(X, P, dtype)
        out = np.zeros((v.shape[0], self.m, self.n_x), dtype=dtype)
        out[:, row, col] = v
        return out

    def dense_hess(self, X, P, lam, sigma=1.0, dtype=np.float64):
        colind, row, col, _ = self.hess_structure()
        v = self.eval_hess(X, P, lam, sigma, dtype)
        out = np.zeros((v.shape[0], self.n_x, self.n_x), dtype=dtype)
        out[:, row, col] = v
        out[:, col, row] = v
        return out
