"""oracle/sx.py -- TEST INFRASTRUCTURE ONLY (the checker, never the product path).

A small scalar expression-graph engine that restates, on the CPU, how the reference's
numerical hot path is actually produced: hippopt only *builds* CasADi graphs
(`/root/reference/src/hippopt/base/opti_solver.py:113,479`); every f / g / Jacobian /
Hessian number IPOPT sees is computed by CasADi's SX machinery [ext: casadi is not
vendored under /root/reference and is not installed here; un-pinned in
`/root/reference/setup.cfg:52-78`].  The published algorithm restated here is:

  * scalar expression nodes with construction-time simplification
    (0*x -> 0, 1*x -> x, x+0 -> x, x-x -> 0 ...) and hash-consing (what the reference
    asks for with ``casadi_function_options = {"cse": True}``,
    `main_single_step_flat_ground.py:105`);
  * reverse-mode AD as a graph transformation (``cs.gradient`` / ``nlp_grad_f`` /
    the gradient of the Lagrangian behind ``nlp_hess_l``);
  * structural sparsity by dependency propagation (bit-vectors), which is what fixes
    the ``jac_g`` / ``hess_l`` ``Sparsity`` patterns the evaluator must reproduce;
  * evaluation of the instruction tape (the "SX virtual machine"), plus forward-mode
    directional sweeps over a tape for Jacobian / Hessian values.

parity status: UNPINNED against CasADi itself (no casadi in this container); pinned
against the reference's own known-answer tests where they exist (see tests/).
"""
from __future__ import annotations

import math
from typing import Iterable, Sequence

import numpy as np

(
    OP_CONST,
    OP_SYM,
    OP_ADD,
    OP_SUB,
    OP_MUL,
    OP_DIV,
    OP_NEG,
    OP_SQ,
    OP_SQRT,
    OP_SIN,
    OP_COS,
    OP_TANH,
    OP_EXP,
    OP_POWC,
    OP_FABS,
) = range(15)

OP_NAMES = [
    "const", "sym", "add", "sub", "mul", "div", "neg", "sq", "sqrt", "sin", "cos",
    "tanh", "exp", "powc", "fabs",
]
BINARY = {OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_POWC}


class _Graph:
    def __init__(self) -> None:
        self.nodes = 0
        self.consts: dict = {}
        self.cache: dict = {}


_G = _Graph()


def reset() -> None:
    """Drop the hash-consing tables (existing nodes stay valid)."""
    global _G
    _G = _Graph()


class SX:
    __slots__ = ("op", "a", "b", "val", "name", "id")
    __array_priority__ = 1000  # numpy object arrays defer to our operators

    def __init__(self, op, a=None, b=None, val=0.0, name=None):
        self.op = op
        self.a = a
        self.b = b
        self.val = val
        self.name = name
        self.id = _G.nodes
        _G.nodes += 1

    # -- predicates -------------------------------------------------------------
    def is_const(self) -> bool:
        return self.op == OP_CONST

    def is_zero(self) -> bool:
        return self.op == OP_CONST and self.val == 0.0

    def is_one(self) -> bool:
        return self.op == OP_CONST and self.val == 1.0

    def is_minus_one(self) -> bool:
        return self.op == OP_CONST and self.val == -1.0

    # -- operators ---------------------------------------------------------------
    def __add__(self, o):
        return add(self, _wrap(o))

    def __radd__(self, o):
        return add(_wrap(o), self)

    def __sub__(self, o):
        return sub(self, _wrap(o))

    def __rsub__(self, o):
        return sub(_wrap(o), self)

    def __mul__(self, o):
        return mul(self, _wrap(o))

    def __rmul__(self, o):
        return mul(_wrap(o), self)

    def __truediv__(self, o):
        return div(self, _wrap(o))

    def __rtruediv__(self, o):
        return div(_wrap(o), self)

    def __neg__(self):
        return neg(self)

    def __pos__(self):
        return self

    def __pow__(self, e):
        return powc(self, e)

    def __repr__(self):
        if self.op == OP_CONST:
            return f"{self.val!r}"
        if self.op == OP_SYM:
            return self.name
        return f"<{OP_NAMES[self.op]}#{self.id}>"

    def __float__(self):
        if self.op != OP_CONST:
            raise TypeError("symbolic SX has no float value")
        return self.val


def const(v: float) -> SX:
    v = float(v)
    key = (v, math.copysign(1.0, v)) if v == 0.0 else v
    n = _G.consts.get(key)
    if n is None:
        n = SX(OP_CONST, val=v)
        _G.consts[key] = n
    return n


def sym(name: str) -> SX:
    return SX(OP_SYM, name=name)


def syms(name: str, n: int) -> np.ndarray:
    out = np.empty(n, dtype=object)
    for i in range(n):
        out[i] = sym(f"{name}_{i}")
    return out


def _wrap(o) -> SX:
    if isinstance(o, SX):
        return o
    return const(float(o))


def _node(op, a, b=None) -> SX:
    key = (op, a.id, b.id if b is not None else -1)
    n = _G.cache.get(key)
    if n is None:
        n = SX(op, a, b)
        _G.cache[key] = n
    return n


def add(a: SX, b: SX) -> SX:
    if a.op == OP_CONST and b.op == OP_CONST:
        return const(a.val + b.val)
    if a.is_zero():
        return b
    if b.is_zero():
        return a
    if b.op == OP_NEG:
        return sub(a, b.a)
    if a.op == OP_NEG:
        return sub(b, a.a)
    return _node(OP_ADD, a, b)


def sub(a: SX, b: SX) -> SX:
    if a.op == OP_CONST and b.op == OP_CONST:
        return const(a.val - b.val)
    if b.is_zero():
        return a
    if a.is_zero():
        return neg(b)
    if a is b:
        return const(0.0)
    if b.op == OP_NEG:
        return add(a, b.a)
    return _node(OP_SUB, a, b)


def mul(a: SX, b: SX) -> SX:
    if a.op == OP_CONST and b.op == OP_CONST:
        return const(a.val * b.val)
    if a.is_zero() or b.is_zero():
        return const(0.0)
    if a.is_one():
        return b
    if b.is_one():
        return a
    if a.is_minus_one():
        return neg(b)
    if b.is_minus_one():
        return neg(a)
    if a is b:
        return sq(a)
    return _node(OP_MUL, a, b)


def div(a: SX, b: SX) -> SX:
    if a.op == OP_CONST and b.op == OP_CONST:
        return const(a.val / b.val)
    if a.is_zero():
        return const(0.0)
    if b.is_one():
        return a
    if b.is_minus_one():
        return neg(a)
    return _node(OP_DIV, a, b)


def neg(a: SX) -> SX:
    if a.op == OP_CONST:
        return const(-a.val)
    if a.op == OP_NEG:
        return a.a
    return _node(OP_NEG, a)


def sq(a) -> SX:
    a = _wrap(a)
    if a.op == OP_CONST:
        return const(a.val * a.val)
    if a.op == OP_NEG:
        return sq(a.a)
    return _node(OP_SQ, a)


def _unary(op, fn, a) -> SX:
    a = _wrap(a)
    if a.op == OP_CONST:
        return const(fn(a.val))
    return _node(op, a)


def sqrt(a) -> SX:
    return _unary(OP_SQRT, math.sqrt, a)


def sin(a) -> SX:
    return _unary(OP_SIN, math.sin, a)


def cos(a) -> SX:
    return _unary(OP_COS, math.cos, a)


def tanh(a) -> SX:
    return _unary(OP_TANH, math.tanh, a)


def exp(a) -> SX:
    return _unary(OP_EXP, math.exp, a)


def fabs(a) -> SX:
    return _unary(OP_FABS, abs, a)


def powc(a, e: float) -> SX:
    """a ** e with a *constant* float exponent (``cs.constpow`` / ``x**20.0``)."""
    a = _wrap(a)
    e = float(e)
    if e == 1.0:
        return a
    if e == 2.0:
        return sq(a)
    if e == 0.0:
        return const(1.0)
    if a.op == OP_CONST:
        return const(math.pow(a.val, e))
    return _node(OP_POWC, a, const(e))


# ---------------------------------------------------------------------------------
# graph utilities
# ---------------------------------------------------------------------------------
def topo(outputs: Iterable[SX]) -> list[SX]:
    """Children-first ordering of every node reachable from ``outputs`` (iterative DFS)."""
    order: list[SX] = []
    seen: set[int] = set()
    for root in outputs:
        if root.id in seen:
            continue
        stack = [(root, 0)]
        while stack:
            node, state = stack.pop()
            if state == 0:
                if node.id in seen:
                    continue
                seen.add(node.id)
                stack.append((node, 1))
                if node.b is not None and node.b.id not in seen:
                    stack.append((node.b, 0))
                if node.a is not None and node.a.id not in seen:
                    stack.append((node.a, 0))
            else:
                order.append(node)
    return order


def gradient(out: SX, wrt: Sequence[SX], seed: SX | None = None) -> list[SX]:
    """Reverse-mode AD as a source transformation: d out / d wrt[i] as new SX graphs."""
    order = topo([out])
    adj: dict[int, SX] = {out.id: seed if seed is not None else const(1.0)}
    for node in reversed(order):
        bar = adj.get(node.id)
        if bar is None or node.op in (OP_CONST, OP_SYM):
            continue
        if bar.is_zero():
            continue
        op, a, b = node.op, node.a, node.b

        def push(child: SX, contrib: SX) -> None:
            if child.op == OP_CONST or contrib.is_zero():
                return
            prev = adj.get(child.id)
            adj[child.id] = contrib if prev is None else add(prev, contrib)

        if op == OP_ADD:
            push(a, bar)
            push(b, bar)
        elif op == OP_SUB:
            push(a, bar)
            push(b, neg(bar))
        elif op == OP_MUL:
            push(a, mul(bar, b))
            push(b, mul(bar, a))
        elif op == OP_DIV:
            # d(a/b) = da/b - (a/b) db / b
            push(a, div(bar, b))
            push(b, neg(mul(bar, div(node, b))))
        elif op == OP_NEG:
            push(a, neg(bar))
        elif op == OP_SQ:
            push(a, mul(bar, mul(const(2.0), a)))
        elif op == OP_SQRT:
            push(a, div(bar, mul(const(2.0), node)))
        elif op == OP_SIN:
            push(a, mul(bar, cos(a)))
        elif op == OP_COS:
            push(a, neg(mul(bar, sin(a))))
        elif op == OP_TANH:
            push(a, mul(bar, sub(const(1.0), sq(node))))
        elif op == OP_EXP:
            push(a, mul(bar, node))
        elif op == OP_POWC:
            e = b.val
            push(a, mul(bar, mul(const(e), powc(a, e - 1.0))))
        elif op == OP_FABS:
            raise NotImplementedError("fabs is not differentiated by the oracle")
        else:  # pragma: no cover
            raise AssertionError(op)
    zero = const(0.0)
    return [adj.get(s.id, zero) for s in wrt]


def dependency_bits(outputs: Sequence[SX], inputs: Sequence[SX]) -> list[int]:
    """For each output, a bitmask over ``inputs`` it structurally depends on."""
    index = {s.id: i for i, s in enumerate(inputs)}
    bits: dict[int, int] = {}
    for node in topo(outputs):
        if node.op == OP_SYM:
            i = index.get(node.id)
            bits[node.id] = (1 << i) if i is not None else 0
        elif node.op == OP_CONST:
            bits[node.id] = 0
        else:
            m = bits[node.a.id]
            if node.b is not None:
                m |= bits[node.b.id]
            bits[node.id] = m
    return [bits[o.id] for o in outputs]


def jac_pattern(outputs: Sequence[SX], inputs: Sequence[SX]) -> list[list[int]]:
    """rows[i] = sorted input indices output i depends on (structural Jacobian pattern)."""
    out = []
    for m in dependency_bits(outputs, inputs):
        cols = []
        i = 0
        while m:
            if m & 1:
                cols.append(i)
            m >>= 1
            i += 1
        out.append(cols)
    return out


def count_ops(outputs: Sequence[SX]) -> int:
    """Number of non-trivial instructions on the tape (CasADi's n_instructions minus I/O)."""
    return sum(1 for n in topo(outputs) if n.op not in (OP_CONST, OP_SYM))


# ---------------------------------------------------------------------------------
# the "virtual machine": evaluate a tape with numpy, batched over instances
# ---------------------------------------------------------------------------------
class Tape:
    """Instruction tape for ``outputs`` as functions of ``inputs`` (other syms are errors)."""

    def __init__(self, outputs: Sequence[SX], inputs: Sequence[SX]):
        self.outputs = list(outputs)
        self.inputs = list(inputs)
        self.order = topo(self.outputs)
        self.in_index = {s.id: i for i, s in enumerate(self.inputs)}
        for n in self.order:
            if n.op == OP_SYM and n.id not in self.in_index:
                raise ValueError(f"free symbol {n.name} is not an input of the tape")
        # liveness: index of the last instruction using each node
        last: dict[int, int] = {}
        for k, n in enumerate(self.order):
            if n.a is not None:
                last[n.a.id] = k
            if n.b is not None:
                last[n.b.id] = k
        keep = {o.id for o in self.outputs}
        self.free_after: list[list[int]] = [[] for _ in self.order]
        for nid, k in last.items():
            if nid not in keep:
                self.free_after[k].append(nid)
        self.n_ops = sum(1 for n in self.order if n.op not in (OP_CONST, OP_SYM))

    # values only ------------------------------------------------------------------
    # ``dtype`` is the floating type of the whole evaluation (inputs, every intermediate, tangents and outputs);
    # np.longdouble runs the same tape with a 64-bit mantissa where the platform has one.  The tape's constants
    # stay the float64 numbers the graph was built with.
    def eval(self, X: np.ndarray, dtype=np.float64) -> np.ndarray:
        X = np.atleast_2d(np.asarray(X, dtype=dtype))
        B = X.shape[0]
        w: dict[int, np.ndarray | float] = {}
        for k, n in enumerate(self.order):
            w[n.id] = _apply(n, w, X, self.in_index)
            for nid in self.free_after[k]:
                w.pop(nid, None)
        out = np.empty((B, len(self.outputs)), dtype=dtype)
        for j, o in enumerate(self.outputs):
            out[:, j] = w[o.id]
        return out

    # values + forward-mode tangents along the unit directions of inputs[seed_idx] ---
    def eval_fwd(self, X: np.ndarray, seed_idx: Sequence[int], dtype=np.float64):
        X = np.atleast_2d(np.asarray(X, dtype=dtype))
        B = X.shape[0]
        D = len(seed_idx)
        seed_pos = {int(i): d for d, i in enumerate(seed_idx)}
        w: dict[int, np.ndarray | float] = {}
        t: dict[int, np.ndarray | None] = {}
        for k, n in enumerate(self.order):
            v = _apply(n, w, X, self.in_index)
            w[n.id] = v
            op = n.op
            if op == OP_CONST:
                t[n.id] = None
            elif op == OP_SYM:
                d = seed_pos.get(self.in_index[n.id])
                if d is None:
                    t[n.id] = None
                else:
                    tt = np.zeros((B, D), dtype=dtype)
                    tt[:, d] = 1.0
                    t[n.id] = tt
            else:
                ta = t[n.a.id]
                tb = t[n.b.id] if n.b is not None else None
                t[n.id] = _tangent(n, v, w, ta, tb)
            for nid in self.free_after[k]:
                w.pop(nid, None)
                t.pop(nid, None)
        vals = np.empty((B, len(self.outputs)), dtype=dtype)
        tang = np.zeros((B, len(self.outputs), D), dtype=dtype)
        for j, o in enumerate(self.outputs):
            vals[:, j] = w[o.id]
            if t[o.id] is not None:
                tang[:, j, :] = t[o.id]
        return vals, tang


def _col(v):
    return v[:, None] if isinstance(v, np.ndarray) else v


def _apply(n: SX, w, X, in_index):
    op = n.op
    if op == OP_CONST:
        return n.val
    if op == OP_SYM:
        return X[:, in_index[n.id]]
    a = w[n.a.id]
    if op == OP_ADD:
        return a + w[n.b.id]
    if op == OP_SUB:
        return a - w[n.b.id]
    if op == OP_MUL:
        return a * w[n.b.id]
    if op == OP_DIV:
        return a / w[n.b.id]
    if op == OP_NEG:
        return -a
    if op == OP_SQ:
        return a * a
    if op == OP_SQRT:
        return np.sqrt(a)
    if op == OP_SIN:
        return np.sin(a)
    if op == OP_COS:
        return np.cos(a)
    if op == OP_TANH:
        return np.tanh(a)
    if op == OP_EXP:
        return np.exp(a)
    if op == OP_POWC:
        return np.power(a, n.b.val)
    if op == OP_FABS:
        return np.abs(a)
    raise AssertionError(op)


def _tangent(n: SX, v, w, ta, tb):
    op = n.op
    if ta is None and tb is None:
        return None
    a = w[n.a.id]
    if op == OP_ADD:
        if ta is None:
            return tb
        if tb is None:
            return ta
        return ta + tb
    if op == OP_SUB:
        if ta is None:
            return -tb
        if tb is None:
            return ta
        return ta - tb
    if op == OP_MUL:
        b = w[n.b.id]
        if ta is None:
            return _col(a) * tb
        if tb is None:
            return ta * _col(b)
        return ta * _col(b) + _col(a) * tb
    if op == OP_DIV:
        b = w[n.b.id]
        r = None
        if ta is not None:
            r = ta / _col(b)
        if tb is not None:
            s = -(_col(v) / _col(b)) * tb
            r = s if r is None else r + s
        return r
    if op == OP_NEG:
        return -ta
    if op == OP_SQ:
        return _col(2.0 * a) * ta
    if op == OP_SQRT:
        return ta / _col(2.0 * v)
    if op == OP_SIN:
        return _col(np.cos(a)) * ta
    if op == OP_COS:
        return _col(-np.sin(a)) * ta
    if op == OP_TANH:
        return _col(1.0 - v * v) * ta
    if op == OP_EXP:
        return _col(v) * ta
    if op == OP_POWC:
        e = n.b.val
        return _col(e * np.power(a, e - 1.0)) * ta
    raise AssertionError(op)


# ---------------------------------------------------------------------------------
# small dense linear-algebra helpers that work on floats, numpy arrays *and* SX
# (object arrays); explicit loops keep the operation order deterministic.
# ---------------------------------------------------------------------------------
def zeros(*shape) -> np.ndarray:
    out = np.empty(shape, dtype=object)
    z = const(0.0)
    for idx in np.ndindex(*shape):
        out[idx] = z
    return out


def eye(n: int) -> np.ndarray:
    out = zeros(n, n)
    for i in range(n):
        out[i, i] = const(1.0)
    return out


def lift(a) -> np.ndarray:
    """numeric array -> object array of SX constants (so 0/1 entries are *structural*)."""
    a = np.asarray(a, dtype=np.float64)
    out = np.empty(a.shape, dtype=object)
    for idx in np.ndindex(*a.shape):
        out[idx] = const(a[idx])
    return out


def matmul(A, B):
    A = np.asarray(A, dtype=object)
    B = np.asarray(B, dtype=object)
    vec = B.ndim == 1
    if vec:
        B = B[:, None]
    n, k = A.shape
    k2, m = B.shape
    assert k == k2
    out = np.empty((n, m), dtype=object)
    for i in range(n):
        for j in range(m):
            acc = _wrap(0.0)
            for l in range(k):
                acc = acc + _wrap(A[i, l]) * _wrap(B[l, j])
            out[i, j] = acc
    return out[:, 0] if vec else out


def cross(a, b):
    out = np.empty(3, dtype=object)
    out[0] = _wrap(a[1]) * _wrap(b[2]) - _wrap(a[2]) * _wrap(b[1])
    out[1] = _wrap(a[2]) * _wrap(b[0]) - _wrap(a[0]) * _wrap(b[2])
    out[2] = _wrap(a[0]) * _wrap(b[1]) - _wrap(a[1]) * _wrap(b[0])
    return out


def dot(a, b):
    acc = _wrap(0.0)
    for x, y in zip(a, b):
        acc = acc + _wrap(x) * _wrap(y)
    return acc


def sumsqr(a):
    acc = _wrap(0.0)
    for x in np.asarray(a, dtype=object).ravel():
        acc = acc + sq(_wrap(x))
    return acc


def norm2(a):
    return sqrt(sumsqr(a))


def skew(v):
    z = const(0.0)
    out = np.empty((3, 3), dtype=object)
    out[0, 0], out[0, 1], out[0, 2] = z, -_wrap(v[2]), _wrap(v[1])
    out[1, 0], out[1, 1], out[1, 2] = _wrap(v[2]), z, -_wrap(v[0])
    out[2, 0], out[2, 1], out[2, 2] = -_wrap(v[1]), _wrap(v[0]), z
    return out


def vec(*items) -> np.ndarray:
    flat = []
    for it in items:
        if isinstance(it, np.ndarray):
            flat.extend(it.ravel().tolist())
        elif isinstance(it, (list, tuple)):
            flat.extend(it)
        else:
            flat.append(it)
    out = np.empty(len(flat), dtype=object)
    for i, x in enumerate(flat):
        out[i] = _wrap(x)
    return out
