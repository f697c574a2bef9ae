"""oracle/cvm.py -- TEST / MEASUREMENT INFRASTRUCTURE ONLY.

Compiles the tapes of oracle/sx.py for the C virtual machine oracle/sxvm.c (work-vector slot allocation
by liveness, "has a tangent" flags by dependency propagation) and runs them batched with OpenMP.
`enable()` routes `sx.Tape.eval` / `eval_fwd` through the C VM; results are identical to the numpy
interpreter up to the last bit of libm's transcendental functions.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

from . import sx

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "_build", "libsxvm.so")
_lib = None
N_THREADS = 0  # 0: OpenMP default (all cores)


def available() -> bool:
    return os.path.exists(LIB)


def lib():
    global _lib
    if _lib is None:
        L = ctypes.CDLL(LIB)
        ip, dp, up = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_ubyte)
        L.sxvm_run.restype = ctypes.c_int
        L.sxvm_run.argtypes = [ctypes.c_int, ip, ip, ip, ip, dp, up, ctypes.c_int, ip, ctypes.c_int, ip, up,
                               ctypes.c_int, ctypes.c_int, ctypes.c_int, dp, dp, dp, ctypes.c_int]
        L.sxvm_max_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def max_threads() -> int:
    return int(lib().sxvm_max_threads())


class _Program:
    def __init__(self, tape: sx.Tape, seed_idx):
        order = tape.order
        n = len(order)
        seeds = {int(i): d for d, i in enumerate(seed_idx)}
        self.D = len(seeds)
        pos = {node.id: k for k, node in enumerate(order)}
        op = np.zeros(n, dtype=np.int32)
        a = -np.ones(n, dtype=np.int32)
        b = -np.ones(n, dtype=np.int32)
        dst = np.zeros(n, dtype=np.int32)
        cval = np.zeros(n)
        has = np.zeros(n, dtype=np.uint8)
        node_t = np.zeros(n, dtype=bool)
        slot_of = {}
        free = []
        n_slots = 0
        keep = {o.id for o in tape.outputs}
        in_seed = -np.ones(len(tape.inputs), dtype=np.int32)
        for i, d in seeds.items():
            in_seed[i] = d
        for k, node in enumerate(order):
            op[k] = node.op
            if node.op == sx.OP_CONST:
                cval[k] = node.val
            elif node.op == sx.OP_SYM:
                j = tape.in_index[node.id]
                a[k] = j
                node_t[k] = j in seeds
                has[k] = 1 if node_t[k] else 0
            else:
                ka = pos[node.a.id]
                a[k] = slot_of[node.a.id]
                ta = node_t[ka]
                tb = False
                if node.b is not None:
                    if node.op == sx.OP_POWC:
                        cval[k] = node.b.val
                    else:
                        kb = pos[node.b.id]
                        b[k] = slot_of[node.b.id]
                        tb = node_t[kb]
                node_t[k] = ta or tb
                has[k] = (1 if node_t[k] else 0) | (2 if ta else 0) | (4 if tb else 0)
            if free:
                s = free.pop()
            else:
                s = n_slots
                n_slots += 1
            slot_of[node.id] = s
            dst[k] = s
            for nid in tape.free_after[k]:
                if nid not in keep:
                    free.append(slot_of[nid])
        self.n = n
        self.n_slots = n_slots
        self.arrays = (op, dst, a, b, cval, has)
        self.in_seed = in_seed
        self.out_slot = np.array([slot_of[o.id] for o in tape.outputs], dtype=np.int32)
        self.out_has = np.array([1 if node_t[pos[o.id]] else 0 for o in tape.outputs], dtype=np.uint8)
        self.n_in, self.n_out = len(tape.inputs), len(tape.outputs)

    def run(self, X):
        X = np.ascontiguousarray(np.atleast_2d(X), dtype=np.float64)
        B = X.shape[0]
        vals = np.empty((B, self.n_out))
        tang = np.empty((B, self.n_out, self.D)) if self.D else None
        ip, dp, up = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_ubyte)
        op, dst, a, b, cval, has = self.arrays
        rc = lib().sxvm_run(
            self.n, op.ctypes.data_as(ip), dst.ctypes.data_as(ip), a.ctypes.data_as(ip), b.ctypes.data_as(ip),
            cval.ctypes.data_as(dp), has.ctypes.data_as(up), self.n_in, self.in_seed.ctypes.data_as(ip), self.n_out,
            self.out_slot.ctypes.data_as(ip), self.out_has.ctypes.data_as(up), self.n_slots, self.D, B,
            X.ctypes.data_as(dp), vals.ctypes.data_as(dp), tang.ctypes.data_as(dp) if tang is not None else None,
            N_THREADS)
        if rc:
            raise MemoryError("sxvm_run: allocation failed")
        return vals, tang


def _program(tape: sx.Tape, seed_idx):
    cache = tape.__dict__.setdefault("_cvm", {})
    key = tuple(int(i) for i in seed_idx)
    prog = cache.get(key)
    if prog is None:
        prog = cache[key] = _Program(tape, key)
    return prog


_numpy_eval, _numpy_eval_fwd = sx.Tape.eval, sx.Tape.eval_fwd


def _c_eval(self, X, dtype=np.float64):
    if np.dtype(dtype) != np.float64:  # the C VM computes in double only
        return _numpy_eval(self, X, dtype)
    return _program(self, ()).run(X)[0]


def _c_eval_fwd(self, X, seed_idx, dtype=np.float64):
    if np.dtype(dtype) != np.float64:
        return _numpy_eval_fwd(self, X, seed_idx, dtype)
    vals, tang = _program(self, seed_idx).run(X)
    return vals, tang


def enable(n_threads: int = 0) -> None:
    """Route every tape evaluation through the C VM (raises if it has not been built)."""
    global N_THREADS
    if not available():
        raise RuntimeError(f"{LIB} missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    N_THREADS = n_threads
    sx.Tape.eval = _c_eval
    sx.Tape.eval_fwd = _c_eval_fwd


def disable() -> None:
    sx.Tape.eval = _numpy_eval
    sx.Tape.eval_fwd = _numpy_eval_fwd
