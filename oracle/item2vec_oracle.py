"""ctypes binding of oracle/item2vec_oracle.c (TEST INFRASTRUCTURE ONLY): the Item2Vec sampler, step and user rows in C."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "item2vec_oracle.c")
_SO = os.path.join(_HERE, "_build", "libitem2vec_oracle.so")
OPT_KIND = {"sgd": 0, "adam": 1, "adagrad": 2, "rmsprop": 3}
_lib = None


def build(force=False):
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                               "-shared", "-o", _SO, _SRC, "-lm"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.orc_sgns_sample.restype = C.c_int64
        L.orc_sgns_sample.argtypes = [C.c_void_p] * 3 + [C.c_int64] + [C.c_void_p] * 2 + [C.c_int32] * 2 + [C.c_void_p, C.c_int64]
        L.orc_item2vec_step.restype = C.c_double
        L.orc_item2vec_step.argtypes = ([C.c_void_p, C.c_int32, C.c_int32] + [C.c_void_p] * 3 + [C.c_int64, C.c_int32]
                                        + [C.c_float] * 4 + [C.c_void_p] * 2 + [C.c_int64, C.c_int32])
        L.orc_item2vec_user_embed.restype = None
        L.orc_item2vec_user_embed.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 2 + [C.c_void_p]
        _lib = L
    return _lib


def _c(a, dt):
    a = np.asarray(a)
    assert a.dtype == dt and a.flags.c_contiguous, (a.dtype, dt)
    return a.ctypes.data


def sgns_sample(mt_state, users, items, row_ptr, col, item_num, window):
    """-> int64 [T, 3] rows (or numpy's (0,) float64 array when T == 0); advances mt_state (uint32[625]) in place.
    ValueError as numpy raises it for a position with context and an empty complement."""
    users = np.ascontiguousarray(users, np.int32)
    items = np.ascontiguousarray(items, np.int32)
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32) if len(col) else np.zeros(1, np.int32)
    cap = 4 * int(window) * len(users) + 1
    out = np.empty((cap, 3), np.int64)
    T = lib().orc_sgns_sample(_c(mt_state, np.uint32), _c(users, np.int32), _c(items, np.int32), len(users),
                              _c(row_ptr, np.int64), _c(col, np.int32), int(item_num), int(window), out.ctypes.data, cap)
    if T == -2:
        raise ValueError("'a' cannot be empty unless no samples are taken")
    assert T >= 0
    return out[:T].copy() if T else np.array([])


def item2vec_step(Q, triples, opt, lr, state=None, step_count=1, apply=True, beta1=0.9, beta2=0.999, eps=1e-8):
    """One step on Q (fp32 [I, F], updated in place) -> fp64 loss.  state: dict with 'm' / 'v' arrays (created if empty)."""
    I, F = Q.shape
    t = np.ascontiguousarray(triples[:, 0], np.int32)
    c = np.ascontiguousarray(triples[:, 1], np.int32)
    y = np.ascontiguousarray(triples[:, 2], np.int32)
    if state is None:
        state = {}
    m = state.setdefault("m", np.zeros_like(Q))
    v = state.setdefault("v", np.zeros_like(Q))
    return lib().orc_item2vec_step(_c(Q, np.float32), I, F, t.ctypes.data, c.ctypes.data, y.ctypes.data, len(t), OPT_KIND[opt],
                                   lr, beta1, beta2, eps, _c(m, np.float32), _c(v, np.float32), int(step_count),
                                   1 if apply else 0)


def user_embed(row_ptr, col, Q, P):
    """P[u] = sum of Q over row u of the sorted CSR (non-empty rows only), in place; returns P."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    col = np.ascontiguousarray(col, np.int32) if len(col) else np.zeros(1, np.int32)
    lib().orc_item2vec_user_embed(_c(row_ptr, np.int64), _c(col, np.int32), _c(Q, np.float32), P.shape[0], P.shape[1],
                                  _c(P, np.float32))
    return P
