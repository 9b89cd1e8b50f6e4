"""CPU oracle of the Markov clustering stage (``oracle/mcl.c``) - TEST INFRASTRUCTURE ONLY.

``run(n, src, dst, w, inflation, min_weight, iters)`` returns the CSC matrix after ``iters`` iterations (or at
convergence), the iteration count, per-iteration nnz / products / chaos and one component root per node.  The
product package never imports it.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(HERE, "libmcloracle.so")
_lib = None

THETA, S, TAU, MAX_ITER = 1e-4, 1024, 1e-4, 100      # include/pgdbg.h PG_MCL_*


def build(force=False):
    src = os.path.join(HERE, "mcl.c")
    if force or not os.path.isfile(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        tmp = "%s.%d.tmp" % (_LIB_PATH, os.getpid())
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-std=gnu11", "-shared", "-fPIC", "-o", tmp, src, "-lm"])
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        vp, i64 = ctypes.c_void_p, ctypes.c_int64
        L.mclo_new.restype = vp
        L.mclo_new.argtypes = [i64, i64, vp, vp, vp, i64]
        L.mclo_iterate.argtypes = [vp, ctypes.c_double]
        L.mclo_components.argtypes = [vp, vp]
        for name in ("n", "nnz", "products"):
            getattr(L, "mclo_" + name).restype = i64
            getattr(L, "mclo_" + name).argtypes = [vp]
        L.mclo_chaos.restype = ctypes.c_float
        L.mclo_chaos.argtypes = [vp]
        for name, ct in (("colptr", ctypes.c_int64), ("rows", ctypes.c_int32), ("vals", ctypes.c_float)):
            getattr(L, "mclo_" + name).restype = ctypes.POINTER(ct)
            getattr(L, "mclo_" + name).argtypes = [vp]
        L.mclo_free.argtypes = [vp]
        _lib = L
    return _lib


def _csc(L, h):
    n, nnz = L.mclo_n(h), L.mclo_nnz(h)
    cp = np.ctypeslib.as_array(L.mclo_colptr(h), shape=(n + 1,)).copy()
    rows = np.ctypeslib.as_array(L.mclo_rows(h), shape=(nnz,)).copy() if nnz else np.zeros(0, np.int32)
    vals = np.ctypeslib.as_array(L.mclo_vals(h), shape=(nnz,)).copy() if nnz else np.zeros(0, np.float32)
    return cp, rows, vals


def run(n, src, dst, w, inflation=1.5, min_weight=1, iters=None, trace=None):
    """``iters`` = None: iterate until max chaos < TAU or MAX_ITER; else exactly ``iters`` iterations.
    ``trace(it, colptr, rows, vals)`` is called after every iteration when given."""
    L = lib()
    src = np.ascontiguousarray(src, dtype=np.int64)
    dst = np.ascontiguousarray(dst, dtype=np.int64)
    w = np.ascontiguousarray(w, dtype=np.int64)
    h = L.mclo_new(int(n), int(src.size), src.ctypes.data, dst.ctypes.data, w.ctypes.data, int(min_weight))
    try:
        stats = []
        it = 0
        limit = MAX_ITER if iters is None else int(iters)
        while it < limit:
            L.mclo_iterate(h, float(inflation))
            it += 1
            chaos = float(L.mclo_chaos(h))
            stats.append({"nnz": int(L.mclo_nnz(h)), "products": int(L.mclo_products(h)), "chaos": chaos})
            if trace is not None:
                trace(it, *_csc(L, h))
            if iters is None and np.float32(chaos) < np.float32(TAU):      # the float32 compare the GPU side makes
                break
        cp, rows, vals = _csc(L, h)
        root = np.empty(max(int(n), 1), dtype=np.int32)
        L.mclo_components(h, root.ctypes.data)
        return {"colptr": cp, "rows": rows, "vals": vals, "iterations": it, "stats": stats, "root": root[:int(n)]}
    finally:
        L.mclo_free(h)


def partition(root):
    """Canonical form of a partition given one root per node: sorted tuple of sorted member tuples."""
    groups = {}
    for i, r in enumerate(np.asarray(root).tolist()):
        groups.setdefault(r, []).append(i)
    return sorted(tuple(g) for g in groups.values())
