"""TEST INFRASTRUCTURE ONLY -- ctypes loader for oracle/libctc_ref.so (the C restatement of
the reference's CPU CTC operator, oracle/ctc_ref.c).  Used by tests/ as a second oracle and
by bench.py as the timed CPU baseline (`cpu_baseline.kind == "port"`)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libctc_ref.so")
    srcs = [os.path.join(_HERE, f) for f in ("ctc_ref.c", "ctc_ref_impl.h")]
    stale = (not os.path.exists(so)) or any(
        os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", "libctc_ref.so"],
                              stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
        for suf, ct in (("f32", ctypes.c_float), ("f64", ctypes.c_double)):
            fn = getattr(_LIB, "ctc_ref_loss_grad_" + suf)
            fn.restype = ctypes.c_int
            P = ctypes.POINTER
            fn.argtypes = [P(ct), ctypes.c_long, ctypes.c_long, P(ct), ctypes.c_long, ctypes.c_long,
                           P(ctypes.c_int), ctypes.c_int, P(ctypes.c_int), P(ctypes.c_int),
                           P(ct), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                           P(ct), P(ctypes.c_int), ctypes.c_int]
        _LIB.ctc_ref_max_threads.restype = ctypes.c_int
    return _LIB


def max_threads() -> int:
    return int(lib().ctc_ref_max_threads())


def _to_i32(a):
    """Truncated toward zero, then saturated to int32: the library clamps lengths to [0, T] / [0, Lmax] and labels
    to [0, V-1], so values beyond int32 (a length of 2^40, a label of 1e10) keep their meaning."""
    a = np.asarray(a)
    a = a.astype(np.int64) if a.dtype.kind in "iu" else np.trunc(a.astype(np.float64)).astype(np.int64)
    return np.clip(a, np.iinfo(np.int32).min, np.iinfo(np.int32).max).astype(np.int32)


def ctc_ref(data, label, T_b, L_b, blank=0, head_grad=None, layout="TNC", dtype=np.float32,
            need_grad=True, num_threads=0, out_grad=None):
    """Loss (B,) and gradient (same layout as data) of the C restatement.

    data: (T,B,V) for layout 'TNC' or (B,T,V) for 'NTC' (addressed through strides, no copy).
    """
    ct = ctypes.c_float if dtype == np.float32 else ctypes.c_double
    x = np.ascontiguousarray(data, dtype=dtype)
    if layout == "TNC":
        T, B, V = x.shape
        st_t, st_b = B * V, V
    else:
        B, T, V = x.shape
        st_t, st_b = V, T * V
    lab = np.ascontiguousarray(_to_i32(label))
    Lmax = lab.shape[1] if lab.ndim == 2 and lab.shape[1] > 0 else 0
    if Lmax == 0:
        lab = np.zeros((B, 1), np.int32)
    tl = np.ascontiguousarray(_to_i32(T_b))
    ll = np.ascontiguousarray(_to_i32(L_b))
    costs = np.zeros((B,), dtype=dtype)
    feas = np.zeros((B,), dtype=np.int32)
    g = None
    if need_grad:
        g = out_grad if out_grad is not None else np.empty_like(x)
    hg = None if head_grad is None else np.ascontiguousarray(head_grad, dtype=dtype)
    P = ctypes.POINTER
    fn = getattr(lib(), "ctc_ref_loss_grad_" + ("f32" if dtype == np.float32 else "f64"))
    rc = fn(x.ctypes.data_as(P(ct)), st_t, st_b,
            g.ctypes.data_as(P(ct)) if g is not None else None, st_t, st_b,
            lab.ctypes.data_as(P(ctypes.c_int)), max(Lmax, 1) if Lmax == 0 else Lmax,
            ll.ctypes.data_as(P(ctypes.c_int)), tl.ctypes.data_as(P(ctypes.c_int)),
            hg.ctypes.data_as(P(ct)) if hg is not None else None,
            T, B, V, int(blank), costs.ctypes.data_as(P(ct)),
            feas.ctypes.data_as(P(ctypes.c_int)), int(num_threads))
    if rc != 0:
        raise ValueError("ctc_ref: invalid arguments")
    return costs, g, feas.astype(bool)
