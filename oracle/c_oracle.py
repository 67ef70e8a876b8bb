"""ctypes binding of oracle/libgf_oracle.so (the C restatement).  TEST INFRASTRUCTURE ONLY --
see the header of oracle/gf_oracle.c.  Never imported by the product package."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "libgf_oracle.so")
    src = os.path.join(_HERE, "gf_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "lib"], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = ctypes.CDLL(build())
        fp = ctypes.POINTER(ctypes.c_float)
        dp = ctypes.POINTER(ctypes.c_double)
        i64 = ctypes.c_int64
        ci = ctypes.c_int
        L.gf_oracle_num_threads.restype = ci
        L.gf_oracle_box_mean_f32.argtypes = [fp, fp, ci, ci, i64, i64, ci, ci, ci]
        L.gf_oracle_guided_gray_f32.argtypes = [fp, fp, fp, fp, fp, ci, ci, i64, ci, ctypes.c_float, ci, ci]
        L.gf_oracle_guided_gray_f64.argtypes = [dp, dp, dp, dp, dp, ci, ci, i64, ci, ctypes.c_double, ci, ci]
        L.gf_oracle_guided_color_f32.argtypes = [fp, fp, fp, ci, ci, i64, i64, i64, ci, ctypes.c_float, ci, ci]
        _LIB = L
    return _LIB


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def num_threads() -> int:
    return lib().gf_oracle_num_threads()


def box_mean_f32(src, r, border, nthreads=1):
    src = np.ascontiguousarray(src, dtype=np.float32)
    h, w = src.shape
    dst = np.empty_like(src)
    rc = lib().gf_oracle_box_mean_f32(_fp(src), _fp(dst), w, h, w, w, r, border, nthreads)
    assert rc == 0, rc
    return dst


def guided_gray_f32(I, p, r, eps, border=0, nthreads=1, return_ab=False):
    I = np.ascontiguousarray(I, dtype=np.float32)
    p = np.ascontiguousarray(p, dtype=np.float32)
    h, w = I.shape
    q = np.empty_like(I)
    A = np.empty_like(I) if return_ab else None
    B = np.empty_like(I) if return_ab else None
    rc = lib().gf_oracle_guided_gray_f32(_fp(I), _fp(p), _fp(q), _fp(A) if return_ab else None,
                                         _fp(B) if return_ab else None, w, h, w, r, eps, border, nthreads)
    assert rc == 0, rc
    return (q, A, B) if return_ab else q


def guided_gray_f64(I, p, r, eps, border=0, nthreads=1, return_ab=False):
    I = np.ascontiguousarray(I, dtype=np.float64)
    p = np.ascontiguousarray(p, dtype=np.float64)
    h, w = I.shape
    q = np.empty_like(I)
    A = np.empty_like(I) if return_ab else None
    B = np.empty_like(I) if return_ab else None
    rc = lib().gf_oracle_guided_gray_f64(_dp(I), _dp(p), _dp(q), _dp(A) if return_ab else None,
                                         _dp(B) if return_ab else None, w, h, w, r, eps, border, nthreads)
    assert rc == 0, rc
    return (q, A, B) if return_ab else q


def guided_color_f32(I3, p, r, eps, border=0, nthreads=1):
    I3 = np.ascontiguousarray(I3, dtype=np.float32)
    p = np.ascontiguousarray(p, dtype=np.float32)
    h, w, c = I3.shape
    assert c == 3
    q = np.empty_like(p)
    rc = lib().gf_oracle_guided_color_f32(_fp(I3), _fp(p), _fp(q), w, h, 3 * w, w, w, r, eps, border, nthreads)
    assert rc == 0, rc
    return q
