"""ctypes front end of the cv::cuda-semantics restatement (oracle/tvl1_oracle_cuda.c).

TEST INFRASTRUCTURE ONLY, same rules as oracle/oracle.py: the product package never imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from .oracle import OrcParams, default_params  # noqa: F401  (the parameter block is shared)

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libtvl1_oracle_cuda.so")
_SRC = [os.path.join(_HERE, f) for f in ("tvl1_oracle_cuda.c", "tvl1_oracle_cuda.h", "tvl1_oracle.c", "tvl1_oracle.h")]
# the flags of oracle/Makefile: every fp32 operation rounds once
CMD = ["/usr/bin/gcc", "-O3", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall",
       "-Wno-misleading-indentation", "-shared", "-o", _SO, os.path.join(_HERE, "tvl1_oracle_cuda.c"), "-lm"]


def build(force=False):
    if force or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in _SRC):
        subprocess.check_call(CMD, cwd=_HERE)
    return _SO


_lib = None
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_SO)
    L.orc_resize_cuda.argtypes = [_f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_int, C.c_double]
    L.orc_resize_cuda.restype = None
    L.orc_warp_cuda.argtypes = [_f32p] * 4 + [C.c_int, C.c_int, C.c_void_p] + [_f32p] * 4
    L.orc_warp_cuda.restype = None
    L.orc_tvl1_calc_cuda.argtypes = [C.POINTER(OrcParams), C.c_int, _u8p, C.c_long, _u8p, C.c_long, C.c_int,
                                     C.c_int, _f32p, _f32p, C.c_void_p]
    L.orc_tvl1_calc_cuda.restype = C.c_int
    _lib = L
    return L


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def resize_cuda(src, dw=None, dh=None, inv_scale=0.0):
    """cuda::resize(INTER_LINEAR): by inv_scale (> 0; size round-half-even) or to dw x dh."""
    src = _f32(src)
    h, w = src.shape
    if inv_scale > 0:
        dw, dh = int(np.rint(w * inv_scale)), int(np.rint(h * inv_scale))
    dst = np.empty((dh, dw), np.float32)
    lib().orc_resize_cuda(src, w, h, dst, dw, dh, float(inv_scale))
    return dst


def warp_cuda(I0, I1, u1, u2):
    """warpBackward + calcGradRho: (I1w, I1wx, I1wy, grad, rho_c)."""
    I0, I1, u1, u2 = map(_f32, (I0, I1, u1, u2))
    h, w = I0.shape
    out = [np.empty_like(I0) for _ in range(5)]
    lib().orc_warp_cuda(I0, I1, u1, u2, w, h, out[0].ctypes.data, out[1], out[2], out[3], out[4])
    return tuple(out)


def tvl1_calc_cuda(I0, I1, iterations=300, params=None, **kw):
    """The whole solve in cv::cuda's algorithm: (u, v, iters[nscales][warps], levels_used).  kw: fields of
    orc_params (tau, lambda, theta, epsilon, scale_step, nscales, warps, nthreads)."""
    p = params if params is not None else default_params(**kw)
    I0 = np.ascontiguousarray(I0, np.uint8)
    I1 = np.ascontiguousarray(I1, np.uint8)
    h, w = I0.shape
    u = np.empty((h, w), np.float32)
    v = np.empty((h, w), np.float32)
    iters = np.full((p.nscales, p.warps), -1, np.int32)
    n = lib().orc_tvl1_calc_cuda(C.byref(p), int(iterations), I0, w, I1, w, w, h, u, v, iters.ctypes.data)
    if n < 0:
        raise RuntimeError("orc_tvl1_calc_cuda failed: %d" % n)
    return u, v, iters, n
