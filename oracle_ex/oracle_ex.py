"""ctypes front end of oracle_ex/tvl1_oracle_ex.c: fp32 frames and an initial flow in both restatements.

TEST INFRASTRUCTURE ONLY, same rules as oracle/oracle.py: the product package never imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle.oracle import OrcParams, default_params  # noqa: F401  (the parameter block is shared)

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORC = os.path.join(os.path.dirname(_HERE), "oracle")
_SO = os.path.join(_HERE, "libtvl1_oracle_ex.so")
_SRC = [os.path.join(_HERE, f) for f in ("tvl1_oracle_ex.c", "tvl1_oracle_ex.h")] + [
    os.path.join(_ORC, f) for f in ("tvl1_oracle_cuda.c", "tvl1_oracle_cuda.h", "tvl1_oracle.c", "tvl1_oracle.h")]
# the flags of oracle/Makefile: every fp32 operation rounds once
CMD = ["/usr/bin/gcc", "-O3", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall",
       "-Wno-misleading-indentation", "-shared", "-o", _SO, os.path.join(_HERE, "tvl1_oracle_ex.c"), "-lm"]

FRAME_U8 = 0
FRAME_F32 = 1


def build(force=False):
    if force or not os.path.exists(_SO) or any(os.path.getmtime(_SO) < os.path.getmtime(s) for s in _SRC):
        subprocess.check_call(CMD, cwd=_HERE)
    return _SO


_lib = None
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_SO)
    L.orc_convert_f32.argtypes = [_f32p, C.c_long, C.c_int, C.c_int, _f32p]
    L.orc_convert_f32.restype = None
    for n in ("orc_flow_down", "orc_flow_down_cuda"):
        getattr(L, n).argtypes = [_f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_int, C.c_double]
        getattr(L, n).restype = None
    L.orc_tvl1_calc_ex.argtypes = [C.POINTER(OrcParams), C.c_int, C.c_void_p, C.c_long, C.c_void_p, C.c_long, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p, _f32p, _f32p, C.c_void_p]
    L.orc_tvl1_calc_ex.restype = C.c_int
    L.orc_tvl1_calc_cuda_ex.argtypes = [C.POINTER(OrcParams), C.c_int] + L.orc_tvl1_calc_ex.argtypes[1:]
    L.orc_tvl1_calc_cuda_ex.restype = C.c_int
    _lib = L
    return L


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def convert_f32(frame):
    """Level 0 of an fp32 frame: convertTo(CV_32F, 255.0)."""
    frame = _f32(frame)
    h, w = frame.shape
    dst = np.empty((h, w), np.float32)
    lib().orc_convert_f32(frame, w, w, h, dst)
    return dst


def flow_down(src, step, cuda=False):
    """One level of the initial flow's pyramid: resize by `step`, then times `step` (CPU class: cv::multiply's
    double scalar; cuda: fp32)."""
    src = _f32(src)
    h, w = src.shape
    dw, dh = int(np.rint(w * step)), int(np.rint(h * step))
    dst = np.empty((dh, dw), np.float32)
    (lib().orc_flow_down_cuda if cuda else lib().orc_flow_down)(src, w, h, dst, dw, dh, float(step))
    return dst


def _frames(I0, I1):
    if I0.dtype != I1.dtype or I0.shape != I1.shape or I0.ndim != 2:
        raise ValueError("frames must be 2-D arrays of one dtype and size")
    if I0.dtype == np.uint8:
        return FRAME_U8, np.ascontiguousarray(I0), np.ascontiguousarray(I1)
    if I0.dtype == np.float32:
        return FRAME_F32, np.ascontiguousarray(I0), np.ascontiguousarray(I1)
    raise ValueError("frames must be uint8 or float32, not %s" % I0.dtype)


def _calc(fn, lead, I0, I1, init, p):
    ft, I0, I1 = _frames(np.asarray(I0), np.asarray(I1))
    h, w = I0.shape
    u0 = v0 = None
    if init is not None:
        u0, v0 = _f32(init[0]), _f32(init[1])
        assert u0.shape == (h, w) and v0.shape == (h, w)
    u = np.empty((h, w), np.float32)
    v = np.empty((h, w), np.float32)
    iters = np.full((p.nscales, p.warps), -1, np.int32)
    n = fn(C.byref(p), *lead, ft, I0.ctypes.data, w, I1.ctypes.data, w, w, h,
           None if u0 is None else u0.ctypes.data, None if v0 is None else v0.ctypes.data, u, v, iters.ctypes.data)
    if n < 0:
        raise RuntimeError("%s failed: %d" % (fn.__name__, n))
    return u, v, iters, n


def tvl1_calc_ex(I0, I1, init=None, params=None, **kw):
    """The CPU-class solve of uint8 or float32 frames from the initial flow init = (u0, v0) (None: zero):
    (u, v, iters[nscales][warps], levels_used).  kw: fields of orc_params."""
    p = params if params is not None else default_params(**kw)
    return _calc(lib().orc_tvl1_calc_ex, (), I0, I1, init, p)


def tvl1_calc_cuda_ex(I0, I1, init=None, iterations=300, params=None, **kw):
    """The same in cv::cuda's algorithm (`iterations` per (level, warp))."""
    p = params if params is not None else default_params(**kw)
    return _calc(lib().orc_tvl1_calc_cuda_ex, (int(iterations),), I0, I1, init, p)
