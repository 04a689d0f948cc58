"""ctypes binding of libtvl1_b200.so (the C ABI in include/tvl1_b200.h).

There is NO fallback: if the shared library is missing, or no CUDA device is present when
a compute entry point is called, this module raises.  Nothing here imports oracle/.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("TVL1_SO") or os.path.join(_HERE, "csrc", "libtvl1_b200.so")   # TVL1_SO: developer builds

MAX_LEVELS = 32
MAX_WARPS = 64


class Tvl1Error(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [
        ("tau", C.c_double), ("lambda_", C.c_double), ("theta", C.c_double),
        ("epsilon", C.c_double), ("scale_step", C.c_double), ("gamma", C.c_double),
        ("nscales", C.c_int), ("warps", C.c_int), ("iterations", C.c_int),
        ("inner_iterations", C.c_int), ("outer_iterations", C.c_int),
        ("median_filtering", C.c_int), ("use_initial_flow", C.c_int),
        ("reserved", C.c_int * 3),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("levels", C.c_int), ("warps", C.c_int),
        ("width", C.c_int * MAX_LEVELS), ("height", C.c_int * MAX_LEVELS),
        ("iters", C.c_int * (MAX_LEVELS * MAX_WARPS)),
        ("outer", C.c_int * (MAX_LEVELS * MAX_WARPS)),
        ("total_iterations", C.c_longlong), ("px_iterations", C.c_longlong),
        ("algorithmic_bytes", C.c_double),
        ("ms_total", C.c_float), ("ms_pyramid", C.c_float), ("ms_warp", C.c_float),
        ("ms_iterate", C.c_float), ("ms_median", C.c_float), ("ms_other", C.c_float),
        ("ms_iterate_level", C.c_float * MAX_LEVELS),
        ("launches", C.c_longlong),
    ]

    def iters_array(self):
        a = np.ctypeslib.as_array(self.iters)[: self.levels * self.warps]
        return a.reshape(self.levels, self.warps).copy()

    def outer_array(self):
        a = np.ctypeslib.as_array(self.outer)[: self.levels * self.warps]
        return a.reshape(self.levels, self.warps).copy()

    def level_sizes(self):
        return [(self.width[i], self.height[i]) for i in range(self.levels)]


class FeatureParams(C.Structure):
    _fields_ = [
        ("nfeatures", C.c_int), ("scale_factor", C.c_float), ("nlevels", C.c_int), ("edge_threshold", C.c_int),
        ("first_level", C.c_int), ("patch_size", C.c_int), ("fast_threshold", C.c_int), ("ratio", C.c_float),
        ("ransac", C.c_double), ("homo", C.c_int), ("debug", C.c_int), ("reserved", C.c_int * 4),
    ]


class StackIO(C.Structure):
    _fields_ = [
        ("h_slices", C.POINTER(C.c_void_p)), ("pitch", C.c_size_t),
        ("n_slices", C.c_int), ("width", C.c_int), ("height", C.c_int), ("apply_mask", C.c_int),
        ("h_u", C.POINTER(C.c_void_p)), ("h_v", C.POINTER(C.c_void_p)), ("pitch_out", C.c_size_t),
        ("npoints", C.c_int), ("scale", C.c_float), ("seed", C.c_longlong),
        ("px", C.c_void_p), ("py", C.c_void_p), ("qx", C.c_void_p), ("qy", C.c_void_p), ("w", C.c_void_p),
        ("n_out", C.c_void_p), ("stats", C.POINTER(Stats)), ("prescale", C.c_double),
        ("pair_p", C.POINTER(C.c_int)), ("pair_q", C.POINTER(C.c_int)), ("n_pairs", C.c_int),
    ]


# every symbol include/tvl1_b200.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "tvl1_version", "tvl1_last_error", "tvl1_default_params", "tvl1_create", "tvl1_destroy",
    "tvl1_set_params", "tvl1_set_option", "tvl1_set_timing", "tvl1_calc_u8", "tvl1_calc_u8_host",
    "tvl1_prescaled_size", "tvl1_prescale_u8", "tvl1_prescale_u8_host",
    "tvl1_mask_flow_u8", "tvl1_finish_flow_u8", "tvl1_sample_matches", "tvl1_sample_matches_skip", "tvl1_sample_matches_ex",
    "tvl1_default_feature_params", "tvl1_find_alignment", "tvl1_warp_affine_u8", "tvl1_warp_affine_f32", "tvl1_stack_run", "tvl1_k_convert_u8", "tvl1_k_resize",
    "tvl1_k_centered_gradient", "tvl1_k_warp", "tvl1_k_iterate", "tvl1_k_iterate_fused2", "tvl1_k_outer", "tvl1_k_iterate_gamma", "tvl1_k_median5", "tvl1_k_median3", "tvl1_k_last_ms",
    "tvl1_k_gauss7_u8", "tvl1_k_fast_corners", "tvl1_k_describe", "tvl1_k_knn2", "tvl1_features_extract",
    "tvl1_pyramid_sizes", "tvl1_glibc_rand", "tvl1_selftest_arith", "tvl1_dev_count", "tvl1_dev_alloc", "tvl1_dev_free",
    "tvl1_dev_memset", "tvl1_dev_h2d", "tvl1_dev_d2h", "tvl1_dev_sync", "tvl1_set_device", "tvl1_stream_create",
    "tvl1_stream_destroy", "tvl1_stream_sync", "tvl1_stream_query", "tvl1_stream_wait", "tvl1_dev_h2d_async", "tvl1_dev_d2h_async",
    "tvl1_host_alloc_pinned", "tvl1_host_free_pinned",
]

_lib = None
_vp = C.c_void_p
_sz = C.c_size_t


def lib():
    """Loads the library; raises if it has not been built (python fibsem_optflow_b200/csrc/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise Tvl1Error(
            "%s is missing: build it with `python fibsem_optflow_b200/csrc/build.py` "
            "(there is no CPU fallback)" % SO_PATH)
    L = C.CDLL(SO_PATH)
    if os.environ.get("TVL1_SO"):
        # developer A/B builds may predate newer entry points: give them inert placeholders
        class _Missing:
            argtypes = restype = None
        for name in EXPORTS:
            if not hasattr(L, name):
                setattr(L, name, _Missing())
    L.tvl1_version.restype = C.c_char_p
    L.tvl1_last_error.restype = C.c_char_p
    L.tvl1_default_params.argtypes = [C.POINTER(Params)]
    L.tvl1_default_params.restype = None
    L.tvl1_create.argtypes = [C.POINTER(Params), C.c_int, C.POINTER(_vp)]
    L.tvl1_destroy.argtypes = [_vp]
    L.tvl1_destroy.restype = None
    L.tvl1_set_params.argtypes = [_vp, C.POINTER(Params)]
    L.tvl1_set_timing.argtypes = [_vp, C.c_int]
    L.tvl1_set_option.argtypes = [_vp, C.c_char_p, C.c_double]
    L.tvl1_calc_u8.argtypes = [_vp, _vp, _sz, _vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz, _vp,
                               C.POINTER(Stats)]
    L.tvl1_calc_u8_host.argtypes = [_vp, _vp, _sz, _vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz,
                                    C.POINTER(Stats)]
    L.tvl1_mask_flow_u8.argtypes = [_vp, _vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz, _vp]
    L.tvl1_finish_flow_u8.argtypes = [_vp, _vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz, C.c_int, _vp]
    L.tvl1_sample_matches.argtypes = [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _sz, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                      C.c_longlong, _vp, _vp, _vp, _vp, _vp, _vp,
                                      C.POINTER(C.c_int), _vp]
    L.tvl1_sample_matches_ex.argtypes = [_vp, _vp, _sz, _vp, _sz, _vp, _vp, _sz, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                         C.c_longlong, C.c_longlong, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp,
                                         C.POINTER(C.c_int), C.POINTER(C.c_longlong), _vp]
    L.tvl1_default_feature_params.argtypes = [C.POINTER(FeatureParams)]
    L.tvl1_default_feature_params.restype = None
    L.tvl1_find_alignment.argtypes = [_vp, _vp, _sz, C.c_int, C.c_int, _vp, _sz, C.c_int, C.c_int,
                                      C.POINTER(FeatureParams), _vp, C.POINTER(C.c_int), C.POINTER(C.c_int), _vp]
    L.tvl1_warp_affine_u8.argtypes = [_vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz, C.c_int, C.c_int, _vp]
    L.tvl1_warp_affine_f32.argtypes = [_vp, _sz, C.c_int, C.c_int, _vp, _vp, _sz, C.c_int, C.c_int, _vp]
    L.tvl1_stack_run.argtypes = [_vp, C.POINTER(StackIO), C.POINTER(C.c_float)]
    L.tvl1_k_convert_u8.argtypes = [_vp, _sz, C.c_int, C.c_int, _vp, C.c_int, _vp]
    L.tvl1_k_resize.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, C.c_int, C.c_int, C.c_int,
                                C.c_double, C.c_float, _vp]
    L.tvl1_k_centered_gradient.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]
    L.tvl1_k_warp.argtypes = [_vp] * 4 + [C.c_int, C.c_int, C.c_int] + [_vp] * 6
    L.tvl1_k_iterate.argtypes = [_vp] * 10 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_float,
                                              C.c_float, C.c_int, _vp, _vp]
    L.tvl1_k_iterate_fused2.argtypes = L.tvl1_k_iterate.argtypes
    L.tvl1_k_outer.argtypes = L.tvl1_k_iterate.argtypes
    L.tvl1_k_iterate_gamma.argtypes = [_vp] * 12 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                                    C.c_float, C.c_int, _vp, _vp]
    L.tvl1_prescaled_size.argtypes = [C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.tvl1_prescale_u8.argtypes = [_vp, _sz, C.c_int, C.c_int, C.c_double, _vp, _sz, _vp]
    L.tvl1_prescale_u8_host.argtypes = [C.c_int, _vp, _sz, C.c_int, C.c_int, C.c_double, _vp, _sz]
    L.tvl1_k_median5.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp]
    L.tvl1_k_median3.argtypes = L.tvl1_k_median5.argtypes
    L.tvl1_k_last_ms.argtypes = [C.POINTER(C.c_float)]
    L.tvl1_k_gauss7_u8.argtypes = [_vp, _sz, C.c_int, C.c_int, _vp, _sz, _vp]
    L.tvl1_k_fast_corners.argtypes = [_vp, _sz, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp]
    L.tvl1_k_describe.argtypes = [_vp, _sz, _vp, _sz, _vp, C.c_int, C.c_float, C.c_int, _vp, _vp, _vp]
    L.tvl1_k_knn2.argtypes = [_vp, C.c_int, _vp, C.c_int, _vp, _vp, _vp, _vp]
    L.tvl1_features_extract.argtypes = [_vp, _vp, _sz, C.c_int, C.c_int, C.POINTER(FeatureParams), _vp, _vp, C.c_int,
                                        C.POINTER(C.c_int), _vp]
    L.tvl1_pyramid_sizes.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, _vp, _vp]
    L.tvl1_glibc_rand.argtypes = [C.c_longlong, C.c_longlong, C.c_int, _vp]
    L.tvl1_selftest_arith.argtypes = [C.c_longlong, C.c_uint, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.tvl1_dev_alloc.argtypes = [C.c_int, _sz, C.POINTER(_vp)]
    L.tvl1_dev_free.argtypes = [C.c_int, _vp]
    L.tvl1_dev_memset.argtypes = [_vp, C.c_int, _sz]
    L.tvl1_dev_h2d.argtypes = [_vp, _vp, _sz]
    L.tvl1_dev_d2h.argtypes = [_vp, _vp, _sz]
    L.tvl1_dev_sync.argtypes = [C.c_int]
    L.tvl1_set_device.argtypes = [C.c_int]
    L.tvl1_stream_create.argtypes = [C.c_int, C.POINTER(_vp)]
    for _n in ("tvl1_stream_destroy", "tvl1_stream_sync", "tvl1_stream_query"):
        getattr(L, _n).argtypes = [_vp]
    L.tvl1_stream_wait.argtypes = [_vp, _vp]
    L.tvl1_dev_h2d_async.argtypes = [_vp, _vp, _sz, _vp]
    L.tvl1_dev_d2h_async.argtypes = [_vp, _vp, _sz, _vp]
    L.tvl1_host_alloc_pinned.argtypes = [_sz, C.POINTER(_vp)]
    L.tvl1_host_free_pinned.argtypes = [_vp]
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise Tvl1Error("tvl1 error %d: %s" % (rc, lib().tvl1_last_error().decode()))
    return rc


def device_count():
    return lib().tvl1_dev_count()


def require_device():
    n = device_count()
    if n <= 0:
        raise Tvl1Error("no CUDA device visible; fibsem_optflow_b200 has no CPU path")
    return n


def default_params(**kw):
    p = Params()
    lib().tvl1_default_params(C.byref(p))
    for k, v in kw.items():
        k = {"lambda": "lambda_", "scaleStep": "scale_step", "useInitialFlow": "use_initial_flow",
             "innerIterations": "inner_iterations", "outerIterations": "outer_iterations",
             "medianFiltering": "median_filtering"}.get(k, k)
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


def pyramid_sizes(w, h, nscales, scale_step):
    ws = (C.c_int * (MAX_LEVELS + 1))()
    hs = (C.c_int * (MAX_LEVELS + 1))()
    n = check(lib().tvl1_pyramid_sizes(w, h, nscales, scale_step, ws, hs))
    return [(ws[i], hs[i]) for i in range(n)]


def prescale_u8(src, scale, device=0):
    """8-bit cv::resize(src, Size(), scale, scale) of the reference's loader, on the device."""
    src = np.ascontiguousarray(src, np.uint8)
    h, w = src.shape
    dw, dh = C.c_int(0), C.c_int(0)
    check(lib().tvl1_prescaled_size(w, h, float(scale), C.byref(dw), C.byref(dh)))
    dst = np.empty((dh.value, dw.value), np.uint8)
    check(lib().tvl1_prescale_u8_host(device, src.ctypes.data, w, w, h, float(scale), dst.ctypes.data, dw.value))
    return dst


def k_last_ms():
    ms = C.c_float(0)
    check(lib().tvl1_k_last_ms(C.byref(ms)))
    return ms.value


def selftest_arith(n, seed=1, elo=-30, ehi=30, with_unvouched=False):
    bad, unv = C.c_longlong(-1), C.c_longlong(-1)
    check(lib().tvl1_selftest_arith(n, seed, elo, ehi, C.byref(bad), C.byref(unv)))
    return (bad.value, unv.value) if with_unvouched else bad.value


def glibc_rand(seed, skip, n):
    out = np.zeros(n, np.int32)
    check(lib().tvl1_glibc_rand(seed, skip, n, out.ctypes.data))
    return out


class DevBuf:
    """A device allocation (tvl1_dev_alloc) with NumPy upload/download helpers."""

    def __init__(self, nbytes, device=0):
        self.device = device
        self.nbytes = int(nbytes)
        p = _vp()
        check(lib().tvl1_dev_alloc(device, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def free(self):
        if self.ptr:
            lib().tvl1_dev_free(self.device, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        check(lib().tvl1_dev_h2d(self.ptr, arr.ctypes.data, arr.nbytes))
        return self

    def download(self, shape, dtype):
        out = np.empty(shape, dtype)
        assert out.nbytes <= self.nbytes
        check(lib().tvl1_dev_d2h(out.ctypes.data, self.ptr, out.nbytes))
        return out

    def zero(self):
        check(lib().tvl1_dev_memset(self.ptr, 0, self.nbytes))
        return self


def pitch_of(w):
    return (w + 31) // 32 * 32


class Plane:
    """A pitched fp32 device plane (pitch multiple of 32 floats, pad columns zeroed)."""

    def __init__(self, h, w, device=0, data=None):
        self.h, self.w, self.pitch = h, w, pitch_of(w)
        self.buf = DevBuf(self.h * self.pitch * 4, device)
        if data is None:
            self.buf.zero()
        else:
            self.set(data)

    @property
    def ptr(self):
        return self.buf.ptr

    def set(self, data):
        a = np.zeros((self.h, self.pitch), np.float32)
        a[:, : self.w] = data
        self.buf.upload(a)

    def get(self):
        return self.buf.download((self.h, self.pitch), np.float32)[:, : self.w].copy()


class Solver:
    """One solver handle on one device (tvl1_create .. tvl1_destroy)."""

    def __init__(self, params=None, device=0, **kw):
        require_device()
        self.params = params if params is not None else default_params(**kw)
        self.device = device
        h = _vp()
        check(lib().tvl1_create(C.byref(self.params), device, C.byref(h)))
        self.handle = h.value
        self.stats = Stats()

    def close(self):
        if getattr(self, "handle", None):
            lib().tvl1_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        check(lib().tvl1_set_option(self.handle, key.encode(), float(value)))

    def set_timing(self, enabled=True):
        """Per-stage CUDA-event times in `stats` (off by default: only ms_total is measured)."""
        check(lib().tvl1_set_timing(self.handle, int(bool(enabled))))

    def set_params(self, params):
        check(lib().tvl1_set_params(self.handle, C.byref(params)))
        self.params = params

    def calc(self, I0, I1):
        """Host uint8 images -> (u, v) host float32; H2D and D2H inside (tvl1_calc_u8_host)."""
        I0 = np.ascontiguousarray(I0, np.uint8)
        I1 = np.ascontiguousarray(I1, np.uint8)
        if I0.ndim != 2 or I0.shape != I1.shape:
            raise Tvl1Error("frames must be 2-D uint8 arrays of equal size")
        h, w = I0.shape
        u = np.empty((h, w), np.float32)
        v = np.empty((h, w), np.float32)
        check(lib().tvl1_calc_u8_host(self.handle, I0.ctypes.data, w, I1.ctypes.data, w, w, h,
                                      u.ctypes.data, v.ctypes.data, w * 4, C.byref(self.stats)))
        return u, v

    def calc_device(self, d_f0, pitch0, d_f1, pitch1, w, h, d_u, d_v, pitch_out, stream=None):
        check(lib().tvl1_calc_u8(self.handle, d_f0, pitch0, d_f1, pitch1, w, h, d_u, d_v,
                                 pitch_out, stream, C.byref(self.stats)))

    def mask_flow_device(self, d_f1, pitch1, w, h, d_u, d_v, pitch_out, stream=None):
        check(lib().tvl1_mask_flow_u8(self.handle, d_f1, pitch1, w, h, d_u, d_v, pitch_out, stream))

    def finish_flow_device(self, d_f1, pitch1, w, h, d_u, d_v, pitch_out, add_grid, stream=None):
        """output_type "map": + coordinate grid; then flow = 0 where frame1 <= 1 (src/optflow.cpp:445-473).
        add_grid -1 subtracts the grid (the "flow" output of the features path, :434-438); d_f1 None: no mask."""
        g = int(add_grid)
        check(lib().tvl1_finish_flow_u8(self.handle, d_f1, pitch1, w, h, d_u, d_v, pitch_out, (g > 0) - (g < 0), stream))

    def find_alignment(self, moving, fixed, pitch_moving=None, pitch_fixed=None, pad_value=255, **kw):
        """find_alignment (src/features.cpp:46-167): host uint8 frames in, (affine 2x3 float32 mapping `moving`
        coordinates to `fixed` coordinates, n_matches, n_good) out.  kw: fields of tvl1_feature_params.
        pitch_*: the frames go up as rows of that many bytes, the padding filled with pad_value."""
        moving = np.ascontiguousarray(moving, np.uint8)
        fixed = np.ascontiguousarray(fixed, np.uint8)
        p = feature_params(**kw)
        bm, pm = upload_u8(moving, pitch_moving, pad_value, self.device)
        bf, pf = upload_u8(fixed, pitch_fixed, pad_value, self.device)
        aff = np.zeros(6, np.float32)
        nm, ng = C.c_int(0), C.c_int(0)
        try:
            check(lib().tvl1_find_alignment(self.handle, bm.ptr, pm, moving.shape[1], moving.shape[0],
                                            bf.ptr, pf, fixed.shape[1], fixed.shape[0], C.byref(p),
                                            aff.ctypes.data, C.byref(nm), C.byref(ng), None))
        finally:
            bm.free()
            bf.free()
        return aff.reshape(2, 3), nm.value, ng.value

    def features_extract(self, img, pitch=None, pad_value=255, **kw):
        """One frame's keypoints (KEYPT_DTYPE) and descriptors ((n, 8) uint32) as tvl1_find_alignment computes
        them (tvl1_features_extract).  kw: fields of tvl1_feature_params."""
        img = np.ascontiguousarray(img, np.uint8)
        p = feature_params(**kw)
        b, pb = upload_u8(img, pitch, pad_value, self.device)
        kp = DevBuf(p.nfeatures * KEYPT_DTYPE.itemsize, self.device)
        desc = DevBuf(p.nfeatures * 32, self.device)
        n = C.c_int(0)
        try:
            check(lib().tvl1_features_extract(self.handle, b.ptr, pb, img.shape[1], img.shape[0], C.byref(p),
                                              kp.ptr, desc.ptr, p.nfeatures, C.byref(n), None))
            n = n.value
            return kp.download(n, KEYPT_DTYPE), desc.download((n, 8), np.uint32)
        finally:
            for x in (b, kp, desc):
                x.free()

    def sample_matches_device(self, d_f0, pitch0, d_f1, pitch1, d_u, d_v, pitch_flow, w, h,
                              roi0=(0, 0), roi1=(0, 0), scale=0.5, npoints=25, seed=-1,
                              stream=None, q_is_map=False):
        n = max(int(npoints), 1)
        px, py, qx, qy, wg = (np.zeros(n, np.float64) for _ in range(5))
        pos = np.zeros((n, 2), np.int32)
        k = C.c_int(0)
        check(lib().tvl1_sample_matches_ex(self.handle, d_f0, pitch0, d_f1, pitch1, d_u, d_v,
                                           pitch_flow, w, h, roi0[0], roi0[1], roi1[0], roi1[1],
                                           scale, npoints, seed, 0, int(bool(q_is_map)), px.ctypes.data, py.ctypes.data,
                                           qx.ctypes.data, qy.ctypes.data, wg.ctypes.data,
                                           pos.ctypes.data, C.byref(k), None, stream))
        k = k.value
        return px[:k], py[:k], qx[:k], qy[:k], wg[:k], pos[:k]

    def run_stack(self, slices, flows=True, apply_mask=False, npoints=-1, scale=0.5, seed=-1,
                  out_u=None, out_v=None, slice_ptrs=None, pitch=None, shape=None, prescale=0.0, pairs=None):
        """Pairs (k, k+1) of a stack of uint8 slices -- or the explicit `pairs` [(p, q), ...] of slice
        indices -- through tvl1_stack_run.  Returns a dict with
        'u', 'v' (lists of planes, if flows), 'matches' (per pair px,py,qx,qy,w, if npoints >= 0),
        'stats' (per pair), 'ms' (CUDA-event time of the whole stack).  slice_ptrs/out_u/out_v let
        the caller pass pinned host memory (bench.py); otherwise NumPy arrays are used."""
        if slice_ptrs is None:
            slices = [np.ascontiguousarray(s, np.uint8) for s in slices]
            h, w = slices[0].shape
            slice_ptrs = [s.ctypes.data for s in slices]
            pitch = w
        else:
            h, w = shape
        n = len(slice_ptrs)
        npairs = n - 1 if pairs is None else len(pairs)
        io = StackIO()
        if pairs is not None:   # explicit (p, q) slice indices instead of the chain (k, k+1)
            ap = (C.c_int * npairs)(*[int(p) for p, _ in pairs])
            aq = (C.c_int * npairs)(*[int(q) for _, q in pairs])
            io.pair_p, io.pair_q, io.n_pairs = ap, aq, npairs
        arr = (C.c_void_p * n)(*slice_ptrs)
        io.h_slices = arr
        io.pitch = pitch
        io.n_slices, io.width, io.height = n, w, h
        io.apply_mask = int(bool(apply_mask))
        io.prescale = float(prescale)
        if prescale not in (0.0, 1.0):   # the flow planes have the prescaled size
            dw, dh = C.c_int(0), C.c_int(0)
            check(lib().tvl1_prescaled_size(w, h, float(prescale), C.byref(dw), C.byref(dh)))
            w, h = dw.value, dh.value
        us = vs = None
        if flows:
            if out_u is None:
                us = [np.empty((h, w), np.float32) for _ in range(npairs)]
                vs = [np.empty((h, w), np.float32) for _ in range(npairs)]
                out_u = [a.ctypes.data for a in us]
                out_v = [a.ctypes.data for a in vs]
            au = (C.c_void_p * npairs)(*out_u)
            av = (C.c_void_p * npairs)(*out_v)
            io.h_u, io.h_v = au, av
            io.pitch_out = w * 4
        io.npoints = int(npoints)
        io.scale = float(scale)
        io.seed = int(seed)
        cap = max(int(npoints), 1)
        if npoints >= 0:
            m = [np.zeros(npairs * cap, np.float64) for _ in range(5)]
            nout = np.zeros(npairs, np.int32)
            io.px, io.py, io.qx, io.qy, io.w = (a.ctypes.data for a in m)
            io.n_out = nout.ctypes.data
        stats = (Stats * npairs)()
        io.stats = stats
        ms = C.c_float(0)
        check(lib().tvl1_stack_run(self.handle, C.byref(io), C.byref(ms)))
        res = {"ms": ms.value, "stats": list(stats)}
        if flows:
            res["u"], res["v"] = us, vs
        if npoints >= 0:
            res["matches"] = [tuple(a[k * cap: k * cap + int(nout[k])] for a in m) for k in range(npairs)]
        return res

    def sample_matches(self, f0, f1, u, v, **kw):
        """Host arrays in, match arrays out (uploads the four planes)."""
        f0 = np.ascontiguousarray(f0, np.uint8)
        f1 = np.ascontiguousarray(f1, np.uint8)
        u = np.ascontiguousarray(u, np.float32)
        v = np.ascontiguousarray(v, np.float32)
        h, w = f0.shape
        b0 = DevBuf(f0.nbytes, self.device).upload(f0)
        b1 = DevBuf(f1.nbytes, self.device).upload(f1)
        bu = DevBuf(u.nbytes, self.device).upload(u)
        bv = DevBuf(v.nbytes, self.device).upload(v)
        try:
            return self.sample_matches_device(b0.ptr, w, b1.ptr, w, bu.ptr, bv.ptr, w * 4, w, h, **kw)
        finally:
            for b in (b0, b1, bu, bv):
                b.free()


# ---- stage-level helpers (tests / profiling): host arrays in, host arrays out

def k_convert_u8(img, device=0):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    src = DevBuf(img.nbytes, device).upload(img)
    dst = Plane(h, w, device)
    check(lib().tvl1_k_convert_u8(src.ptr, w, w, h, dst.ptr, dst.pitch, None))
    check(lib().tvl1_dev_sync(device))
    return dst.get()


def k_resize(src, dw=None, dh=None, inv_scale=0.0, mul=1.0, device=0):
    src = np.asarray(src, np.float32)
    sh, sw = src.shape
    if inv_scale > 0:   # resize(src, Size(), f, f): dsize = round-half-even(n * f)
        dw, dh = int(np.rint(sw * inv_scale)), int(np.rint(sh * inv_scale))
    s = Plane(sh, sw, device, src)
    d = Plane(dh, dw, device)
    check(lib().tvl1_k_resize(s.ptr, sw, sh, s.pitch, d.ptr, dw, dh, d.pitch, inv_scale, mul, None))
    check(lib().tvl1_dev_sync(device))
    return d.get()


def k_centered_gradient(src, device=0):
    src = np.asarray(src, np.float32)
    h, w = src.shape
    s = Plane(h, w, device, src)
    dx, dy = Plane(h, w, device), Plane(h, w, device)
    check(lib().tvl1_k_centered_gradient(s.ptr, w, h, s.pitch, dx.ptr, dy.ptr, None))
    check(lib().tvl1_dev_sync(device))
    return dx.get(), dy.get()


def k_warp(I0, I1, u1, u2, device=0):
    """Returns I1w, I1wx, I1wy, grad, rho_c (the centred gradients of I1 are formed in-kernel)."""
    h, w = np.asarray(I0).shape
    ins = [Plane(h, w, device, np.asarray(a, np.float32)) for a in (I0, I1, u1, u2)]
    outs = [Plane(h, w, device) for _ in range(5)]
    check(lib().tvl1_k_warp(*[p.ptr for p in ins], w, h, ins[0].pitch, *[p.ptr for p in outs], None))
    check(lib().tvl1_dev_sync(device))
    return tuple(p.get() for p in outs)


def k_iterate(I1wx, I1wy, grad, rho_c, u1, u2, p11, p12, p21, p22, l_t, theta, taut, n=1, device=0,
              fused=False):
    """n iterations; returns (u1,u2,p11,p12,p21,p22, errors[n]).  fused: two per launch;
    fused="outer": all n in one cooperative k_outer launch (the shipped schedule)."""
    h, w = np.asarray(u1).shape
    consts = [Plane(h, w, device, np.asarray(a, np.float32)) for a in (I1wx, I1wy, grad, rho_c)]
    state = [Plane(h, w, device, np.asarray(a, np.float32)) for a in (u1, u2, p11, p12, p21, p22)]
    errs = np.zeros(max(n, 1), np.float64)
    fn = lib().tvl1_k_outer if fused == "outer" else (lib().tvl1_k_iterate_fused2 if fused else lib().tvl1_k_iterate)
    check(fn(*[p.ptr for p in consts], *[p.ptr for p in state], w, h,
             state[0].pitch, l_t, theta, taut, n, errs.ctypes.data, None))
    return tuple(p.get() for p in state) + (errs[:n],)


def k_iterate_gamma(I1wx, I1wy, rho_c, u1, u2, u3, p11, p12, p21, p22, p31, p32, l_t, theta, taut, gamma, n=1, device=0):
    """n iterations of the three-channel form (gamma != 0); returns (u1,u2,u3,p11..p32, errors[n])."""
    h, w = np.asarray(u1).shape
    consts = [Plane(h, w, device, np.asarray(a, np.float32)) for a in (I1wx, I1wy, rho_c)]
    state = [Plane(h, w, device, np.asarray(a, np.float32)) for a in (u1, u2, u3, p11, p12, p21, p22, p31, p32)]
    errs = np.zeros(max(n, 1), np.float64)
    check(lib().tvl1_k_iterate_gamma(*[p.ptr for p in consts], *[p.ptr for p in state], w, h, state[0].pitch,
                                     l_t, theta, taut, gamma, n, errs.ctypes.data, None))
    return tuple(p.get() for p in state) + (errs[:n],)


def warp_affine(src, affine, dsize, device=0, spitch=None, dpitch=None):
    """cv::warpAffine(src, affine, dsize = (w, h), INTER_LINEAR, BORDER_CONSTANT 0) on the device; uint8 or float32.
    spitch / dpitch: row pitches in ELEMENTS of the device copies (default: the widths); padding holds a marker
    value (255 resp. NaN) that must neither be read nor be overwritten."""
    src = np.ascontiguousarray(src)
    aff = np.ascontiguousarray(affine, np.float32).reshape(6)
    dw, dh = int(dsize[0]), int(dsize[1])
    sh, sw = src.shape
    sp, dp = spitch or sw, dpitch or dw
    mark = 255 if src.dtype == np.uint8 else np.nan
    a = np.full((sh, sp), mark, src.dtype)
    a[:, :sw] = src
    bs = DevBuf(a.nbytes, device).upload(a)
    bd = DevBuf(dh * dp * src.itemsize, device).upload(np.full((dh, dp), mark, src.dtype))
    e = src.itemsize
    if src.dtype == np.uint8:
        check(lib().tvl1_warp_affine_u8(bs.ptr, sp, sw, sh, aff.ctypes.data, bd.ptr, dp, dw, dh, None))
    else:
        assert src.dtype == np.float32
        check(lib().tvl1_warp_affine_f32(bs.ptr, sp * e, sw, sh, aff.ctypes.data, bd.ptr, dp * e, dw, dh, None))
    check(lib().tvl1_dev_sync(device))
    out = bd.download((dh, dp), src.dtype)
    bs.free()
    bd.free()
    pad = out[:, dw:]
    assert (pad == 255).all() if src.dtype == np.uint8 else np.isnan(pad).all(), "warp_affine wrote into the row padding"
    return np.ascontiguousarray(out[:, :dw])


# ---- the feature kernels (tvl1_k_gauss7_u8 .. tvl1_features_extract)

CAND_DTYPE = np.dtype([("harris", "<f4"), ("x", "<u2"), ("y", "<u2")])            # struct Cand
KEYPT_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("angle", "<f4"), ("level", "<i4")])   # struct KeyPt


def feature_params(**kw):
    """tvl1_default_feature_params with the given fields replaced (OpenCV's ORB names accepted)"""
    p = FeatureParams()
    lib().tvl1_default_feature_params(C.byref(p))
    for k, v in kw.items():
        k = {"scaleFactor": "scale_factor", "edgeThreshold": "edge_threshold", "firstLevel": "first_level",
             "patchSize": "patch_size", "fastThreshold": "fast_threshold"}.get(k, k)
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


def upload_u8(img, pitch=None, pad_value=255, device=0):
    """(DevBuf, pitch): an 8-bit image on the device as rows of `pitch` bytes (default: its width), the
    padding filled with pad_value"""
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    pitch = int(pitch or w)
    a = np.full((h, pitch), pad_value, np.uint8)
    a[:, :w] = img
    return DevBuf(a.nbytes, device).upload(a), pitch


def k_gauss7_u8(img, spitch=None, dpitch=None, device=0):
    """7x7 Gaussian (sigma 2) of an 8-bit image; the output's row padding must stay untouched"""
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    s, sp = upload_u8(img, spitch, 255, device)
    dp = int(dpitch or w)
    d = DevBuf(h * dp, device).upload(np.full((h, dp), 77, np.uint8))
    check(lib().tvl1_k_gauss7_u8(s.ptr, sp, w, h, d.ptr, dp, None))
    check(lib().tvl1_dev_sync(device))
    out = d.download((h, dp), np.uint8)
    assert (out[:, w:] == 77).all(), "k_gauss7_u8 wrote into the row padding"
    return np.ascontiguousarray(out[:, :w])


def k_fast_corners(img, border, t, pitch=None, spitch=None, cap=None, device=0):
    """k_fast_score + k_nms_harris: (score plane, candidates (CAND_DTYPE, device order), count, 2048-bin histogram)"""
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    b, pb = upload_u8(img, pitch, 255, device)
    sp = int(spitch or w)
    cap = int(cap if cap is not None else h * w // 2 + 1)
    score = DevBuf(h * sp * 4, device).zero()
    cand = DevBuf(max(cap, 1) * CAND_DTYPE.itemsize, device)
    cnt = DevBuf((1 + 2048) * 4, device).zero()
    check(lib().tvl1_k_fast_corners(b.ptr, pb, w, h, border, t, score.ptr, sp, cand.ptr, cap, cnt.ptr, cnt.ptr + 4, None))
    check(lib().tvl1_dev_sync(device))
    counters = cnt.download(1 + 2048, np.int32)
    n = int(counters[0])
    out = (score.download((h, sp), np.float32)[:, :w].copy(), cand.download(min(n, cap), CAND_DTYPE), n, counters[1:])
    for x in (b, score, cand, cnt):
        x.free()
    return out


def k_describe(img, blur, cand, scale=1.0, level=0, pitch=None, bpitch=None, device=0):
    """k_describe of the candidates `cand` (CAND_DTYPE or (x, y) pairs): keypoints (KEYPT_DTYPE), (n, 8) uint32"""
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    c = np.asarray(cand)
    if c.dtype != CAND_DTYPE:
        xy = np.asarray(c, np.int64).reshape(-1, 2)
        c = np.zeros(len(xy), CAND_DTYPE)
        c["x"], c["y"] = xy[:, 0], xy[:, 1]
    n = len(c)
    bi, pi = upload_u8(img, pitch, 255, device)
    bb, pbb = upload_u8(blur, bpitch, 255, device)
    bc = DevBuf(max(n, 1) * CAND_DTYPE.itemsize, device).upload(c)
    kp = DevBuf(max(n, 1) * KEYPT_DTYPE.itemsize, device)
    desc = DevBuf(max(n, 1) * 32, device)
    check(lib().tvl1_k_describe(bi.ptr, pi, bb.ptr, pbb, bc.ptr, n, scale, level, kp.ptr, desc.ptr, None))
    check(lib().tvl1_dev_sync(device))
    out = kp.download(n, KEYPT_DTYPE), desc.download((n, 8), np.uint32)
    for x in (bi, bb, bc, kp, desc):
        x.free()
    return out


def k_knn2(q, t, device=0):
    """Hamming 2-NN of (nq, 8) uint32 query descriptors among (nt, 8) train descriptors: idx1, d1, d2"""
    q = np.ascontiguousarray(q, np.uint32).reshape(-1, 8)
    t = np.ascontiguousarray(t, np.uint32).reshape(-1, 8)
    nq, nt = len(q), len(t)
    bq = DevBuf(max(q.nbytes, 4), device).upload(q)
    bt = DevBuf(max(t.nbytes, 4), device).upload(t)
    outs = [DevBuf(max(nq, 1) * 4, device) for _ in range(3)]
    check(lib().tvl1_k_knn2(bq.ptr, nq, bt.ptr, nt, *[o.ptr for o in outs], None))
    check(lib().tvl1_dev_sync(device))
    res = tuple(o.download(nq, np.int32) for o in outs)
    for x in [bq, bt] + outs:
        x.free()
    return res


def k_median3(src, device=0):
    src = np.asarray(src, np.float32)
    h, w = src.shape
    s = Plane(h, w, device, src)
    d = Plane(h, w, device)
    check(lib().tvl1_k_median3(s.ptr, w, h, s.pitch, d.ptr, None))
    check(lib().tvl1_dev_sync(device))
    return d.get()


def k_median5(src, device=0):
    src = np.asarray(src, np.float32)
    h, w = src.shape
    s = Plane(h, w, device, src)
    d = Plane(h, w, device)
    check(lib().tvl1_k_median5(s.ptr, w, h, s.pitch, d.ptr, None))
    check(lib().tvl1_dev_sync(device))
    return d.get()
