"""tvl1_calc_ex on the GPU: fp32 frames and an initial flow (useInitialFlow) in both semantics, bit for bit against
the CPU restatements (oracle_ex/), plus the cases in which the new entry point must reproduce tvl1_calc_u8."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth
from oracle_ex import oracle_ex as OX

pytestmark = pytest.mark.gpu

MODES = ["cpu", "cuda"]


def same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def params(gpu, mode, **kw):
    """small-pair parameters of either mode (CPU mode: explicit inner / outer counts)"""
    if mode == "cuda":
        kw.setdefault("iterations", 60)
        return gpu.default_params(semantics=gpu.SEMANTICS_CUDA, **kw)
    kw.setdefault("inner_iterations", 30)
    kw.setdefault("outer_iterations", 10)
    kw.setdefault("lambda_", 0.15)
    kw.setdefault("nscales", 5)
    return gpu.default_params(**kw)


def oracle(p, I0, I1, init):
    kw = dict(tau=p.tau, theta=p.theta, epsilon=p.epsilon, scale_step=p.scale_step, nscales=p.nscales, warps=p.warps,
              **{"lambda": p.lambda_})
    if p.semantics == 1:
        u, v, it, lev = OX.tvl1_calc_cuda_ex(I0, I1, init, iterations=p.iterations, **kw)
    else:
        u, v, it, lev = OX.tvl1_calc_ex(I0, I1, init, gamma=p.gamma, inner_iterations=p.inner_iterations,
                                        outer_iterations=p.outer_iterations, median_filtering=p.median_filtering, **kw)
    return u, v, it[:lev], lev


def f32_pair(h, w, seed):
    I0, I1 = synth.make_pair(h, w, seed=seed)
    rng = np.random.default_rng(seed)
    f = lambda a: ((a.astype(np.float32) * 257 + rng.integers(0, 257, a.shape)) / np.float32(65535)).astype(np.float32)
    return f(I0), f(I1)


def init_flow(kind, h, w, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    if kind == "shift":
        return np.full((h, w), -1.1, np.float32), np.full((h, w), 0.6, np.float32)
    if kind == "smooth":
        return ((-1.3 + 0.6 * np.sin(xx / 17.0)).astype(np.float32), (0.7 + 0.4 * np.cos(yy / 11.0)).astype(np.float32))
    if kind == "true":
        return synth.true_flow(h, w)
    if kind == "noise":      # several px per pixel: k_warp's window and global fallbacks, k_warp_cuda's gather path
        return (rng.standard_normal((h, w)) * 4).astype(np.float32), (rng.standard_normal((h, w)) * 4).astype(np.float32)
    if kind == "outside":    # every sample position outside the frame
        return np.full((h, w), 3.0 * w, np.float32), (-2.0 * h - yy).astype(np.float32)
    if kind == "huge":       # |u| up to 1e4: int16 saturation of the remap coordinates
        return ((rng.random((h, w)) * 2 - 1) * 1e4).astype(np.float32), ((rng.random((h, w)) * 2 - 1) * 1e4).astype(np.float32)
    raise KeyError(kind)


def upload_f32(a, pitch, device=0):
    """(DevBuf, byte pitch): an fp32 plane as rows of `pitch` elements, padding NaN"""
    h, w = a.shape
    buf = np.full((h, pitch), np.nan, np.float32)
    buf[:, :w] = a
    return gpu_mod().DevBuf(buf.nbytes, device).upload(buf), pitch * 4


def gpu_mod():
    from fibsem_optflow_b200 import _native
    return _native


def solve_device(s, I0, I1, init=None, frame_pitch=None, init_pitch=None, alias=False):
    """tvl1_calc_ex on device buffers.  frame_pitch / init_pitch in elements; alias: the output planes ARE the
    initial-flow planes (OpenCV's in/out flow).  Returns (u, v, iters)."""
    N = gpu_mod()
    h, w = I0.shape
    if I0.dtype == np.uint8:
        ft = N.FRAME_U8
        (b0, p0), (b1, p1) = N.upload_u8(I0, frame_pitch), N.upload_u8(I1, frame_pitch)
    else:
        ft = N.FRAME_F32
        (b0, p0), (b1, p1) = upload_f32(I0, frame_pitch or w), upload_f32(I1, frame_pitch or w)
    bufs = [b0, b1]
    ip = int(init_pitch or w)
    if init is not None:
        (bu0, pi), (bv0, _) = upload_f32(init[0], ip), upload_f32(init[1], ip)
        bufs += [bu0, bv0]
        d_u0, d_v0 = bu0.ptr, bv0.ptr
    else:
        d_u0 = d_v0 = None
        pi = 0
    if alias:
        bu, bv, po = bu0, bv0, pi
    else:
        bu, bv, po = N.DevBuf(h * w * 4).zero(), N.DevBuf(h * w * 4).zero(), w * 4
        bufs += [bu, bv]
    s.calc_ex_device(ft, b0.ptr, p0, b1.ptr, p1, w, h, d_u0, d_v0, pi, bu.ptr, bv.ptr, po)
    pw = po // 4
    u = bu.download((h, pw), np.float32)[:, :w].copy()
    v = bv.download((h, pw), np.float32)[:, :w].copy()
    for b in bufs:
        b.free()
    return u, v, s.stats.iters_array()


# ---- 1. the fp32 conversion kernel

@pytest.mark.parametrize("h,w,spitch", [(5, 1, None), (7, 3, 5), (9, 37, 37), (16, 130, 131), (33, 64, 67), (3, 257, 260)])
def test_k_convert_f32(gpu, h, w, spitch):
    rng = np.random.default_rng(h * w)
    x = np.concatenate([rng.random(h * w // 2), rng.standard_normal(h * w - h * w // 2) * 1e3]).astype(np.float32)
    x = x.reshape(h, w)
    out = gpu.k_convert_f32(x, spitch=spitch)
    assert same(out[:, :w], x * np.float32(255))
    assert not np.isnan(out).any()                          # the source's NaN padding is never read
    assert (out[:, w:(w + 3) // 4 * 4] == 0).all()         # pad columns of the 4-wide stores get 0


# ---- 2-4. the new entry point reproduces tvl1_calc_u8

@pytest.mark.parametrize("mode", MODES)
def test_ex_u8_without_init_is_calc_u8(gpu, mode):
    h, w = 97, 131
    I0, I1 = synth.make_pair(h, w, seed=3)
    s = gpu.Solver(params(gpu, mode))
    (b0, p0), (b1, p1) = gpu.upload_u8(I0, 133), gpu.upload_u8(I1, 133)
    bu, bv = gpu.DevBuf(h * w * 4), gpu.DevBuf(h * w * 4)
    s.calc_device(b0.ptr, p0, b1.ptr, p1, w, h, bu.ptr, bv.ptr, w * 4)          # tvl1_calc_u8
    it = s.stats.iters_array()
    u, v = bu.download((h, w), np.float32), bv.download((h, w), np.float32)
    gu, gv, git = solve_device(s, I0, I1, frame_pitch=133)                      # tvl1_calc_ex(U8, NULL)
    assert np.array_equal(git, it) and same(gu, u) and same(gv, v)
    hu, hv = s.calc(I0, I1)                                                      # tvl1_calc_u8_host
    assert np.array_equal(s.stats.iters_array(), it) and same(hu, u) and same(hv, v)
    for b in (b0, b1, bu, bv):
        b.free()
    s.close()


@pytest.mark.parametrize("mode", MODES)
def test_zero_init_and_u8_equivalent_f32_frames(gpu, mode):
    """a zero initial flow is no initial flow; fp32 frames holding k/255 are the 8-bit frames"""
    I0, I1 = synth.make_pair(90, 121, seed=5)
    s = gpu.Solver(params(gpu, mode))
    u, v = s.calc(I0, I1)
    it = s.stats.iters_array()
    z = np.zeros(I0.shape, np.float32)
    f0, f1 = (I0 / np.float32(255)).astype(np.float32), (I1 / np.float32(255)).astype(np.float32)
    for args in ((I0, I1, (z, z)), (f0, f1, None), (f0, f1, (z, z))):
        gu, gv = s.calc_ex(*args[:2], init=args[2])
        assert np.array_equal(s.stats.iters_array(), it) and same(gu, u) and same(gv, v)
    s.close()


# ---- 5. initial flows against the oracle

CASES = [
    # (mode, h, w, frames, init, kw)
    ("cpu", 97, 131, "u8", "shift", {}),
    ("cpu", 96, 128, "f32", "true", {}),
    ("cpu", 101, 77, "u8", "noise", {}),
    ("cpu", 96, 128, "f32", "outside", {"nscales": 3}),
    ("cpu", 80, 96, "u8", "huge", {"nscales": 3, "warps": 3}),
    ("cpu", 121, 97, "f32", "smooth", {"scale_step": 0.5, "nscales": 4}),
    ("cpu", 96, 128, "u8", "noise", {"scale_step": 0.5, "nscales": 10}),
    ("cpu", 95, 129, "f32", "smooth", {"gamma": 0.1, "nscales": 3}),
    ("cpu", 96, 128, "u8", "noise", {"gamma": 0.1, "scale_step": 0.5, "nscales": 3}),
    ("cpu", 97, 131, "u8", "smooth", {"median_filtering": 3}),
    ("cuda", 97, 131, "u8", "shift", {}),
    ("cuda", 96, 128, "f32", "true", {}),
    ("cuda", 101, 77, "u8", "noise", {}),
    ("cuda", 96, 128, "f32", "outside", {"nscales": 3}),
    ("cuda", 80, 96, "u8", "huge", {"nscales": 3, "warps": 3}),
    ("cuda", 121, 97, "f32", "smooth", {"scale_step": 0.5, "nscales": 4}),
    ("cuda", 96, 128, "u8", "noise", {"scale_step": 0.5, "nscales": 10, "iterations": 41}),
]


@pytest.mark.parametrize("mode,h,w,frames,init,kw", CASES)
def test_initial_flow_matches_oracle(gpu, mode, h, w, frames, init, kw):
    I0, I1 = f32_pair(h, w, seed=h + w) if frames == "f32" else synth.make_pair(h, w, seed=h + w)
    fl = init_flow(init, h, w, seed=w)
    p = params(gpu, mode, **kw)
    s = gpu.Solver(p)
    u, v = s.calc_ex(I0, I1, init=fl)
    it = s.stats.iters_array()
    ou, ov, oit, lev = oracle(p, I0, I1, fl)
    assert s.stats.levels == lev and np.array_equal(it, oit)
    assert same(u, ou) and same(v, ov)
    s.close()


@pytest.mark.parametrize("mode", MODES)
def test_pitched_and_aliased_init(gpu, mode):
    """device planes: a pitched initial flow (NaN padding never read), pitched fp32 frames, and the initial-flow
    planes used as the output planes (calc's in/out flow)"""
    h, w = 75, 103
    I0, I1 = f32_pair(h, w, seed=2)
    fl = init_flow("smooth", h, w)
    p = params(gpu, mode)
    ou, ov, oit, lev = oracle(p, I0, I1, fl)
    s = gpu.Solver(p)
    for kw in (dict(init_pitch=128), dict(init_pitch=107, frame_pitch=105, alias=True), dict(alias=True)):
        u, v, it = solve_device(s, I0, I1, fl, **kw)
        assert np.array_equal(it, oit) and same(u, ou) and same(v, ov), kw
    s.close()


@pytest.mark.parametrize("mode", MODES)
def test_large_pair_matches_oracle(gpu, mode):
    """the configs[0] 2048^2 pair, warm-started from a smooth flow"""
    I0, I1 = synth.make_pair(2048, 2048, seed=7)
    fl = init_flow("smooth", 2048, 2048)
    if mode == "cuda":
        p = params(gpu, mode, lambda_=0.05, nscales=10, iterations=40, warps=2)
    else:
        p = params(gpu, mode, nscales=5, warps=5)
    s = gpu.Solver(p)
    u, v = s.calc_ex(I0, I1, init=fl)
    it = s.stats.iters_array()
    ou, ov, oit, lev = oracle(p, I0, I1, fl)
    assert s.stats.levels == lev and np.array_equal(it, oit)
    assert same(u, ou) and same(v, ov)
    s.close()


# ---- 6. schedule options

@pytest.mark.parametrize("mode", MODES)
def test_every_schedule_gives_the_same_result(gpu, mode):
    I0, I1 = synth.make_pair(200, 264, seed=8)
    fl = init_flow("noise", 200, 264, seed=1)
    p = params(gpu, mode, nscales=6)
    s = gpu.Solver(p)
    u0, v0 = s.calc_ex(I0, I1, init=fl)
    it0 = s.stats.iters_array()
    s.close()
    assert it0.max() > 2
    for opts in ((("coop_outer", 0),), (("multi_iter", 0),), (("fused_min_px", 1e18),)):
        s = gpu.Solver(p)
        for k, val in opts:
            s.set_option(k, val)
        u, v = s.calc_ex(I0, I1, init=fl)
        assert np.array_equal(s.stats.iters_array(), it0), opts
        assert same(u, u0) and same(v, v0), opts
        s.close()


# ---- 7. host entry point = device entry point

@pytest.mark.parametrize("mode", MODES)
def test_host_equals_device(gpu, mode):
    h, w = 88, 120
    I0, I1 = f32_pair(h, w, seed=11)
    fl = init_flow("noise", h, w, seed=2)
    s = gpu.Solver(params(gpu, mode))
    u, v = s.calc_ex(I0, I1, init=fl)
    it = s.stats.iters_array()
    du, dv, dit = solve_device(s, I0, I1, fl)
    assert np.array_equal(dit, it) and same(du, u) and same(dv, v)
    # the staging grows from 8-bit to fp32 rows and back on one handle
    u8 = s.calc_ex(*synth.make_pair(h, w, seed=11))
    u32 = s.calc_ex(I0, I1, init=fl)
    assert same(u32[0], u) and same(u32[1], v) and not same(u8[0], u)
    s.close()


# ---- 8. refused calls

@pytest.mark.parametrize("mode", MODES)
def test_refused_calls_leave_the_handle_usable(gpu, mode):
    N = gpu
    h, w = 64, 80
    I0, I1 = f32_pair(h, w, seed=4)
    fl = init_flow("smooth", h, w)
    s = gpu.Solver(params(gpu, mode))
    u, v = s.calc_ex(I0, I1, init=fl)
    it = s.stats.iters_array()
    (b0, p0), (b1, p1) = upload_f32(I0, w + 1), upload_f32(I1, w + 1)
    (bu0, pi), (bv0, _) = upload_f32(fl[0], w), upload_f32(fl[1], w)
    bu, bv = N.DevBuf(h * w * 4), N.DevBuf(h * w * 4)
    L = N.lib()

    def call(ft=N.FRAME_F32, pa=p0, pb=p1, u0=bu0.ptr, v0=bv0.ptr, pinit=pi):
        return L.tvl1_calc_ex(s.handle, ft, b0.ptr, pa, b1.ptr, pb, w, h, u0, v0, pinit, bu.ptr, bv.ptr, w * 4, None,
                              None)

    assert call(u0=None) == -1                       # one initial-flow plane only
    assert call(v0=None) == -1
    assert call(ft=2) == -1 and call(ft=-1) == -1    # unknown frame type
    assert call(pa=p0 - 2) == -1                     # fp32 pitch not a multiple of 4
    assert call(pb=4 * w - 4) == -1                  # fp32 pitch below a row
    assert call(pinit=pi + 2) == -1                  # initial-flow pitch not a multiple of 4
    hu, hv = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
    assert L.tvl1_calc_ex_host(s.handle, N.FRAME_F32, I0.ctypes.data, 4 * w, I1.ctypes.data, 4 * w, w, h,
                               fl[0].ctypes.data, None, 4 * w, hu.ctypes.data, hv.ctypes.data, 4 * w, None) == -1
    assert call() == 0
    got = bu.download((h, w), np.float32), bv.download((h, w), np.float32)
    assert same(got[0], u) and same(got[1], v)
    u2, v2 = s.calc_ex(I0, I1, init=fl)
    assert np.array_equal(s.stats.iters_array(), it) and same(u2, u) and same(v2, v)
    with pytest.raises(gpu.Tvl1Error):
        s.calc_ex(I0.astype(np.float64), I1.astype(np.float64))
    with pytest.raises(gpu.Tvl1Error):
        s.calc_ex(I0, I1, init=(fl[0][:-1], fl[1][:-1]))
    for b in (b0, b1, bu0, bv0, bu, bv):
        b.free()
    s.close()


def test_use_initial_flow_param_stays_refused(gpu):
    with pytest.raises(gpu.Tvl1Error):
        gpu.Solver(gpu.default_params(use_initial_flow=1))


# ---- 9. a warm start from the true flow stays on it

@pytest.mark.parametrize("mode", MODES)
def test_true_flow_start_is_solved(gpu, mode):
    """Sanity, not parity: started from the true flow, the solve stays on it (mean EPE over the interior, the
    reference wrapper's defaults).  cv::cuda's algorithm lands within 0.05 px.  The CPU class does not, from any
    start: its 1/32-px remap and median leave ~0.052 px on these pairs (from zero too), so it gets the 0.08 px bar
    the suite uses for it elsewhere, and must end no farther from the truth than the zero start does."""
    for seed, (h, w) in ((3, (256, 256)), (21, (320, 384))):
        I0, I1 = synth.make_pair(h, w, seed=seed, shear=1.0 / h)
        tu, tv = synth.true_flow(h, w, shear=1.0 / h)
        p = gpu.default_params(semantics=gpu.SEMANTICS_CUDA if mode == "cuda" else gpu.SEMANTICS_CPU)
        s = gpu.Solver(p)
        u, v = s.calc_ex(I0, I1, init=(tu, tv))
        u0, v0 = s.calc_ex(I0, I1)
        s.close()
        m = 32
        epe = np.hypot(u - tu, v - tv)[m:-m, m:-m].mean()
        epe0 = np.hypot(u0 - tu, v0 - tv)[m:-m, m:-m].mean()
        assert epe <= (0.05 if mode == "cuda" else 0.08), (seed, epe)
        assert epe <= epe0 + 1e-3, (seed, epe, epe0)


def test_api_init_flow(gpu):
    from fibsem_optflow_b200 import api
    h, w = 96, 128
    I0, I1 = synth.make_pair(h, w, seed=21)
    fl = init_flow("smooth", h, w)
    tv = api.generate_TV_args({}, {})
    u, v = api.TVL1_solve(I0, I1, tv, init_flow=fl)
    p = api.params_from_TV_args(tv)
    s = gpu.Solver(p)
    ou, ov = s.calc_ex(I0, I1, init=fl)
    s.close()
    assert same(u, ou) and same(v, ov)
    u0, v0 = api.TVL1_solve(I0, I1, tv)
    assert not same(u, u0)
