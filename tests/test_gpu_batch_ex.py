"""tvl1_calc_batch_ex: every pair of a batch against tvl1_calc_ex of that pair alone (flow planes array_equal, iteration
and outer-iteration counts equal) in cv::cuda semantics, with gamma, fp32 frames and initial flows, and on small sizes
against the CPU oracles directly."""
import ctypes as C

import numpy as np
import pytest

from fibsem_optflow_b200 import _native as N, api, synth
from oracle import oracle as O, oracle_cuda as OC
from oracle_ex import oracle_ex as OX
from test_gpu_batch import mixed_pairs

pytestmark = pytest.mark.gpu


def cuda_params(**kw):
    return N.default_params(semantics=N.SEMANTICS_CUDA, **kw)


def oracle_kw(p):
    return dict(tau=p.tau, theta=p.theta, epsilon=p.epsilon, scale_step=p.scale_step, nscales=p.nscales,
                warps=p.warps, **{"lambda": p.lambda_})


def oracle(p, I0, I1, init=None):
    """(u, v, iters of the levels used) of the oracle of p's semantics"""
    kw = oracle_kw(p)
    if p.semantics == N.SEMANTICS_CUDA:
        if init is None and I0.dtype == np.uint8:
            u, v, it, lev = OC.tvl1_calc_cuda(I0, I1, iterations=p.iterations, **kw)
        else:
            u, v, it, lev = OX.tvl1_calc_cuda_ex(I0, I1, init, iterations=p.iterations, **kw)
        return u, v, it[:lev]
    kw.update(gamma=p.gamma, median_filtering=p.median_filtering)
    if p.inner_iterations > 0:   # otherwise both derive them from `iterations`, as the solver does
        kw.update(inner_iterations=p.inner_iterations, outer_iterations=p.outer_iterations)
    if init is None and I0.dtype == np.uint8:
        u, v, it, lev = O.tvl1_calc(I0, I1, **kw)
    else:
        u, v, it, lev = OX.tvl1_calc_ex(I0, I1, init, **kw)
    return u, v, it[:lev]


def singles(s, pairs, init=None):
    res = []
    for k, (I0, I1) in enumerate(pairs):
        u, v = s.calc_ex(I0, I1, init=None if init is None else init[k])
        res.append((u, v, s.stats.iters_array(), s.stats.outer_array()))
    return res


def assert_batch_matches(s, pairs, init=None, want=None):
    got = s.calc_batch_ex([p[0] for p in pairs], [p[1] for p in pairs], init)
    stats = s.batch_stats
    want = want if want is not None else singles(s, pairs, init)
    assert len(got) == len(pairs) == len(stats)
    for k, ((u, v), (wu, wv, wit, wout)) in enumerate(zip(got, want)):
        assert np.array_equal(u, wu) and np.array_equal(v, wv), "pair %d: flow differs from tvl1_calc_ex" % k
        assert np.array_equal(stats[k].iters_array(), wit), "pair %d: iteration counts differ" % k
        assert np.array_equal(stats[k].outer_array(), wout), "pair %d: outer iteration counts differ" % k
    return got, stats


def assert_oracle(p, pairs, got, stats, init=None, which=None):
    for k in which if which is not None else range(len(pairs)):
        ou, ov, oit = oracle(p, pairs[k][0], pairs[k][1], None if init is None else init[k])
        assert np.array_equal(stats[k].iters_array(), oit), "pair %d: iteration counts differ from the oracle" % k
        assert np.array_equal(got[k][0], ou) and np.array_equal(got[k][1], ov), "pair %d differs from the oracle" % k


def f32_pairs(pairs, seed=0):
    """fp32 frames in [0, 1] whose x 255 is not an integer"""
    rng = np.random.default_rng(seed)
    f = lambda a: ((a.astype(np.float32) * 257 + rng.integers(0, 257, a.shape)) / np.float32(65535)).astype(np.float32)
    return [(f(I0), f(I1)) for I0, I1 in pairs]


def random_flows(h, w, n, seed=0, amp=2.0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    out = []
    for k in range(n):
        a, b = rng.uniform(-1, 1, 2)
        u = (amp * a * np.sin(xx / (7.0 + k)) + rng.standard_normal((h, w)) * 0.3).astype(np.float32)
        v = (amp * b * np.cos(yy / (5.0 + k)) + rng.standard_normal((h, w)) * 0.3).astype(np.float32)
        out.append((u, v))
    return out


# ---- cuda semantics

def test_cuda_mixed_stops_against_single_and_oracle(gpu):
    p = cuda_params(lambda_=0.15, nscales=5, iterations=120)
    pairs = mixed_pairs(96, 128, 7)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs)
    totals = {st.total_iterations for st in stats}
    assert len(totals) >= 3, "the pairs were meant to stop at different counts: %s" % totals
    assert_oracle(p, pairs, got, stats)
    assert all((st.outer_array() == 0).all() and st.ms_median == 0 for st in stats)
    s.close()


@pytest.mark.parametrize("n", [1, 2, 7, 33])
def test_cuda_batch_sizes(gpu, n):
    s = N.Solver(cuda_params(nscales=4, iterations=80))
    assert_batch_matches(s, mixed_pairs(48, 72, n, seed=n))
    s.close()


@pytest.mark.parametrize("hw", [(37, 101), (50, 203), (33, 259)])
def test_cuda_odd_widths(gpu, hw):
    h, w = hw
    p = cuda_params(lambda_=0.15, nscales=6, iterations=100)
    pairs = mixed_pairs(h, w, 5, seed=w)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs)
    assert_oracle(p, pairs, got, stats, which=[0, 4])
    s.close()


def test_cuda_roi_strip(gpu):
    """the production shape, 100-row strips of 4096 px, with the wrapper defaults in cuda semantics"""
    s = N.Solver(cuda_params())
    _, stats = assert_batch_matches(s, mixed_pairs(100, 4096, 3, seed=5))
    assert all((st.outer_array() == 0).all() for st in stats)
    s.close()


@pytest.mark.parametrize("kw", [
    dict(iterations=1), dict(iterations=2), dict(iterations=7), dict(epsilon=0.0, iterations=40),
    dict(scale_step=0.5), dict(nscales=1), dict(warps=1),
])
def test_cuda_parameters(gpu, kw):
    p = cuda_params(**dict(dict(lambda_=0.15, nscales=5, iterations=90), **kw))
    pairs = mixed_pairs(57, 83, 5, seed=3)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs)
    assert_oracle(p, pairs, got, stats, which=[0, 1])
    assert all((st.outer_array() == 0).all() for st in stats)
    s.close()


# ---- gamma (CPU-class semantics)

@pytest.mark.parametrize("gamma", [0.25, 1.0])
@pytest.mark.parametrize("median", [1, 3, 5])
def test_gamma(gpu, gamma, median):
    p = N.default_params(lambda_=0.15, nscales=4, gamma=gamma, median_filtering=median)
    pairs = mixed_pairs(53, 91, 5, seed=int(gamma * 8) + median)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs)
    assert_oracle(p, pairs, got, stats, which=[0, 1, 4])
    s.close()


# ---- fp32 frames

@pytest.mark.parametrize("mode", ["cpu", "cuda"])
def test_f32_frames(gpu, mode):
    p = cuda_params(lambda_=0.15, nscales=5, iterations=90) if mode == "cuda" else \
        N.default_params(lambda_=0.15, nscales=5, inner_iterations=20, outer_iterations=6)
    pairs = f32_pairs(mixed_pairs(61, 99, 5, seed=11), seed=1)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs)
    assert_oracle(p, pairs, got, stats, which=[0, 1])
    s.close()


# ---- initial flows

def mode_params(mode, **kw):
    if mode == "cuda":
        return cuda_params(**dict(dict(lambda_=0.15, nscales=5, iterations=90), **kw))
    return N.default_params(**dict(dict(lambda_=0.15, nscales=5, inner_iterations=20, outer_iterations=6), **kw))


@pytest.mark.parametrize("mode", ["cpu", "cuda"])
@pytest.mark.parametrize("f32", [False, True])
def test_initial_flows(gpu, mode, f32):
    h, w = 58, 87
    pairs = mixed_pairs(h, w, 5, seed=21)
    if f32:
        pairs = f32_pairs(pairs, seed=2)
    init = random_flows(h, w, 5, seed=3)
    p = mode_params(mode)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs, init)
    assert_oracle(p, pairs, got, stats, init=init, which=[0, 1, 3])
    s.close()


@pytest.mark.parametrize("mode", ["cpu", "cuda"])
def test_initial_flow_gamma_and_half_step(gpu, mode):
    kw = dict(scale_step=0.5) if mode == "cuda" else dict(scale_step=0.5, gamma=0.25, median_filtering=3)
    h, w = 64, 90
    pairs = mixed_pairs(h, w, 4, seed=31)
    init = random_flows(h, w, 4, seed=4, amp=3.0)
    p = mode_params(mode, **kw)
    s = N.Solver(p)
    got, stats = assert_batch_matches(s, pairs, init)
    assert_oracle(p, pairs, got, stats, init=init, which=[0])
    s.close()


@pytest.mark.parametrize("mode", ["cpu", "cuda"])
def test_zero_initial_flow_is_zero_start(gpu, mode):
    h, w = 45, 77
    pairs = mixed_pairs(h, w, 5, seed=41)
    s = N.Solver(mode_params(mode))
    a = s.calc_batch_ex([p[0] for p in pairs], [p[1] for p in pairs])
    sa = [st.iters_array() for st in s.batch_stats]
    zero = [(np.zeros((h, w), np.float32), np.zeros((h, w), np.float32)) for _ in pairs]
    b = s.calc_batch_ex([p[0] for p in pairs], [p[1] for p in pairs], zero)
    for k in range(len(pairs)):
        assert np.array_equal(a[k][0], b[k][0]) and np.array_equal(a[k][1], b[k][1])
        assert np.array_equal(sa[k], s.batch_stats[k].iters_array())
    s.close()


def upload_f32(a, pitch):
    """(DevBuf, byte pitch): an fp32 plane as rows of `pitch` elements, padding NaN"""
    h, w = a.shape
    buf = np.full((h, pitch), np.nan, np.float32)
    buf[:, :w] = a
    return N.DevBuf(buf.nbytes, 0).upload(buf), pitch * 4


@pytest.mark.parametrize("mode", ["cpu", "cuda"])
@pytest.mark.parametrize("alias", [False, True])
def test_pitched_poisoned_aliased_and_repeated(gpu, mode, alias):
    """fp32 frames and initial flows at pitches that are not multiples of 32 with NaN padding, entries that repeat,
    and (alias) the output planes being the initial-flow planes; nothing past column w - 1 is written"""
    h, w = 45, 77
    pairs = f32_pairs(mixed_pairs(h, w, 4, seed=9), seed=5)
    init = random_flows(h, w, 4, seed=6)
    s = N.Solver(mode_params(mode))
    want = singles(s, pairs, init)
    pf, pi, po = 83, 81, 85   # row pitches in elements
    order = [0, 1, 2, 3, 1, 1]
    f0 = [upload_f32(I0, pf)[0] for I0, _ in pairs]
    f1 = [upload_f32(I1, pf)[0] for _, I1 in pairs]
    if alias:   # one in/out plane per entry (a repeated entry gets planes of its own)
        u0 = [upload_f32(init[k][0], pi)[0] for k in order]
        v0 = [upload_f32(init[k][1], pi)[0] for k in order]
        outs_u, outs_v, pitch_out = u0, v0, pi * 4
    else:       # shared initial-flow planes for repeated entries
        u0 = [upload_f32(init[k][0], pi)[0] for k in range(4)]
        v0 = [upload_f32(init[k][1], pi)[0] for k in range(4)]
        u0, v0 = [u0[k] for k in order], [v0[k] for k in order]
        outs_u = [N.DevBuf(h * po * 4, 0).upload(np.full((h, po), np.nan, np.float32)) for _ in order]
        outs_v = [N.DevBuf(h * po * 4, 0).upload(np.full((h, po), np.nan, np.float32)) for _ in order]
        pitch_out = po * 4
    s.calc_batch_ex_device(N.FRAME_F32, [f0[k].ptr for k in order], pf * 4, [f1[k].ptr for k in order], pf * 4, w, h,
                           [b.ptr for b in u0], [b.ptr for b in v0], pi * 4, [b.ptr for b in outs_u],
                           [b.ptr for b in outs_v], pitch_out)
    pw = pitch_out // 4
    for j, k in enumerate(order):
        u = outs_u[j].download((h, pw), np.float32)
        v = outs_v[j].download((h, pw), np.float32)
        assert np.isnan(u[:, w:]).all() and np.isnan(v[:, w:]).all(), "the output padding was written"
        assert np.array_equal(u[:, :w], want[k][0]) and np.array_equal(v[:, :w], want[k][1]), "entry %d" % j
        assert np.array_equal(s.batch_stats[j].iters_array(), want[k][2])
    for b in set(f0 + f1 + list(u0) + list(v0) + list(outs_u) + list(outs_v)):
        b.free()
    s.close()


# ---- one handle, many kinds of solve

def test_handle_reuse_deterministic_and_interleaved(gpu):
    pairs = mixed_pairs(64, 96, 6, seed=4)
    f0, f1 = [p[0] for p in pairs], [p[1] for p in pairs]
    pg = N.default_params(lambda_=0.15, nscales=5, gamma=0.25)
    p0 = N.default_params(lambda_=0.15, nscales=5)
    s = N.Solver(pg)
    a = s.calc_batch_ex(f0, f1)                                      # a gamma batch
    s.set_params(p0)
    small = [(I0[:40, :50].copy(), I1[:40, :50].copy()) for I0, I1 in pairs[:3]]
    b = s.calc_batch_ex([p[0] for p in small], [p[1] for p in small])   # a non-gamma batch of another size
    want_b = singles(s, small)                                       # single-pair solves
    s.set_params(pg)
    single_g = singles(s, pairs[:2])
    c = s.calc_batch_ex(f0, f1)                                      # the first batch again
    for k in range(len(pairs)):
        assert np.array_equal(a[k][0], c[k][0]) and np.array_equal(a[k][1], c[k][1])
    for k in range(2):
        assert np.array_equal(a[k][0], single_g[k][0]) and np.array_equal(a[k][1], single_g[k][1])
    for k in range(len(small)):
        assert np.array_equal(b[k][0], want_b[k][0]) and np.array_equal(b[k][1], want_b[k][1])
    s.close()


# ---- refusals

def raw_call(s, n, ft, f0, p0, f1, p1, w, h, u0, v0, pi, u, v, po):
    arr = lambda xs: None if xs is None else (C.c_void_p * max(len(xs), 1))(*xs)
    return N.lib().tvl1_calc_batch_ex(s.handle, n, ft, arr(f0), p0, arr(f1), p1, w, h, arr(u0), arr(v0), pi, arr(u),
                                      arr(v), po, None, None)


def last_error():
    return N.lib().tvl1_last_error().decode()


def test_refusals(gpu):
    h, w = 24, 40
    bufs = [N.DevBuf(h * 64 * 4, 0).zero() for _ in range(6)]
    f, g, u, v, a, b = (x.ptr for x in bufs)
    U8, F32 = N.FRAME_U8, N.FRAME_F32
    s = N.Solver(cuda_params(nscales=3, iterations=20))
    call = lambda *args: raw_call(s, *args)
    assert call(2, F32, [f, f], 256, [g, g], 256, w, h, [a, a], [b, b], 256, [u, u], [v, v], 256) == 0, last_error()
    assert call(1, F32, [f], 256, [g], 256, w, h, [a], None, 256, [u], [v], 256) == -1 and "both" in last_error()
    assert call(1, F32, [f], 256, [g], 256, w, h, None, [b], 256, [u], [v], 256) == -1 and "both" in last_error()
    assert call(2, F32, [f, f], 256, [g, g], 256, w, h, [a, None], [b, b], 256, [u, u], [v, v], 256) == -1 \
        and "entry 1" in last_error()
    assert call(1, 2, [f], 256, [g], 256, w, h, None, None, 0, [u], [v], 256) == -1 and "frame_type" in last_error()
    assert call(1, F32, [f], 254, [g], 256, w, h, None, None, 0, [u], [v], 256) == -1 and "pitch" in last_error()
    assert call(1, F32, [f], 256, [g], 256, 40, h, [a], [b], 162, [u], [v], 256) == -1 and "pitch" in last_error()
    assert call(1, U8, [f], 39, [g], 64, w, h, None, None, 0, [u], [v], 256) == -1 and "pitch" in last_error()
    assert call(0, U8, [], 64, [], 64, w, h, None, None, 0, [], [], 256) == -1 and "n must be" in last_error()
    assert call(32768, U8, [f], 64, [g], 64, w, h, None, None, 0, [u], [v], 256) == -1 and "n must be" in last_error()
    # a batch whose state does not fit on the device: nothing of it stays allocated and the handle keeps working
    big = 8192
    fb = N.DevBuf(big * big, 0).zero()
    ub = N.DevBuf(big * big * 4, 0)
    n = 64   # ~4 GB of state per 8192^2 pair
    rc = raw_call(s, n, U8, [fb.ptr] * n, big, [fb.ptr] * n, big, big, big, None, None, 0, [ub.ptr] * n, [ub.ptr] * n,
                  big * 4)
    assert rc == -4 and "batch" in last_error()
    assert call(2, U8, [f, f], 64, [g, g], 64, w, h, None, None, 0, [u, u], [v, v], 256) == 0, last_error()
    I0, I1 = synth.make_pair(h, w, seed=1, margin=6)
    u1, v1 = s.calc_ex(I0, I1)
    (u2, v2), = s.calc_batch_ex([I0], [I1])
    assert np.array_equal(u1, u2) and np.array_equal(v1, v2)
    for x in bufs + [fb, ub]:
        x.free()
    s.close()


# ---- Python

@pytest.mark.parametrize("extra", [{"semantics": "cuda", "iterations": 80}, {"gamma": 0.25}, {"init": True},
                                   {"semantics": "cuda", "init": True}])
def test_api_solve_batch(gpu, extra):
    extra = dict(extra)
    use_init = extra.pop("init", False)
    h, w = 50, 70
    pairs = mixed_pairs(h, w, 3, seed=6)
    tv = api.generate_TV_args({}, dict({"lambda": 0.15, "nscales": 4}, **extra))
    init = random_flows(h, w, 3, seed=7) if use_init else None
    got = api.TVL1_solve_batch([p[0] for p in pairs], [p[1] for p in pairs], tv, init_flows=init)
    for k, ((u, v), (I0, I1)) in enumerate(zip(got, pairs)):
        wu, wv = api.TVL1_solve(I0, I1, tv, init_flow=None if init is None else init[k])
        assert np.array_equal(u, wu) and np.array_equal(v, wv)
