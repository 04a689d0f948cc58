"""tvl1_calc_batch_u8: every pair of a batch against tvl1_calc_u8 of that pair alone (flow planes array_equal, iteration
and outer-iteration counts equal) and, on small sizes, against the C oracle directly."""
import ctypes as C

import numpy as np
import pytest

from fibsem_optflow_b200 import _native as N, api, synth

pytestmark = pytest.mark.gpu


def mixed_pairs(h, w, n, seed=0):
    """n pairs whose solves stop at very different counts: textures and shifts of their own, identical frames, an
    all-zero pair and a pair with zero bands, cycled"""
    out = []
    for k in range(n):
        kind = k % 5
        if kind == 3:
            out.append((np.zeros((h, w), np.uint8), np.zeros((h, w), np.uint8)))
            continue
        I0, I1 = synth.make_pair(h, w, seed=seed + 13 * k, dx=0.4 + 0.9 * (k % 4), dy=-1.1 + 0.5 * (k % 3),
                                 margin=min(32, h // 4, w // 4))
        if kind == 2:
            I1 = I0.copy()
        elif kind == 4:
            I0, I1 = I0.copy(), I1.copy()
            I0[: h // 4] = 0
            I1[:, w // 3: w // 3 + max(w // 6, 1)] = 0
        out.append((I0, I1))
    return out


def singles(s, pairs):
    res = []
    for I0, I1 in pairs:
        u, v = s.calc(I0, I1)
        res.append((u, v, s.stats.iters_array(), s.stats.outer_array()))
    return res


def assert_batch_matches(s, pairs, want=None):
    got = s.calc_batch([p[0] for p in pairs], [p[1] for p in pairs])
    stats = s.batch_stats
    want = want if want is not None else singles(s, pairs)
    assert len(got) == len(pairs) == len(stats)
    for k, ((u, v), (wu, wv, wit, wout)) in enumerate(zip(got, want)):
        assert np.array_equal(u, wu) and np.array_equal(v, wv), "pair %d: flow differs from tvl1_calc_u8" % k
        assert np.array_equal(stats[k].iters_array(), wit), "pair %d: iteration counts differ" % k
        assert np.array_equal(stats[k].outer_array(), wout), "pair %d: outer iteration counts differ" % k
    return got, stats


def test_mixed_stops_against_single_and_oracle(gpu, orc):
    kw = dict(lambda_=0.15, nscales=5)
    pairs = mixed_pairs(96, 128, 7)
    s = N.Solver(N.default_params(**kw))
    got, stats = assert_batch_matches(s, pairs)
    totals = {st.total_iterations for st in stats}
    assert len(totals) >= 3, "the pairs were meant to stop at different counts: %s" % totals
    for k, (I0, I1) in enumerate(pairs):
        ou, ov, oit, lev = orc.tvl1_calc(I0, I1, lambda_=0.15, nscales=5)
        assert stats[k].levels == lev
        assert np.array_equal(stats[k].iters_array(), oit[:lev])
        assert np.array_equal(got[k][0], ou) and np.array_equal(got[k][1], ov), "pair %d differs from the oracle" % k
    assert stats[0].launches > 0 and all(st.launches == stats[0].launches for st in stats)
    assert all(st.ms_total == stats[0].ms_total > 0 for st in stats)
    s.close()


@pytest.mark.parametrize("n", [1, 2, 7, 33])
def test_batch_sizes(gpu, n):
    s = N.Solver(N.default_params(nscales=4))
    assert_batch_matches(s, mixed_pairs(48, 72, n, seed=n))
    s.close()


@pytest.mark.parametrize("hw", [(37, 101), (50, 203), (61, 130), (33, 259)])
def test_odd_widths(gpu, orc, hw):
    h, w = hw
    pairs = mixed_pairs(h, w, 5, seed=w)
    s = N.Solver(N.default_params(lambda_=0.15, nscales=6))
    got, stats = assert_batch_matches(s, pairs)
    I0, I1 = pairs[0]
    ou, ov, oit, lev = orc.tvl1_calc(I0, I1, lambda_=0.15, nscales=6)
    assert np.array_equal(got[0][0], ou) and np.array_equal(got[0][1], ov)
    s.close()


def test_roi_strip(gpu):
    """the production shape: 100-row strips of 4096 px, wrapper defaults"""
    s = N.Solver(N.default_params())
    assert_batch_matches(s, mixed_pairs(100, 4096, 3, seed=5))
    s.close()


def test_level_stop_rule(gpu, orc):
    """sizes whose pyramid ends early (a level under 16 px is built then dropped)"""
    pairs = mixed_pairs(40, 300, 4, seed=2)
    s = N.Solver(N.default_params())
    got, stats = assert_batch_matches(s, pairs)
    assert stats[0].levels == len(N.pyramid_sizes(300, 40, 10, 0.8)) < 10
    ou, ov, _, _ = orc.tvl1_calc(*pairs[1], lambda_=0.05, nscales=10)   # the wrapper defaults
    assert np.array_equal(got[1][0], ou) and np.array_equal(got[1][1], ov)
    s.close()


@pytest.mark.parametrize("kw", [
    dict(median_filtering=1), dict(median_filtering=3), dict(scale_step=0.5), dict(nscales=1), dict(warps=1),
    dict(inner_iterations=7, outer_iterations=3), dict(inner_iterations=1, outer_iterations=4), dict(epsilon=0.0),
])
def test_parameters(gpu, kw):
    s = N.Solver(N.default_params(**dict(dict(lambda_=0.15, nscales=5), **kw)))
    assert_batch_matches(s, mixed_pairs(57, 83, 5, seed=3))
    s.close()


def upload_pitched(img, pitch):
    return N.upload_u8(img, pitch, 255)[0]


def test_pitched_io_repeated_pointers_and_poisoned_padding(gpu):
    h, w = 45, 77
    pairs = mixed_pairs(h, w, 4, seed=9)
    s = N.Solver(N.default_params(lambda_=0.15, nscales=5))
    want = singles(s, pairs)
    p0, p1, po = 96, 128, 100 * 4   # byte pitches: frames padded with 255, flow rows with NaN
    f0 = [upload_pitched(I0, p0) for I0, _ in pairs]
    f1 = [upload_pitched(I1, p1) for _, I1 in pairs]
    order = [0, 1, 2, 3, 1, 1]      # entries 4 and 5 repeat pair 1's frames
    outs = [N.DevBuf(h * po, 0).upload(np.full((h, po // 4), np.nan, np.float32)) for _ in range(2 * len(order))]
    s.calc_batch_device([f0[k].ptr for k in order], p0, [f1[k].ptr for k in order], p1, w, h,
                        [o.ptr for o in outs[0::2]], [o.ptr for o in outs[1::2]], po)
    for j, k in enumerate(order):
        u = outs[2 * j].download((h, po // 4), np.float32)
        v = outs[2 * j + 1].download((h, po // 4), np.float32)
        assert np.isnan(u[:, w:]).all() and np.isnan(v[:, w:]).all(), "the output padding was written"
        assert np.array_equal(u[:, :w], want[k][0]) and np.array_equal(v[:, :w], want[k][1]), "entry %d" % j
        assert np.array_equal(s.batch_stats[j].iters_array(), want[k][2])
    for b in f0 + f1 + outs:
        b.free()
    s.close()


def test_deterministic_and_interleaved_with_single(gpu):
    pairs = mixed_pairs(64, 96, 6, seed=4)
    s = N.Solver(N.default_params(lambda_=0.15, nscales=5))
    before = singles(s, pairs)            # tvl1_calc_u8 before any batch
    a = s.calc_batch([p[0] for p in pairs], [p[1] for p in pairs])
    after = singles(s, pairs)             # ... and after one, on the same handle
    b = s.calc_batch([p[0] for p in pairs], [p[1] for p in pairs])
    for k in range(len(pairs)):
        for x, y in ((a[k][0], b[k][0]), (a[k][1], b[k][1]), (a[k][0], before[k][0]), (a[k][1], before[k][1]),
                     (before[k][0], after[k][0]), (before[k][1], after[k][1])):
            assert np.array_equal(x, y)
    # a batch of another size and count in between, then the first again
    s.calc_batch([p[0][:40, :50] for p in pairs[:3]], [p[1][:40, :50] for p in pairs[:3]])
    c = s.calc_batch([p[0] for p in pairs], [p[1] for p in pairs])
    assert all(np.array_equal(a[k][0], c[k][0]) and np.array_equal(a[k][1], c[k][1]) for k in range(len(pairs)))
    s.close()


def test_api_solve_batch(gpu):
    pairs = mixed_pairs(50, 70, 3, seed=6)
    tv = api.generate_TV_args({}, {"lambda": 0.15, "nscales": 4})
    got = api.TVL1_solve_batch([p[0] for p in pairs], [p[1] for p in pairs], tv)
    for (u, v), (I0, I1) in zip(got, pairs):
        wu, wv = api.TVL1_solve(I0, I1, tv)
        assert np.array_equal(u, wu) and np.array_equal(v, wv)


def test_readbacks_cover_the_batch(gpu):
    pairs = mixed_pairs(64, 96, 8, seed=8)
    s = N.Solver(N.default_params(lambda_=0.15, nscales=5))
    s.calc_batch([p[0] for p in pairs], [p[1] for p in pairs])
    rb = s.last_readbacks()
    st = s.batch_stats[0]
    assert rb > st.levels * st.warps   # at least one per (level, warp), plus the final one
    single = 0
    for I0, I1 in pairs:
        s.calc(I0, I1)
        single += s.last_readbacks()
    assert rb < single                 # one read-back per chunk covers every pair
    s.close()


# ---- refusals

def raw_call(s, n, f0, p0, f1, p1, w, h, u, v, po):
    arr = lambda xs: (C.c_void_p * max(len(xs), 1))(*xs)
    return N.lib().tvl1_calc_batch_u8(s.handle, n, arr(f0), p0, arr(f1), p1, w, h, arr(u), arr(v), po, None, None)


def last_error():
    return N.lib().tvl1_last_error().decode()


def test_refusals(gpu):
    h, w = 24, 40
    bufs = [N.DevBuf(h * 64 * 4, 0).zero() for _ in range(4)]
    f, g, u, v = (b.ptr for b in bufs)
    s = N.Solver(N.default_params(nscales=3))
    ok = raw_call(s, 2, [f, f], 64, [g, g], 64, w, h, [u, u], [v, v], 64 * 4)
    assert ok == 0, last_error()
    assert raw_call(s, 0, [], 64, [], 64, w, h, [], [], 64 * 4) == -1 and "n must be" in last_error()
    assert raw_call(s, 2, [f, None], 64, [g, g], 64, w, h, [u, u], [v, v], 64 * 4) == -1 and "entry 1" in last_error()
    assert raw_call(s, 2, [f, f], 64, [g, g], 64, w, h, [u, u], [v, None], 64 * 4) == -1 and "entry 1" in last_error()
    assert raw_call(s, 1, [f], 39, [g], 64, w, h, [u], [v], 64 * 4) == -1 and "pitch" in last_error()
    assert raw_call(s, 1, [f], 64, [g], 64, w, h, [u], [v], 39 * 4) == -1 and "pitch" in last_error()
    assert raw_call(s, 1, [f], 64, [g], 64, 0, h, [u], [v], 64 * 4) == -1 and "empty" in last_error()
    for kw, text in ((dict(gamma=0.5), "gamma"), (dict(semantics=N.SEMANTICS_CUDA), "cuda semantics")):
        t = N.Solver(N.default_params(nscales=3, **kw))
        assert raw_call(t, 1, [f], 64, [g], 64, w, h, [u], [v], 64 * 4) == -3 and text in last_error()
        t.close()
    # a batch whose state does not fit on the device: nothing of it stays allocated and the handle keeps working
    big = 8192
    fb = N.DevBuf(big * big, 0).zero()
    ub = N.DevBuf(big * big * 4, 0)
    n = 64   # ~4 GB of state per 8192^2 pair
    rc = raw_call(s, n, [fb.ptr] * n, big, [fb.ptr] * n, big, big, big, [ub.ptr] * n, [ub.ptr] * n, big * 4)
    assert rc == -4 and "batch" in last_error()
    assert raw_call(s, 2, [f, f], 64, [g, g], 64, w, h, [u, u], [v, v], 64 * 4) == 0, last_error()
    I0, I1 = synth.make_pair(h, w, seed=1, margin=6)
    u1, v1 = s.calc(I0, I1)
    (u2, v2), = s.calc_batch([I0], [I1])
    assert np.array_equal(u1, u2) and np.array_equal(v1, v2)
    for b in bufs + [fb, ub]:
        b.free()
    s.close()
