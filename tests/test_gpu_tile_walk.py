"""The tile-walking kernels at stage level, bit for bit against the oracle, where the smaller stage tests of
test_gpu_kernels.py do not reach:
  * grids of at least three tiles per resident block (sized from the device's SM count), so that every block of
    k_warp / k_median5 runs its look-ahead loads, swaps its double buffers and flips its mbarrier phases across
    TMA, scalar-copy and global-load tiles, and exits after its last tile;
  * flows steered per tile onto every path and window limit of k_warp and k_warp_cuda (tests/tilefields.py,
    whose coverage tests/test_tilefields.py checks on the CPU);
  * non-32 pitches with NaN in every pad column, NaN rows past the image and NaN-prefilled outputs: an
    in-image output must equal the oracle, and nothing outside the kernel's write width (pinned below, and in
    include/tvl1_b200.h) may change.
The iteration kernels (k_iterate, k_iterate_fused2, k_outer) get the same padding at widths around their
124- / 120-px strips and at a size the grid cannot cover in one round."""
import ctypes as C

import numpy as np
import pytest

import tilefields as T
from test_gpu_kernels import make_iter_inputs

pytestmark = pytest.mark.gpu


def sm_count(device=0):
    """multiprocessors of the device (CUDA driver API)"""
    cu = C.CDLL("libcuda.so.1")
    assert cu.cuInit(0) == 0
    d, n = C.c_int(0), C.c_int(0)
    assert cu.cuDeviceGet(C.byref(d), device) == 0
    assert cu.cuDeviceGetAttribute(C.byref(n), 16, d) == 0   # CU_DEVICE_ATTRIBUTE_MULTIPROCESSOR_COUNT
    return n.value


@pytest.fixture(scope="module")
def sizes(gpu):
    return T.grid_sizes(sm_count())


def pitches(w):
    """row pitches (elements) of the poisoned runs: the width rounded up to 4 -- no padding at all when w is a
    multiple of 4 -- and 8 more (neither a multiple of 32 unless by chance)"""
    p = T.roundup(w, 4)
    return [p, p + 8]


def check_poisoned(got, want, h, w, write_w, name):
    """got: a full (h + POISON_ROWS, pitch) output buffer that was NaN before the call"""
    assert got.shape[0] > h
    img = got[:h, :w]
    bad = np.argwhere(~((img == want) | (np.isnan(img) & np.isnan(want))))
    assert bad.size == 0, "%s: %d pixels differ from the oracle, first (y, x) %s: %r vs %r" % (
        name, len(bad), tuple(bad[0]), img[tuple(bad[0])], want[tuple(bad[0])])
    assert np.isnan(got[:h, write_w:]).all(), "%s wrote pad columns at or past x = %d" % (name, write_w)
    assert np.isnan(got[h:]).all(), "%s wrote rows past h = %d" % (name, h)


# ---------------------------------------------------------------- k_warp


WARP_NAMES = ["I1w", "I1wx", "I1wy", "grad", "rho_c"]


def run_warp(gpu, orc, h, w, u1, u2, seed, pitch):
    rng = np.random.default_rng(seed)
    I0 = (rng.random((h, w)) * 255).astype(np.float32)
    I1 = (rng.random((h, w)) * 255).astype(np.float32)
    I1x, I1y = orc.centered_gradient(I1)
    want = orc.warp(I0, I1, I1x, I1y, u1, u2)
    got = gpu.k_warp(I0, I1, u1, u2, pitch=pitch, poison=True, full=True)
    for g, o, n in zip(got, want, WARP_NAMES):
        check_poisoned(g, o, h, w, w, "k_warp %dx%d pitch %d %s" % (h, w, pitch, n))   # k_warp writes x < w


def test_warp_multi_tile(gpu, orc, sizes):
    """every block walks >= 3 tiles of every regime (tilefields.warp_field) in random order"""
    h, w = sizes["warp"]
    u1, u2 = T.warp_field(h, w, T.SEED)
    run_warp(gpu, orc, h, w, u1, u2, 1, T.roundup(w, 4))


@pytest.mark.parametrize("h,w", T.WARP_SMALL)
def test_warp_small(gpu, orc, h, w):
    for s in range(3):
        u1, u2 = T.warp_field(h, w, T.SEED + s)
        run_warp(gpu, orc, h, w, u1, u2, s, pitches(w)[s % 2])


def test_warp_regime_runs(gpu, orc, sizes):
    """long runs of one window limit at a time: a block's consecutive tiles all take the 17-row (32-row box),
    the 16-row, the 88-wide or the global-load path, and runs of tiles that are wholly outside"""
    h, w = sizes["warp"]
    h = min(h, 600)
    for k, regs in enumerate([[T.RH17], [T.RH16, T.RH17], [T.RW88, T.RW89], [T.FAR, T.SMOOTH], [T.EDGE_R, T.EDGE_B]]):
        u1, u2 = T.warp_field(h, w, T.SEED + 100 + k, regimes=regs)
        run_warp(gpu, orc, h, w, u1, u2, k, pitches(w)[k % 2])


# ---------------------------------------------------------------- k_warp_cuda


def run_warp_cuda(gpu, h, w, u1, u2, seed, pitch):
    from oracle import oracle_cuda as OC
    rng = np.random.default_rng(seed)
    I0 = (rng.random((h, w)) * 255).astype(np.float32)
    I1 = (rng.random((h, w)) * 255).astype(np.float32)
    want = OC.warp_cuda(I0, I1, u1, u2)
    got = gpu.k_warp_cuda(I0, I1, u1, u2, pitch=pitch, poison=True, full=True)
    for g, o, n in zip(got, want, WARP_NAMES):
        check_poisoned(g, o, h, w, w, "k_warp_cuda %dx%d pitch %d %s" % (h, w, pitch, n))   # writes x < w


def test_warp_cuda_multi_tile(gpu, sizes):
    h, w = sizes["warp_cuda"]
    u1, u2 = T.warp_cuda_field(h, w, T.SEED)
    run_warp_cuda(gpu, h, w, u1, u2, 2, T.roundup(w, 4))


@pytest.mark.parametrize("h,w", T.WARP_CUDA_SMALL)
def test_warp_cuda_small(gpu, h, w):
    for k, p in enumerate(pitches(w) + [w]):   # k_warp_cuda takes any pitch >= w
        u1, u2 = T.warp_cuda_field(h, w, T.SEED + k)
        run_warp_cuda(gpu, h, w, u1, u2, k, p)


# ---------------------------------------------------------------- medians


def median_input(h, w, seed):
    rng = np.random.default_rng(seed)
    src = (rng.standard_normal((h, w)) * 3).astype(np.float32)
    src[rng.random((h, w)) < 0.1] = 1.5   # ties
    return src


def run_median(gpu, orc, k, h, w, pitch, seed):
    src = median_input(h, w, seed)
    if k == 5:
        got = gpu.k_median5(src, pitch=pitch, poison=True, full=True)
        # k_median5 stores 4 outputs at a time: it writes up to the width rounded up to 4
        check_poisoned(got, orc.median5(src), h, w, T.roundup(w, 4), "k_median5 %dx%d pitch %d" % (h, w, pitch))
    else:
        got = gpu.k_median3(src, pitch=pitch, poison=True, full=True)
        check_poisoned(got, orc.median3(src), h, w, w, "k_median3 %dx%d pitch %d" % (h, w, pitch))   # x < w


@pytest.mark.parametrize("k", [5, 3])
def test_median_multi_tile(gpu, orc, sizes, k):
    """>= 3 k_median5 tiles per resident block; h = 1 (mod 16) with w >= 260, so one tile row sits exactly at
    y0 + 17 == h, one row short of the TMA interior"""
    h, w = sizes["median5"]
    run_median(gpu, orc, k, h, w, T.roundup(w, 4), 3)


@pytest.mark.parametrize("k", [5, 3])
@pytest.mark.parametrize("h,w", T.MEDIAN_SIZES)
def test_median_small(gpu, orc, k, h, w):
    for j, p in enumerate(pitches(w)):
        run_median(gpu, orc, k, h, w, p, j)


# ---------------------------------------------------------------- iteration kernels

ITER_WIDTHS = [119, 120, 121, 123, 124, 125, 239, 240, 241, 244, 247, 248, 249, 1001, 1003]
L_T, THETA, TAUT = np.float32(0.15 * 0.3), np.float32(0.3), np.float32(0.25 / 0.3)
STATE = ["u1", "u2", "p11", "p12", "p21", "p22"]


def oracle_iterations(orc, consts, state, ns):
    """the oracle's states after each n in ns (ascending) and the per-iteration errors"""
    cur = [s.copy() for s in state]
    errs, out = [], {}
    for i in range(1, max(ns) + 1):
        errs.append(orc.iterate(*consts, *cur, L_T, THETA, TAUT))
        if i in ns:
            out[i] = [s.copy() for s in cur]
    return out, errs


def run_iterate(gpu, consts, state, want, werr, n, fused, h, w, pitch):
    got = gpu.k_iterate(*consts, *state, L_T, THETA, TAUT, n=n, fused=fused, pitch=pitch, poison=True, full=True)
    name = "%s n=%d %dx%d pitch %d" % ({False: "k_iterate", True: "k_iterate_fused2", "outer": "k_outer"}[fused],
                                         n, h, w, pitch)
    # the iteration kernels store 4 pixels at a time: they write up to the width rounded up to 4
    for k in range(6):
        check_poisoned(got[k], want[k], h, w, T.roundup(w, 4), name + " " + STATE[k])
    np.testing.assert_allclose(got[6], werr[:n], rtol=1e-12, err_msg=name)


@pytest.mark.parametrize("w", ITER_WIDTHS)
def test_iterate_strip_widths(gpu, orc, w):
    """widths around the 124-px strip of k_iterate and the 120-px strip of the two-iteration passes, NaN
    padding; an odd count for k_iterate and k_outer (the single pass, and the stage's copy back)"""
    h = 37 if w < 1000 else 70
    rng = np.random.default_rng(w)
    consts, state = make_iter_inputs(rng, h, w)
    want, werr = oracle_iterations(orc, consts, state, [3, 4])
    for j, p in enumerate(pitches(w)):
        run_iterate(gpu, consts, state, want[3], werr, 3, False, h, w, p)
        run_iterate(gpu, consts, state, want[4], werr, 4, True, h, w, p)
        run_iterate(gpu, consts, state, want[3 + j], werr, 3 + j, "outer", h, w, p)


def test_iterate_more_tiles_than_warps(gpu, orc):
    """a size whose tiles outnumber the resident warps at any tile height the launch may choose (64 rows of
    124 px per tile at most, 5 blocks of 4 warps per SM at most for k_iterate, 3 for the two-iteration
    kernels), so that every warp walks several tiles"""
    sms = sm_count()
    w = 4001
    h = 64 * (T.cdiv(sms * 5 * 4, T.cdiv(w, 124)) + 1) + 13
    rng = np.random.default_rng(9)
    consts, state = make_iter_inputs(rng, h, w)
    want, werr = oracle_iterations(orc, consts, state, [2, 3])
    p = T.roundup(w, 4)
    run_iterate(gpu, consts, state, want[2], werr, 2, False, h, w, p)
    run_iterate(gpu, consts, state, want[2], werr, 2, True, h, w, p)
    run_iterate(gpu, consts, state, want[3], werr, 3, "outer", h, w, p)
