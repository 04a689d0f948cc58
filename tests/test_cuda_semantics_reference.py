"""The cv::cuda-semantics mode (TVL1_SEMANTICS_CUDA) on the CPU: its C restatement (oracle/tvl1_oracle_cuda.c)
against the independent NumPy one (oracle/cuda_np.py), properties of its resize and warp that do not rest on
anyone's memory of OpenCV, its whole-pair loop, and the job keys that select it."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth
from oracle import cuda_np as CN
from oracle import oracle_cuda as OC


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same(a, b):
    return np.array_equal(bits(a), bits(b))


def planes(rng, h, w, amp, integer=False):
    I0 = (rng.random((h, w), dtype=np.float32) * 255).astype(np.float32)
    I1 = (rng.random((h, w), dtype=np.float32) * 255).astype(np.float32)
    u1 = (rng.standard_normal((h, w)) * amp).astype(np.float32)
    u2 = (rng.standard_normal((h, w)) * amp).astype(np.float32)
    if integer:
        u1, u2 = np.round(u1).astype(np.float32), np.round(u2).astype(np.float32)
    return I0, I1, u1, u2


@pytest.mark.parametrize("seed", range(12))
def test_warp_c_equals_numpy(seed):
    rng = np.random.default_rng(100 + seed)
    h, w = (int(x) for x in rng.integers(3, 97, 2))
    amp = [0.3, 2.0, 8.0, 40.0][seed % 4]
    I0, I1, u1, u2 = planes(rng, h, w, amp, integer=seed % 3 == 0)
    if seed % 5 == 1:   # whole windows outside the image, on every side
        u1[: h // 2] += 3 * w
        u2[:, : w // 2] -= 3 * h
    got = OC.warp_cuda(I0, I1, u1, u2)
    want = CN.warp_cuda(I0, I1, u1, u2)
    for g, x in zip(got, want):
        assert same(g, x)


@pytest.mark.parametrize("seed", range(10))
def test_resize_c_equals_numpy(seed):
    rng = np.random.default_rng(200 + seed)
    sh, sw = (int(x) for x in rng.integers(2, 140, 2))
    src = (rng.standard_normal((sh, sw)) * 50).astype(np.float32)
    for f in (0.8, 0.5, 0.7):
        if int(np.rint(sw * f)) > 0 and int(np.rint(sh * f)) > 0:
            assert same(OC.resize_cuda(src, inv_scale=f), CN.resize_cuda(src, inv_scale=f))
    dw, dh = int(rng.integers(sw, 2 * sw + 3)), int(rng.integers(sh, 2 * sh + 3))
    assert same(OC.resize_cuda(src, dw, dh), CN.resize_cuda(src, dw, dh))


def test_integer_flow_reproduces_clamped_samples():
    rng = np.random.default_rng(3)
    h, w = 37, 53
    I0, I1, u1, u2 = planes(rng, h, w, 30.0, integer=True)
    iw, iwx, iwy, _, _ = OC.warp_cuda(I0, I1, u1, u2)
    ys, xs = np.mgrid[0:h, 0:w]
    sx = np.clip(xs + u1.astype(np.int64), 0, w - 1)
    sy = np.clip(ys + u2.astype(np.int64), 0, h - 1)
    P = np.pad(I1, 1, mode="edge")
    I1x = np.float32(0.5) * (P[1:-1, 2:] - P[1:-1, :-2])
    I1y = np.float32(0.5) * (P[2:, 1:-1] - P[:-2, 1:-1])
    assert np.array_equal(iw, I1[sy, sx])
    assert np.array_equal(iwx, I1x[sy, sx]) and np.array_equal(iwy, I1y[sy, sx])


@pytest.mark.parametrize("grid", [4, 0])
def test_linear_ramp_is_reproduced_inside(grid):
    """The A = -0.5 cubic reproduces linear functions: a ramp sampled where the whole window lies in the image.
    At quarter-pixel positions the weights are short dyadic fractions: within 2 ulp.  At arbitrary positions the fp32
    sums of 16 rounded products (and the normalisation) stay within 8 ulp (6 measured)."""
    h, w = 64, 80
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    I1 = (np.float32(0.75) * xs + np.float32(0.5) * ys + np.float32(100)).astype(np.float32)
    rng = np.random.default_rng(5)
    u1 = rng.uniform(-3, 3, (h, w)).astype(np.float32)
    u2 = rng.uniform(-3, 3, (h, w)).astype(np.float32)
    if grid:
        u1, u2 = (np.round(u1 * grid) / grid).astype(np.float32), (np.round(u2 * grid) / grid).astype(np.float32)
    iw, _, _, _, _ = OC.warp_cuda(np.zeros_like(I1), I1, u1, u2)
    wx, wy = xs + u1, ys + u2
    inside = (wx >= 3) & (wx <= w - 4) & (wy >= 3) & (wy <= h - 4)
    want = (0.75 * wx.astype(np.float64) + 0.5 * wy.astype(np.float64) + 100).astype(np.float32)
    ulp = np.abs(bits(iw[inside]).astype(np.int64) - bits(want[inside]).astype(np.int64))
    assert inside.sum() > 1000 and ulp.max() <= (2 if grid else 8)


def test_resize_properties():
    rng = np.random.default_rng(6)
    for sh, sw in ((17, 23), (64, 48), (5, 131)):
        c = np.full((sh, sw), np.float32(37.3), np.float32)
        for out in (OC.resize_cuda(c, inv_scale=0.8), OC.resize_cuda(c, 2 * sw + 1, 3 * sh)):
            ulp = np.abs(bits(out).astype(np.int64) - bits(c[0, 0]).astype(np.int64))
            assert ulp.max() <= 2
        src = rng.standard_normal((sh, sw)).astype(np.float32)
        for out in (OC.resize_cuda(src, inv_scale=0.5), OC.resize_cuda(src, 3 * sw, 2 * sh)):
            assert out[0, 0] == src[0, 0]


def test_whole_pair_loop():
    I0, I1 = synth.make_pair(72, 88, seed=3)
    for N, eps in ((300, 0.01), (41, 0.01), (7, 0.01), (12, 0.0)):
        u, v, it, lev = OC.tvl1_calc_cuda(I0, I1, iterations=N, epsilon=eps, nscales=4, warps=3, **{"lambda": 0.05})
        u2, v2, it2, _ = OC.tvl1_calc_cuda(I0, I1, iterations=N, epsilon=eps, nscales=4, warps=3, **{"lambda": 0.05})
        assert same(u, u2) and same(v, v2) and np.array_equal(it, it2)
        it = it[:lev]
        assert ((it == N) | (it % 2 == 0)).all() and (it > 0).all(), it
        if eps == 0.0:
            assert (it == N).all()
        assert np.isfinite(u).all() and np.isfinite(v).all()


def test_tv_args_semantics(native):
    from fibsem_optflow_b200 import api
    tv = api.generate_TV_args({}, {"semantics": "cuda", "iterations": 51})
    assert tv["semantics"] == "cuda"
    p = api.params_from_TV_args(tv)
    assert p.semantics == native.SEMANTICS_CUDA and p.iterations == 51 and p.median_filtering == 1
    tv = api.generate_TV_args({"semantics": "cpu"}, {"semantics": "cuda"})   # the pair's value wins
    assert tv["semantics"] == "cpu" and api.params_from_TV_args(tv).semantics == native.SEMANTICS_CPU
    assert "semantics" not in api.generate_TV_args({}, {})
    assert api.params_from_TV_args(api.generate_TV_args({}, {})).semantics == native.SEMANTICS_CPU
    assert native.default_params(semantics="cuda").semantics == native.SEMANTICS_CUDA
    for bad in ("CUDA", "gpu", 1, ""):
        with pytest.raises(ValueError):
            api.generate_TV_args({"semantics": bad}, {})
    for key in ("innerIterations", "outerIterations", "medianFiltering"):
        with pytest.raises(ValueError):
            api.generate_TV_args({"semantics": "cuda"}, {key: 3})
        with pytest.raises(ValueError):
            api.params_from_TV_args(dict(api.generate_TV_args({}, {key: 3}), semantics="cuda"))
