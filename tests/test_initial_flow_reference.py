"""fp32 frames and an initial flow in the CPU restatements (oracle_ex/): the C solve against the cv2 composition,
the multiply of the initial flow's pyramid against cv2.multiply, cv::cuda's downscale against its NumPy
restatement, and the zero / u8-equivalent cases against the existing oracle entry points.  No GPU needed."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from fibsem_optflow_b200 import synth  # noqa: E402


@pytest.fixture(scope="module")
def ox():
    from oracle_ex import oracle_ex
    oracle_ex.lib()
    return oracle_ex


@pytest.fixture
def cv2_plain():
    cv2.setUseOptimized(False)
    yield cv2
    cv2.setUseOptimized(True)


def f32_pair(h, w, seed):
    """a pair of fp32 frames in [0, 1] that are not multiples of 1/255 (16-bit data, normalised)"""
    I0, I1 = synth.make_pair(h, w, seed=seed)
    rng = np.random.default_rng(seed)
    f = lambda a: ((a.astype(np.float32) * 257 + rng.integers(0, 257, a.shape)) / np.float32(65535)).astype(np.float32)
    return f(I0), f(I1)


def init_flow(kind, h, w, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "smooth":
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        u = (-1.3 + 0.6 * np.sin(xx / 17.0) + 0.002 * yy).astype(np.float32)
        v = (0.7 + 0.4 * np.cos(yy / 11.0)).astype(np.float32)
        return u, v
    if kind == "rough":
        return (rng.standard_normal((h, w)) * 3).astype(np.float32), (rng.standard_normal((h, w)) * 3).astype(np.float32)
    raise KeyError(kind)


CASES = [
    # (h, w, frames, init, kw)
    (96, 128, "u8", "smooth", {}),
    (96, 128, "f32", "rough", {}),
    (97, 127, "f32", "smooth", {"scale_step": 0.5, "nscales": 4}),
    (96, 128, "u8", "rough", {"scale_step": 0.5, "nscales": 10}),       # stops at the < 16 px level
    (95, 129, "f32", "smooth", {"gamma": 0.1, "nscales": 3}),
    (96, 128, "u8", "rough", {"gamma": 0.1, "scale_step": 0.5, "nscales": 3}),
    (96, 128, "f32", "smooth", {"nscales": 12}),                        # 0.8: stops at the < 16 px level
]


@pytest.mark.parametrize("h,w,frames,init,kw", CASES)
def test_ex_vs_cv2_composition(ox, cv2_plain, h, w, frames, init, kw):
    """the C restatement's calc(I0, I1, flow) equals the composition with real cv2: flows and iteration counts"""
    from oracle_ex import ref_ex
    I0, I1 = f32_pair(h, w, seed=h + w) if frames == "f32" else synth.make_pair(h, w, seed=h + w)
    fl = init_flow(init, h, w, seed=w)
    u, v, it, lev = ox.tvl1_calc_ex(I0, I1, fl, **kw)
    ru, rv, rit = ref_ex.tvl1_calc_ex(I0, I1, fl, **{("lambda_" if k == "lambda" else k): x for k, x in kw.items()})
    assert lev == rit.shape[0] and np.array_equal(it[:lev], rit)
    assert np.array_equal(u, ru) and np.array_equal(v, rv)
    assert not np.array_equal(u, ox.tvl1_calc_ex(I0, I1, None, **kw)[0])   # the initial flow was used


@pytest.mark.parametrize("step", [0.8, 0.5, 0.7, 0.93])
def test_flow_multiply_is_cv2_multiply(ox, cv2_plain, step):
    """The multiply of the initial flow's pyramid (CPU class) is cv::multiply by a double Scalar: RN_f32(x * step) in
    fp64, the form the engine's k_resize / k_resize_half use (apply_mul 2), not x * (float)step."""
    rng = np.random.default_rng(int(step * 100))
    x = (rng.standard_normal((211, 317)) * rng.choice([1e-3, 1.0, 40.0, 1e4], (211, 317))).astype(np.float32)
    want = cv2.multiply(x, step)
    engine_form = (x.astype(np.float64) * step).astype(np.float32)
    assert np.array_equal(engine_form, want)
    if step in (0.8, 0.7, 0.93):   # not a power of two: the fp32 form differs on many values, so the check has teeth
        assert (x * np.float32(step) != want).sum() > 1000
    # one level of the C restatement's flow pyramid equals cv2.resize + cv2.multiply
    from oracle_ex import ref_ex
    for h, w in [(96, 128), (77, 61), (20, 33)]:
        u = (rng.standard_normal((h, w)) * 5).astype(np.float32)
        assert np.array_equal(ox.flow_down(u, step), ref_ex.flow_down(u, step)), (h, w)


def test_flow_down_cuda_vs_numpy(ox):
    """cv::cuda's step of the initial flow's pyramid: C restatement against oracle/cuda_np.py's resize times the
    float scalar"""
    from oracle_ex import ref_ex
    rng = np.random.default_rng(3)
    for _ in range(60):
        h, w = int(rng.integers(16, 140)), int(rng.integers(16, 140))
        step = float(rng.choice([0.8, 0.5, 0.75, 0.6]))
        u = (rng.standard_normal((h, w)) * rng.choice([0.5, 8.0, 3e3])).astype(np.float32)
        assert np.array_equal(ox.flow_down(u, step, cuda=True), ref_ex.flow_down_cuda(u, step)), (h, w, step)


def test_convert_f32(ox):
    """level 0 of an fp32 frame: the C restatement's fp64 form equals x * 255.0f"""
    from oracle_ex import ref_ex
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.random(5000), rng.standard_normal(5000) * 1e6, [0.0, -0.0, 1.0, 1e-40, 3e38]]).astype(np.float32)
    x = x.reshape(1, -1)
    assert np.array_equal(ox.convert_f32(x), ref_ex.level0(x))
    k = np.arange(256, dtype=np.float32)
    assert np.array_equal(ref_ex.level0((k / np.float32(255)).astype(np.float32)), k)   # k/255 * 255 rounds back to k


@pytest.mark.parametrize("kw", [{}, {"scale_step": 0.5, "nscales": 4}, {"gamma": 0.1, "nscales": 3}])
def test_zero_init_and_u8_equivalent_f32_reproduce_calc(ox, kw):
    """a zero initial flow, no initial flow and fp32 frames holding k/255 all give the existing entry point's
    result bit for bit"""
    from oracle import oracle as O
    I0, I1 = synth.make_pair(96, 128, seed=4)
    u, v, it, lev = O.tvl1_calc(I0, I1, **kw)
    z = np.zeros(I0.shape, np.float32)
    f0, f1 = (I0 / np.float32(255)).astype(np.float32), (I1 / np.float32(255)).astype(np.float32)
    for args in ((I0, I1, None), (I0, I1, (z, z)), (f0, f1, None), (f0, f1, (z, z))):
        gu, gv, git, glev = ox.tvl1_calc_ex(*args, **kw)
        assert glev == lev and np.array_equal(git, it) and np.array_equal(gu, u) and np.array_equal(gv, v)


@pytest.mark.parametrize("kw", [{}, {"scale_step": 0.5, "nscales": 4}])
def test_zero_init_and_u8_equivalent_f32_reproduce_calc_cuda(ox, kw):
    from oracle import oracle_cuda as OC
    I0, I1 = synth.make_pair(96, 128, seed=6)
    u, v, it, lev = OC.tvl1_calc_cuda(I0, I1, iterations=40, **kw)
    z = np.zeros(I0.shape, np.float32)
    f0, f1 = (I0 / np.float32(255)).astype(np.float32), (I1 / np.float32(255)).astype(np.float32)
    for args in ((I0, I1, None), (I0, I1, (z, z)), (f0, f1, None), (f0, f1, (z, z))):
        gu, gv, git, glev = ox.tvl1_calc_cuda_ex(*args, iterations=40, **kw)
        assert glev == lev and np.array_equal(git, it) and np.array_equal(gu, u) and np.array_equal(gv, v)


def test_cuda_ex_uses_initial_flow(ox):
    """cuda mode: the coarsest level starts from the downscaled initial flow (the result differs from a zero start
    and, started from the true flow, lands closer to it)"""
    h, w = 96, 128
    I0, I1 = synth.make_pair(h, w, seed=9)
    tu, tv = synth.true_flow(h, w)
    u0, v0, _, _ = ox.tvl1_calc_cuda_ex(I0, I1, None, iterations=20)
    u1, v1, _, _ = ox.tvl1_calc_cuda_ex(I0, I1, (tu, tv), iterations=20)
    sl = (slice(8, -8), slice(8, -8))
    e0 = np.hypot(u0 - tu, v0 - tv)[sl].mean()
    e1 = np.hypot(u1 - tu, v1 - tv)[sl].mean()
    assert not np.array_equal(u0, u1) and e1 <= e0


def test_bad_arguments(ox):
    I0, I1 = synth.make_pair(40, 40, seed=1)
    with pytest.raises(ValueError):
        ox.tvl1_calc_ex(I0.astype(np.uint16), I1.astype(np.uint16))
    with pytest.raises(ValueError):
        ox.tvl1_calc_ex(I0, I1.astype(np.float32))
