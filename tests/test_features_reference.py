"""The NumPy restatement of the feature kernels (oracle/features_np.py) against OpenCV, on the CPU: the
GPU tests (tests/test_gpu_features_kernels.py) hold the kernels to this reference bit for bit, so the reference
itself must compute the operations it names."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth
from oracle import features_np as FN

cv2 = pytest.importorskip("cv2")


def frames():
    return [("noise", np.random.default_rng(1).integers(0, 256, (300, 400), dtype=np.uint8)),
            ("texture", synth.to_u8(synth.texture(400, 500, 5, 2.0, coarse=8)))]


def test_gaussian_taps_are_opencvs():
    k = FN.gaussian_taps()
    assert np.array_equal(k, np.float32(cv2.getGaussianKernel(7, 2)).ravel())
    assert abs(float(k.astype(np.float64).sum()) - 1.0) < 1e-6


@pytest.mark.parametrize("name,img", frames())
def test_gauss7_reference_vs_cv2(name, img):
    """within 1 grey level of cv2.GaussianBlur (whose 8-bit path is fixed point and is off by one on a few per
    cent of the pixels), and equal to the exact value rounded wherever that is not near a .5 boundary"""
    got = FN.gauss7(img).astype(int)
    want = cv2.GaussianBlur(img, (7, 7), 2, borderType=cv2.BORDER_REFLECT_101).astype(int)
    assert np.abs(got - want).max() <= 1, name
    assert (got != want).mean() < 0.25, name
    k = cv2.getGaussianKernel(7, 2).ravel()
    p = np.pad(img.astype(np.float64), 3, mode="reflect")
    h, w = img.shape
    r = sum(k[i] * p[:, i:i + w] for i in range(7))
    r = sum(k[i] * r[i:i + h, :] for i in range(7))
    far = np.abs(r - np.floor(r) - 0.5) > 1e-3
    assert np.array_equal(got[far], np.rint(r)[far].astype(int)), name


@pytest.mark.parametrize("t", [1, 20, 60])
@pytest.mark.parametrize("name,img", frames())
def test_fast_score_support_is_cv2_fast9(name, img, t):
    """the pixels with a FAST score > 0 are cv2's FAST-9 corners (no suppression) inside the border"""
    b = 19
    s = FN.fast_score(img, t, b)
    kp = cv2.FastFeatureDetector_create(t, False, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16).detect(img)
    h, w = img.shape
    want = {(int(k.pt[0]), int(k.pt[1])) for k in kp if b <= k.pt[0] < w - b and b <= k.pt[1] < h - b}
    ys, xs = np.nonzero(s > 0)
    assert set(zip(xs.tolist(), ys.tolist())) == want, (name, t)
    assert len(want) > 100 or t == 60


@pytest.mark.parametrize("name,img", frames())
def test_harris_reference_vs_cv2_corner_harris(name, img):
    """ORB's Harris ranking is cv2.cornerHarris(blockSize 7, Sobel 3, k 0.04) up to fp32 rounding"""
    _, ys, xs, hr = FN.fast_corners(img, 20, 19)
    assert len(ys) > 100
    R = cv2.cornerHarris(img, 7, 3, 0.04)[ys, xs].astype(np.float64)
    # the response is a difference of terms: its error is relative to their size
    I = img.astype(np.int64)
    a = b = c = 0
    for dy in range(-3, 4):
        for dx in range(-3, 4):
            Y, X = ys + dy, xs + dx
            ix = I[Y - 1, X + 1] - I[Y - 1, X - 1] + 2 * (I[Y, X + 1] - I[Y, X - 1]) + I[Y + 1, X + 1] - I[Y + 1, X - 1]
            iy = I[Y + 1, X - 1] - I[Y - 1, X - 1] + 2 * (I[Y + 1, X] - I[Y - 1, X]) + I[Y + 1, X + 1] - I[Y - 1, X + 1]
            a, b, c = a + ix * ix, b + iy * iy, c + ix * iy
    sc4 = (1.0 / (4 * 7 * 255)) ** 4
    mag = (a * b + c * c + 0.04 * (a + b) ** 2) * sc4
    exact = (a * b - c * c - 0.04 * (a + b) ** 2) * sc4
    assert np.all(np.abs(np.maximum(exact, 1e-30) - hr) <= 1e-5 * mag + 1e-37), name
    assert np.all(np.abs(R - exact) <= 1e-4 * mag), name
    # the histogram bins follow the response's order
    bins = hr.view(np.uint32) >> 20
    o = np.argsort(hr, kind="stable")
    assert np.all(np.diff(bins[o].astype(np.int64)) >= 0)


def test_nms_tie_rule():
    s = np.zeros((16, 16), np.float32)
    s[5, 5] = s[5, 6] = s[6, 5] = 3.0      # a plateau: only its first pixel in raster order survives
    s[5, 8] = 2.0                          # beaten by nobody within 3x3
    s[8, 8] = 1.0
    s[8, 9] = 4.0                          # beats its left neighbour
    ys, xs = FN.nms(s, 4)
    assert list(zip(ys.tolist(), xs.tolist())) == [(5, 5), (5, 8), (8, 9)]


def test_brief_pattern_and_disc():
    p = FN.brief_pattern()
    assert p.shape == (256, 4) and np.abs(p).max() <= 13
    assert np.array_equal(p, FN.brief_pattern())
    # an isotropic Gaussian of sigma 6.2 clipped to +-13
    assert 4.5 < p.std() < 6.5 and abs(p.mean()) < 1.0
    assert FN.UMAX[0] == 15 and FN.UMAX[15] == 0 and all(a >= b for a, b in zip(FN.UMAX, FN.UMAX[1:]))


def test_describe_flat_disc_and_quadrants():
    img = np.full((80, 80), 100, np.uint8)
    ang, _, _ = FN.describe(img, img, np.array([40]), np.array([40]))
    assert ang[0] == 0.0                   # atan2(0, 0)
    for (dx, dy), want in [((1, 0), 0.0), ((0, 1), np.pi / 2), ((-1, 0), np.pi), ((0, -1), -np.pi / 2)]:
        g = np.clip(100 + 5 * (dx * (np.arange(80)[None, :] - 40) + dy * (np.arange(80)[:, None] - 40)), 0, 255)
        ang, _, _ = FN.describe(g.astype(np.uint8), g.astype(np.uint8), np.array([40]), np.array([40]))
        assert abs(ang[0] - want) < 1e-12, (dx, dy, ang)


def test_knn2_reference_vs_cv2_bfmatcher():
    rng = np.random.default_rng(3)
    q = rng.integers(0, 2 ** 32, (300, 8), dtype=np.uint32)
    t = rng.integers(0, 2 ** 32, (200, 8), dtype=np.uint32)
    t[50] = q[7]                           # exact match
    idx1, d1, d2 = FN.knn2(q, t)
    m = cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch(q.view(np.uint8), t.view(np.uint8), k=2)
    assert [x[0].distance for x in m] == d1.tolist() and [x[1].distance for x in m] == d2.tolist()
    assert idx1[7] == 50 and d1[7] == 0
    # ties: the first index wins, the second distance equals the first
    t2 = np.concatenate([t[:3], t[:3]])
    i, a, b = FN.knn2(t[:3], t2)
    assert i.tolist() == [0, 1, 2] and a.tolist() == [0, 0, 0] and b.tolist() == [0, 0, 0]
    i, a, b = FN.knn2(q[:4], t[:1])
    assert i.tolist() == [0] * 4 and b.tolist() == [1 << 30] * 4


def test_level_quota():
    q = FN.level_quota(5000, float(np.float32(1.2)), 8)
    assert sum(q) == 5000 and q[0] > q[1] > q[-2] and len(q) == 8
    assert FN.level_quota(16, 1.2, 1) == [16]
