"""The feature pre-alignment's kernels one by one, and one frame through extract(), against the NumPy
restatement oracle/features_np.py (itself pinned against OpenCV by tests/test_features_reference.py).

Bit for bit: the 7x7 Gaussian, the FAST score plane, the NMS survivors and their Harris responses, the
histogram, the 2-NN, and the keypoints extract() keeps (position, level, order).  The orientation is compared
with atan2 in fp64 (the device's atan2f / sincosf are not correctly rounded): the angle within 1e-5 rad, the
descriptor bits exactly except where a rotated test offset lies within 1e-4 of a .5 rounding boundary."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth
from oracle import features_np as FN

pytestmark = pytest.mark.gpu


def texture(h, w, seed):
    return synth.to_u8(synth.texture(h, w, seed, 2.0, coarse=8))


def noise(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)


def up512(n):
    return (n + 511) // 512 * 512


@pytest.fixture(scope="module")
def solver(gpu):
    s = gpu.Solver(gpu.default_params())
    yield s
    s.close()


def check_descriptors(kp, desc, ang, want, dontcare, stats=None):
    """angle within 1e-5 rad of the fp64 value, descriptor bits equal outside the don't-care mask"""
    d = np.abs(kp["angle"].astype(np.float64) - ang)
    d = np.minimum(d, 2 * np.pi - d)
    assert d.max() <= 1e-5, d.max()
    bad = (desc ^ want) & ~dontcare
    assert not bad.any(), "%d descriptors differ outside the don't-care bits" % int(bad.any(axis=1).sum())
    if stats is not None:
        stats.append((int(np.bitwise_count(dontcare).sum()), dontcare.size * 32))


# ---------------------------------------------------------------- k_gauss7_u8

@pytest.mark.parametrize("w,h", [(47, 47), (61, 250), (333, 517), (900, 1100), (1, 9), (5, 3)])
@pytest.mark.parametrize("pitched", [False, True])
def test_gauss7_bit_exact(gpu, w, h, pitched):
    """taps = fp32 cv::getGaussianKernel(7, 2), fp32 sums in the kernel's order, reflect-101 (also on frames
    smaller than the aperture), widths not a multiple of 32, heights not a multiple of 8"""
    for img in (noise(h, w, w + h), texture(max(h, 8), max(w, 8), 3)[:h, :w]):
        sp, dp = (up512(w), w + 13) if pitched else (None, None)
        got = gpu.k_gauss7_u8(img, spitch=sp, dpitch=dp)
        want = FN.gauss7(img)
        assert np.array_equal(got, want), (w, h, int(np.abs(got.astype(int) - want).max()))


# ---------------------------------------------------------------- k_fast_score + k_nms_harris

ARC9 = list(range(9))


def ring_frame(t):
    """crafted 7x7 rings on a flat frame, with whether each centre must fire"""
    c = 0 if t > 150 else 100
    hi = min(255, c + max(t + 1, 60))
    lo = c - max(t + 1, 60)
    img = np.full((260, 300), c, np.uint8)
    cases = [
        (c, hi, ARC9, True),                                  # an exact 9-arc
        (c, hi, list(range(8)), False),                       # 8 contiguous: not a corner
        (c, hi, [12, 13, 14, 15, 0, 1, 2, 3, 4], True),       # a 9-arc across ring index 15 -> 0
        (c, hi, list(range(16)), True),                       # the whole ring
        (c, hi, [0, 1, 2, 3, 5, 6, 7, 8, 9], False),          # 9 set but not contiguous
    ]
    if lo >= 0:
        cases += [(c, lo, list(range(3, 12)), True), (c, lo, [13, 14, 15, 0, 1, 2, 3, 4], False),
                  (c, lo, [10, 11, 12, 13, 14, 15, 0, 1, 2], True)]
    cases += [(0, 255, list(range(4, 13)), True), (255, 0, [14, 15, 0, 1, 2, 3, 4, 5, 6], True),   # saturated
              (0, 255, list(range(8)), False)]
    out = []
    for i, (cv, rv, idx, fires) in enumerate(cases):
        y, x = 40 + 20 * (i // 10), 40 + 22 * (i % 10)
        img[y - 4:y + 5, x - 4:x + 5] = cv
        for k in idx:
            ox, oy = FN.RING[k]
            img[y + oy, x + ox] = rv
        fires = fires and abs(int(rv) - int(cv)) > t
        out.append((x, y, fires))
    # a pixel exactly t above the centre breaks the arc (the test is strict)
    if c + t + 1 <= 255:
        y, x = 220, 60
        for k in ARC9:
            ox, oy = FN.RING[k]
            img[y + oy, x + ox] = c + t + (k != 4)
        out.append((x, y, False))
    return img, out


def plateau_frame():
    """small bright blocks on a flat frame: equal FAST scores side by side, for the NMS tie rule"""
    img = np.full((300, 340), 60, np.uint8)
    rng = np.random.default_rng(9)
    for y in range(36, 264, 12):
        for x in range(36, 304, 12):
            bh, bw = rng.integers(1, 4, 2)
            img[y:y + bh, x:x + bw] = 200
    return img


def saturated_frame():
    return (noise(240, 270, 4) > 127).astype(np.uint8) * 255


FRAMES = {"noise": lambda: noise(333, 517, 1), "texture": lambda: texture(600, 700, 5), "plateau": plateau_frame,
          "saturated": saturated_frame}


def run_fast(gpu, img, t, border, pitched=True):
    h, w = img.shape
    score, cand, n, hist = gpu.k_fast_corners(img, border, t, pitch=up512(w) if pitched else None,
                                              spitch=w + 7 if pitched else None)
    s_ref, ys, xs, hr = FN.fast_corners(img, t, border)
    assert np.array_equal(score, s_ref), int((score != s_ref).sum())
    assert n == len(cand) == len(ys)
    o = np.lexsort((cand["x"], cand["y"]))
    c = cand[o]
    assert np.array_equal(c["y"].astype(np.int64), ys) and np.array_equal(c["x"].astype(np.int64), xs)
    assert np.array_equal(c["harris"].view(np.uint32), hr.view(np.uint32))
    assert np.array_equal(hist, FN.harris_bins(c["harris"]))
    return score, c


@pytest.mark.parametrize("t", [1, 20, 254])
@pytest.mark.parametrize("border", [19, 31])
@pytest.mark.parametrize("frame", sorted(FRAMES))
def test_fast_corners_bit_exact(gpu, frame, t, border):
    img = FRAMES[frame]()
    _, c = run_fast(gpu, img, t, border)
    if frame == "plateau" and t < 100:
        assert len(c) > 100


@pytest.mark.parametrize("t", [1, 20, 254])
@pytest.mark.parametrize("border", [19, 31])
def test_fast_corners_crafted_rings(gpu, t, border):
    img, cases = ring_frame(t)
    score, _ = run_fast(gpu, img, t, border)
    for x, y, fires in cases:
        assert (score[y, x] > 0) == fires, (x, y, fires, score[y, x])


def test_fast_corners_list_overflow_still_counts(gpu):
    """past `cap` the list drops entries but the count and the histogram keep every survivor"""
    img = texture(400, 500, 6)
    _, cand, n, hist = gpu.k_fast_corners(img, 19, 20, cap=100)
    _, ys, _, hr = FN.fast_corners(img, 20, 19)
    assert n == len(ys) > 100 and len(cand) == 100
    assert np.array_equal(hist, FN.harris_bins(hr))


# ---------------------------------------------------------------- k_describe

def describe_case(img, border=19, extra=()):
    h, w = img.shape
    rng = np.random.default_rng(h * w)
    pts = [(border, border), (w - border - 1, border), (border, h - border - 1), (w - border - 1, h - border - 1),
           (border, h // 2), (w - border - 1, h // 2), (w // 2, border), (w // 2, h - border - 1)]
    pts += list(extra)
    pts += list(zip(rng.integers(border, w - border, 1500).tolist(), rng.integers(border, h - border, 1500).tolist()))
    return np.array(pts, np.int64)


@pytest.mark.parametrize("scale,level,pitched", [(1.0, 0, False), (1.0, 0, True), (1.44, 2, True)])
def test_describe(gpu, scale, level, pitched, record_property):
    img = texture(300, 420, 8)
    img[100:140, 200:240] = 120                               # a flat disc: angle 0
    blur = FN.gauss7(img)
    pts = describe_case(img, extra=[(220, 120)])
    h, w = img.shape
    kp, desc = gpu.k_describe(img, blur, pts, scale=scale, level=level,
                              pitch=up512(w) if pitched else None, bpitch=w + 3 if pitched else None)
    ang, want, dc = FN.describe(img, blur, pts[:, 1], pts[:, 0])
    assert np.array_equal(kp["x"], pts[:, 0].astype(np.float32) * np.float32(scale))
    assert np.array_equal(kp["y"], pts[:, 1].astype(np.float32) * np.float32(scale))
    assert (kp["level"] == level).all()
    assert kp["angle"][8] == 0.0 and ang[8] == 0.0
    quads = {(bool(np.sin(a) >= 0), bool(np.cos(a) >= 0)) for a in ang}
    assert len(quads) == 4
    stats = []
    check_descriptors(kp, desc, ang, want, dc, stats)
    share = stats[0][0] / stats[0][1]
    record_property("dont_care_share", share)
    print("k_describe don't-care bits: %d of %d (%.4f %%)" % (stats[0][0], stats[0][1], 100 * share))
    assert share < 0.01


# ---------------------------------------------------------------- k_knn2

SIZES = [1, 2, 127, 128, 129, 5000]


def descriptor_set(n, seed):
    rng = np.random.default_rng(seed)
    d = rng.integers(0, 2 ** 32, (n, 8), dtype=np.uint32)
    if n >= 4:
        d[1] = 0
        d[2] = 0xFFFFFFFF
        d[n - 1] = d[0]                                        # a duplicate: d1 == d2 for its neighbours
    if n >= 50:
        d[n // 2: n // 2 + 10] = d[3:13]
    return d


@pytest.mark.parametrize("nt", SIZES)
@pytest.mark.parametrize("nq", SIZES)
def test_knn2_exact(gpu, nq, nt):
    q = descriptor_set(nq, nq)
    t = descriptor_set(nt, 1000 + nt)
    if nq >= 4 and nt >= 4:
        q[3] = t[nt - 1]                                       # equal to t[0] and t[nt-1]: the first index wins
    got = gpu.k_knn2(q, t)
    want = FN.knn2(q, t)
    for g, wv, name in zip(got, want, ("idx1", "d1", "d2")):
        assert np.array_equal(g, wv), (name, nq, nt, int((g != wv).sum()))
    if nt == 1:
        assert (got[2] == 1 << 30).all()
    if nq >= 4 and nt >= 4:
        assert got[0][3] == 0 and got[1][3] == 0 and got[2][3] == 0


# ---------------------------------------------------------------- one frame through extract()

def compare_extract(gpu_out, ref, stats=None):
    kp, desc = gpu_out
    assert len(kp) == len(ref["x"])
    assert np.array_equal(kp["level"], ref["level"])
    assert np.array_equal(kp["x"], ref["x"]) and np.array_equal(kp["y"], ref["y"])
    check_descriptors(kp, desc, ref["angle"], ref["desc"], ref["dontcare"], stats)


@pytest.mark.parametrize("nlevels", [1, 3, 8])
@pytest.mark.parametrize("nfeatures", [16, 500, 5000])
def test_features_extract(solver, nfeatures, nlevels):
    img = texture(700, 900, 13)
    ref = FN.extract(img, nfeatures=nfeatures, nlevels=nlevels)
    assert 0 < len(ref["x"]) <= nfeatures
    compare_extract(solver.features_extract(img, nfeatures=nfeatures, nlevels=nlevels), ref)
    if nfeatures == 500:
        # level 0 of a padded frame is read with the frame's pitch, its smoothed copy with its own
        compare_extract(solver.features_extract(img, pitch=up512(900), nfeatures=nfeatures, nlevels=nlevels), ref)
        compare_extract(solver.features_extract(img, pitch=901, nfeatures=nfeatures, nlevels=nlevels), ref)


@pytest.mark.parametrize("edge", [31, 19])
def test_features_extract_small_frame(solver, edge):
    """a frame just above the 2*border + 8 cutoff: level 0 only"""
    n = 2 * max(edge, 19) + 9
    img = noise(n, n + 3, edge)
    ref = FN.extract(img, nfeatures=500, nlevels=3, edge_threshold=edge)
    assert len(ref["x"]) > 0 and (ref["level"] == 0).all()
    compare_extract(solver.features_extract(img, pitch=up512(n + 3), nfeatures=500, nlevels=3, edgeThreshold=edge), ref)
    # one row fewer: at the cutoff, no level is searched
    assert len(solver.features_extract(img[:-1], nfeatures=500, nlevels=3, edgeThreshold=edge)[0]) == 0


def dot_lattice(h, w, period, bg=40, dot=200):
    img = np.full((h, w), bg, np.uint8)
    img[::period, ::period] = dot
    return img


def test_features_extract_lattice_of_equal_corners(solver):
    """4096^2 frame of isolated dots, period 8: ~262k level-0 candidates with bit-identical responses, far more
    than the quota -- the kept ones are the lowest (y, x), as the reference selects them, run after run"""
    img = dot_lattice(4096, 4096, 8)
    ref = FN.extract(img)
    lv0 = ref["level"] == 0
    q0 = FN.level_quota(5000, float(np.float32(1.2)), 8)[0]
    assert lv0.sum() == q0 and len(np.unique(ref["harris"][lv0])) == 1
    ys, xs = np.nonzero(img[31:-31, 31:-31] == 200)
    assert np.array_equal(ref["cy"][lv0], ys[:q0] + 31) and np.array_equal(ref["cx"][lv0], xs[:q0] + 31)
    a = solver.features_extract(img)
    compare_extract(a, ref)
    b = solver.features_extract(img)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_features_extract_more_survivors_than_the_list(solver):
    """16384 x 8192, a dot every 4 px: 8.3M NMS survivors with one response, more than the candidate list's
    initial 4M entries; the list grows and the kept keypoints are still the first in raster order"""
    img = dot_lattice(8192, 16384, 4)
    ys, xs = np.nonzero(img[31:-31, 31:-31] == 200)
    assert len(ys) > 1 << 22
    kp, _ = solver.features_extract(img, nfeatures=5000, nlevels=1)
    assert len(kp) == 5000 and (kp["level"] == 0).all()
    assert np.array_equal(kp["y"], (ys[:5000] + 31).astype(np.float32))
    assert np.array_equal(kp["x"], (xs[:5000] + 31).astype(np.float32))


# ---------------------------------------------------------------- pitched frames through find_alignment

def moved_pair(h, w, seed, angle_deg, zoom, tx, ty):
    import cv2
    m = 120
    c = texture(h + 2 * m, w + 2 * m, seed)
    th = np.deg2rad(angle_deg)
    M = np.array([[zoom * np.cos(th), -zoom * np.sin(th), tx + m], [zoom * np.sin(th), zoom * np.cos(th), ty + m]])
    f0 = np.ascontiguousarray(c[m:m + h, m:m + w])
    f1 = cv2.warpAffine(c, M, (w, h), flags=cv2.INTER_CUBIC | cv2.WARP_INVERSE_MAP)
    return f0, f1


@pytest.mark.parametrize("pitch", ["512", "w+1"])
def test_find_alignment_pitched_equals_unpitched(solver, pitch):
    h, w = 900, 1100
    f0, f1 = moved_pair(h, w, 5, 0.4, 1.02, 7.3, -4.6)
    p = up512(w) if pitch == "512" else w + 1
    aff, nm, ng = solver.find_alignment(f1, f0)
    assert not np.array_equal(aff, np.array([[1, 0, 0], [0, 1, 0]], np.float32)) and ng > 50
    paff, pnm, png = solver.find_alignment(f1, f0, pitch_moving=p, pitch_fixed=p, pad_value=255)
    assert np.array_equal(aff.view(np.uint32), paff.view(np.uint32)) and (nm, ng) == (pnm, png)
