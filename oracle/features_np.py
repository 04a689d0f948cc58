"""The feature pre-alignment's keypoint and descriptor stage (fibsem_optflow_b200/csrc/tvl1_features.cu:
k_gauss7_u8, k_fast_score, k_nms_harris, the top-N selection of extract(), k_describe, k_knn2) restated in
NumPy.

TEST INFRASTRUCTURE ONLY (tests/, never the product).  The library is built with -fmad=false and without
fast-math, so each fp32 operation of a kernel is rounded once; this module keeps the kernels' fp32 operations
in their order, and the Gaussian, the FAST score, the non-maximum suppression, the Harris response and the
selection are reproduced bit for bit.  Two things are not: the orientation is atan2 in fp64 here (the device's
atan2f / sincosf are not correctly rounded), so `describe` returns the fp64 angle and marks the descriptor bits
whose rotated test offsets lie within DONT_CARE_EPS of a .5 rounding boundary, where the two may round apart.
Against OpenCV the module is pinned by tests/test_features_reference.py (FAST-9 corners, Gaussian, Harris).
"""
import math

import numpy as np

F32 = np.float32
DONT_CARE_EPS = 1e-4
RING = [(0, -3), (1, -3), (2, -2), (3, -1), (3, 0), (3, 1), (2, 2), (1, 3),
        (0, 3), (-1, 3), (-2, 2), (-3, 1), (-3, 0), (-3, -1), (-2, -2), (-1, -3)]   # (dx, dy), k_fast_score's order
UMAX = [int(math.floor(math.sqrt(15.0 * 15.0 - v * v) + 1e-9)) for v in range(16)]   # half-widths of the r-15 disc


# ---------------------------------------------------------------- 7x7 Gaussian

def gaussian_taps():
    """cv::getGaussianKernel(7, 2) as OpenCV computes it (exp(-x^2 / (2 sigma^2)) in fp64, times 1 / sum),
    rounded to fp32: the taps for dx = -3 .. 3"""
    scale2 = -0.5 / (2.0 * 2.0)
    t = [math.exp(scale2 * (i - 3.0) * (i - 3.0)) for i in range(7)]
    s = 0.0
    for v in t:
        s += v
    s = 1.0 / s
    return np.array([v * s for v in t], np.float64).astype(F32)


def _reflect101(p, n):
    p = np.abs(p)
    p = np.where(p >= n, 2 * n - 2 - p, p)
    return np.clip(p, 0, n - 1)


def gauss7(img):
    """k_gauss7_u8: row sums over dx = -3 .. 3 in fp32, then the column over dy = -3 .. 3, round half to even,
    clamp to 0 .. 255; reflect-101 border"""
    img = np.asarray(img, np.uint8)
    h, w = img.shape
    k = gaussian_taps()
    f = img.astype(F32)
    xs, ys = np.arange(w), np.arange(h)
    rows = np.zeros((h, w), F32)
    for dx in range(-3, 4):
        rows = rows + k[dx + 3] * f[:, _reflect101(xs + dx, w)]
    acc = np.zeros((h, w), F32)
    for dy in range(-3, 4):
        acc = acc + k[dy + 3] * rows[_reflect101(ys + dy, h), :]
    return np.clip(np.rint(acc), 0, 255).astype(np.uint8)


# ---------------------------------------------------------------- FAST-9, NMS, Harris

def fast_score(img, t, border):
    """k_fast_score: 0 = no corner (or within `border` of the frame), else the sum of |ring - centre| - t over
    the ring pixels on the corner's side (strictly beyond t) -- the larger side if both sides have a 9-arc"""
    img = np.asarray(img, np.uint8)
    h, w = img.shape
    out = np.zeros((h, w), F32)
    if w - 2 * border <= 0 or h - 2 * border <= 0:
        return out
    I = img.astype(np.int32)
    c = I[border:h - border, border:w - border]
    br = np.zeros(c.shape, np.uint32)
    dk = np.zeros(c.shape, np.uint32)
    sb = np.zeros(c.shape, np.int32)
    sd = np.zeros(c.shape, np.int32)
    for k, (ox, oy) in enumerate(RING):
        d = I[border + oy:h - border + oy, border + ox:w - border + ox] - c
        br |= (d > t).astype(np.uint32) << k
        dk |= (d < -t).astype(np.uint32) << k
        sb += np.where(d > t, d - t, 0)
        sd += np.where(d < -t, -d - t, 0)

    def arc9(m):
        m = m | (m << 16)
        r = m.copy()
        for k in range(1, 9):
            r &= m >> k
        return (r & 0xFFFF) != 0

    cb, cd = arc9(br), arc9(dk)
    out[border:h - border, border:w - border] = np.maximum(np.where(cb, sb, 0), np.where(cd, sd, 0)).astype(F32)
    return out


def nms(score, border):
    """k_nms_harris's suppression: (ys, xs) in raster order of the pixels inside `border` with a positive score
    that no 8-neighbour beats; on equal scores the earlier pixel in raster order wins"""
    s = np.asarray(score, F32)
    h, w = s.shape
    if w - 2 * border <= 0 or h - 2 * border <= 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    c = s[border:h - border, border:w - border]
    keep = c > 0
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dx == 0 and dy == 0:
                continue
            o = s[border + dy:h - border + dy, border + dx:w - border + dx]
            earlier = dy < 0 or (dy == 0 and dx < 0)
            keep &= ~((o > c) | ((o == c) if earlier else False))
    ys, xs = np.nonzero(keep)
    return ys + border, xs + border


def harris(img, ys, xs):
    """k_nms_harris's response at (ys, xs): integer Sobel derivatives over the 7x7 block, a / b / c accumulated
    in fp32 in dy-then-dx order, (a*b - c*c - 0.04*(a+b)*(a+b)) * sc^4 with sc = 1 / (4 * 7 * 255), and
    everything not above 1e-30 raised to 1e-30"""
    I = np.asarray(img, np.uint8).astype(np.int32)
    ys, xs = np.asarray(ys, np.int64), np.asarray(xs, np.int64)
    a = np.zeros(len(ys), F32)
    b = np.zeros(len(ys), F32)
    c = np.zeros(len(ys), F32)
    for dy in range(-3, 4):
        r0, r1, r2 = ys + dy - 1, ys + dy, ys + dy + 1
        for dx in range(-3, 4):
            X = xs + dx
            ix = I[r0, X + 1] - I[r0, X - 1] + 2 * (I[r1, X + 1] - I[r1, X - 1]) + I[r2, X + 1] - I[r2, X - 1]
            iy = I[r2, X - 1] - I[r0, X - 1] + 2 * (I[r2, X] - I[r0, X]) + I[r2, X + 1] - I[r0, X + 1]
            fx, fy = ix.astype(F32), iy.astype(F32)
            a = a + fx * fx
            b = b + fy * fy
            c = c + fx * fy
    sc = F32(1) / F32(4 * 7 * 255)
    sc4 = sc * sc * sc * sc
    hr = (a * b - c * c - F32(0.04) * (a + b) * (a + b)) * sc4
    return np.where(hr > F32(1e-30), hr, F32(1e-30)).astype(F32)


def harris_bins(hr):
    """the 2048-bin histogram k_nms_harris builds: float bits >> 20"""
    return np.bincount(np.asarray(hr, F32).view(np.uint32) >> 20, minlength=2048)


def fast_corners(img, t, border):
    """(score plane, ys, xs, harris) with the candidates in raster order"""
    s = fast_score(img, t, border)
    ys, xs = nms(s, border)
    return s, ys, xs, harris(img, ys, xs)


# ---------------------------------------------------------------- orientation and steered BRIEF

def brief_pattern():
    """upload_tables' 256 test pairs (ax, ay, bx, by): xorshift64, Box-Muller (sigma 6.2) with libm's log / cos /
    sin, pairs outside +-13 drawn again, lrint (half to even)"""
    M = (1 << 64) - 1
    r = 0x2545F4914F6CDD1D

    def uni():
        nonlocal r
        r ^= (r << 13) & M
        r ^= r >> 7
        r ^= (r << 17) & M
        return float((r >> 11) + 1) / 9007199254740993.0

    pat = []
    while len(pat) < 256 * 4:
        while True:
            u1, u2 = uni(), uni()
            m = math.sqrt(-2.0 * math.log(u1)) * 6.2
            gx, gy = m * math.cos(6.283185307179586 * u2), m * math.sin(6.283185307179586 * u2)
            if not (abs(gx) > 13.0 or abs(gy) > 13.0):
                break
        pat += [round(gx), round(gy)]
    return np.array(pat, np.int64).reshape(256, 4)


def moments(img, ys, xs):
    """(m01, m10) of the radius-15 disc around each keypoint, as integers"""
    I = np.asarray(img, np.uint8).astype(np.int64)
    ys, xs = np.asarray(ys, np.int64), np.asarray(xs, np.int64)
    m01 = np.zeros(len(ys), np.int64)
    m10 = np.zeros(len(ys), np.int64)
    for v in range(-15, 16):
        um = UMAX[abs(v)]
        for u in range(-um, um + 1):
            p = I[ys + v, xs + u]
            m10 += u * p
            m01 += v * p
    return m01, m10


def _pack(bits):
    """(n, 256) bool, test i = 8l + k -> byte l bit k -> (n, 8) little-endian uint32 words"""
    n = bits.shape[0]
    by = np.packbits(bits.reshape(n, 32, 8), axis=2, bitorder="little").reshape(n, 32)
    return np.ascontiguousarray(by).view("<u4").astype(np.uint32)


def describe(img, blur, ys, xs):
    """k_describe at (ys, xs): (angle in fp64, descriptors (n, 8) uint32, don't-care mask (n, 8) uint32 of the
    bits whose test offsets under the fp64 angle lie within DONT_CARE_EPS of a .5 rounding boundary)"""
    B = np.asarray(blur, np.uint8)
    ys, xs = np.asarray(ys, np.int64), np.asarray(xs, np.int64)
    m01, m10 = moments(img, ys, xs)
    ang = np.arctan2(m01.astype(np.float64), m10.astype(np.float64))
    cs, sn = np.cos(ang)[:, None], np.sin(ang)[:, None]
    pat = brief_pattern().astype(np.float64)
    t0, t1, t2, t3 = (pat[None, :, k] for k in range(4))
    offs = [t0 * cs - t1 * sn, t0 * sn + t1 * cs, t2 * cs - t3 * sn, t2 * sn + t3 * cs]   # ax, ay, bx, by
    dc = np.zeros((len(ys), 256), bool)
    for o in offs:
        dc |= np.abs(o - np.floor(o) - 0.5) < DONT_CARE_EPS
    ax, ay, bx, by = (np.rint(o).astype(np.int64) for o in offs)
    va = B[ys[:, None] + ay, xs[:, None] + ax]
    vb = B[ys[:, None] + by, xs[:, None] + bx]
    return ang, _pack(va < vb), _pack(dc)


# ---------------------------------------------------------------- Hamming 2-NN

def popcount_distances(q, t):
    """(nq, nt) Hamming distances of (n, 8) uint32 descriptors"""
    q = np.asarray(q, np.uint32).reshape(-1, 8)
    t = np.asarray(t, np.uint32).reshape(-1, 8)
    out = np.zeros((len(q), len(t)), np.int32)
    for k in range(8):
        out += np.bitwise_count(q[:, None, k] ^ t[None, :, k]).astype(np.int32)
    return out


def knn2(q, t):
    """k_knn2: (idx1, d1, d2): the nearest train index (the first on ties), its distance, and the second smallest
    distance over the other train descriptors (1 << 30 when there is only one)"""
    q = np.asarray(q, np.uint32).reshape(-1, 8)
    idx1, d1, d2 = (np.zeros(len(q), np.int32) for _ in range(3))
    for s in range(0, len(q), 512):
        D = popcount_distances(q[s:s + 512], t)
        i = np.argmin(D, axis=1)
        idx1[s:s + 512] = i
        d1[s:s + 512] = D[np.arange(len(i)), i]
        d2[s:s + 512] = np.partition(D, 1, axis=1)[:, 1] if D.shape[1] > 1 else (1 << 30)
    return idx1, d1, d2


# ---------------------------------------------------------------- one frame through extract()

def level_quota(nfeatures, scale_factor, nlevels):
    """ORB's per-level share of nfeatures as extract() computes it (fp64, lrint; the last level gets the rest)"""
    f = 1.0 / scale_factor
    per = nfeatures * (1.0 - f) / (1.0 - f ** nlevels)
    q, s = [], 0
    for _ in range(nlevels - 1):
        q.append(int(round(per)))
        s += q[-1]
        per *= f
    return q + [max(nfeatures - s, 0)]


def extract(img, nfeatures=5000, scale_factor=1.2, nlevels=8, edge_threshold=31, fast_threshold=20, prescale=None):
    """tvl1_features_extract of one frame: level l is the frame shrunk by 1 / scale_factor^l (the loader's 8-bit
    resize, `prescale(img, scale)`, default the C oracle's), its candidates ranked by (harris desc, y, x) and cut
    to the level's quota.  Returns a dict of per-keypoint arrays in the library's order: x, y (fp32, level-0
    pixels), level, cx, cy (level pixels), harris, angle (fp64), desc and dontcare ((n, 8) uint32)."""
    if prescale is None:
        from oracle.oracle import prescale_u8 as prescale
    img = np.asarray(img, np.uint8)
    sf = float(F32(scale_factor))        # tvl1_feature_params.scale_factor is a float
    border = max(edge_threshold, 19)
    quota = level_quota(nfeatures, sf, nlevels)
    parts = []
    total = 0
    for l in range(nlevels):
        if total >= nfeatures:
            break
        sc = sf ** l
        lv = img if l == 0 else prescale(img, 1.0 / sc)
        lh, lw = lv.shape
        if lw <= 2 * border + 8 or lh <= 2 * border + 8:
            break
        _, ys, xs, hr = fast_corners(lv, fast_threshold, border)
        want = min(quota[l], nfeatures - total)
        if len(ys) == 0 or want == 0:
            continue
        o = np.lexsort((xs, ys, -hr))[:want]
        ys, xs, hr = ys[o], xs[o], hr[o]
        ang, desc, dc = describe(lv, gauss7(lv), ys, xs)
        parts.append(dict(x=xs.astype(F32) * F32(sc), y=ys.astype(F32) * F32(sc), level=np.full(len(ys), l, np.int32),
                          cx=xs, cy=ys, harris=hr, angle=ang, desc=desc, dontcare=dc))
        total += len(ys)
    if not parts:
        z = np.zeros(0, np.int64)
        return dict(x=z.astype(F32), y=z.astype(F32), level=z.astype(np.int32), cx=z, cy=z, harris=z.astype(F32),
                    angle=z.astype(np.float64), desc=np.zeros((0, 8), np.uint32), dontcare=np.zeros((0, 8), np.uint32))
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
