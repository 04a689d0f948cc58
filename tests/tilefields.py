"""Flow fields that steer the tile-walking kernels (k_warp, k_warp_cuda, k_median5) down every path they have,
and the kernels' host-visible geometry restated in NumPy, so that a test can count which path each tile,
thread and pixel takes.  CPU only; tests/test_tilefields.py checks that the fields contain every class, and
tests/test_gpu_tile_walk.py runs them through the kernels.

The restatement follows fibsem_optflow_b200/csrc/tvl1_kernels.cuh and must change with it:
  k_warp       64 x 8 tiles; a thread owns one column and 4 consecutive rows (rows 4k .. 4k+3 of the image);
               source(), window(), the TMA / scalar-window / global-load choice, the 16- or 32-row box and
               the register-window ("column") condition of stage_c.
  k_warp_cuda  32 x 16 tiles; the box of the clamped taps and their gradient neighbours, staged when it is at
               most 64 x 48.
  k_median5    128 x 16 tiles; the interior test that sends a tile to TMA instead of clamped copies.
"""
import numpy as np

WP_TW, WP_TH, WP_PX, WP_RW, WP_RH = 64, 8, 4, 88, 32
WC_TW, WC_TH, WC_RW, WC_RH = 32, 16, 64, 48
MED_TW, MED_TH = 128, 16

F32 = np.float32


def cdiv(a, b):
    return -(-a // b)


def roundup(a, b):
    return cdiv(a, b) * b


# ---------------------------------------------------------------- k_warp


def source(w, h, u1, u2):
    """source() of k_warp for every pixel: sx, sy (the taps are columns sx .. sx+3, rows sy .. sy+3) and the
    outside bit of fxy.  fp32 as on the device: mx = x + u1, qx = rn(mx * 32), sx = clamp(qx >> 5) - 1."""
    ys, xs = np.mgrid[0:h, 0:w]
    mx = xs.astype(F32) + u1.astype(F32)
    my = ys.astype(F32) + u2.astype(F32)
    lim = float(2 ** 31 - 128)   # __float2int_rn saturates; the flows here stay far inside int32
    qx = np.rint(np.clip(mx * F32(32), -lim, lim)).astype(np.int64)
    qy = np.rint(np.clip(my * F32(32), -lim, lim)).astype(np.int64)
    sx = np.clip(qx >> 5, -32768, 32767) - 1
    sy = np.clip(qy >> 5, -32768, 32767) - 1
    outside = (sx >= w) | (sx + 4 <= 0) | (sy >= h) | (sy + 4 <= 0)
    return sx, sy, outside


def _tiles(a, th, tw, fill):
    """(h, w) -> (tiles_y, tiles_x, th, tw), the missing part of the last tiles filled with `fill`"""
    h, w = a.shape
    ty, tx = cdiv(h, th), cdiv(w, tw)
    p = np.full((ty * th, tx * tw), fill, a.dtype)
    p[:h, :w] = a
    return p.reshape(ty, th, tx, tw).transpose(0, 2, 1, 3)


def warp_geometry(w, h, u1, u2):
    """What k_warp does with the flow (u1, u2): a dict of per-tile, per-thread and per-pixel arrays.
    per tile (tiles_y, tiles_x):  rw, rh, staged, tma (window inside the image), box16 (TMA box of 16 rows),
                                  empty (no live pixel with an inside source)
    per thread (tiles_y, tiles_x, 2, 64): column (register-window path), sx0 / sy0 (its first source)
    per pixel (h, w): sx, sy, outside, inside (all 16 taps in the image), partial (neither)"""
    sx, sy, outside = source(w, h, u1, u2)
    big = 2 ** 31 - 1
    valid = ~outside
    X0 = _tiles(np.where(valid, sx, big), WP_TH, WP_TW, big).min(axis=(2, 3))
    Y0 = _tiles(np.where(valid, sy, big), WP_TH, WP_TW, big).min(axis=(2, 3))
    X1 = _tiles(np.where(valid, sx, -big), WP_TH, WP_TW, -big).max(axis=(2, 3))
    Y1 = _tiles(np.where(valid, sy, -big), WP_TH, WP_TW, -big).max(axis=(2, 3))
    empty = X1 < X0
    rx0 = ((X0 - 1) >> 2) << 2
    ry0 = Y0 - 1
    rw = X1 + 4 - rx0 + 1
    rh = Y1 + 4 - ry0 + 1
    staged = ~empty & (rw <= WP_RW) & (rh <= WP_RH)
    tma = staged & (rx0 >= 0) & (rx0 + rw - 1 <= w - 1) & (ry0 >= 0) & (ry0 + rh - 1 <= h - 1)
    box16 = tma & (rh <= 16)
    inside = (sx >= 0) & (sx < max(w - 3, 0)) & (sy >= 0) & (sy < max(h - 3, 0))
    # threads: (tiles_y, tiles_x, 2 row groups, 64 columns, 4 pixels)
    T = lambda a, f: _tiles(a, WP_TH, WP_TW, f).reshape(cdiv(h, WP_TH), cdiv(w, WP_TW), 2, WP_PX, WP_TW).transpose(0, 1, 2, 4, 3)
    live = T(np.ones((h, w), bool), False)
    tsx, tsy = T(sx, 0), T(sy, 0)
    k = np.arange(WP_PX)
    column = (staged[:, :, None, None] & live.all(-1) & T(valid, False).all(-1) & T(inside, False).all(-1)
              & (tsx == tsx[..., :1]).all(-1) & (tsy == tsy[..., :1] + k).all(-1))
    return dict(rw=rw, rh=rh, staged=staged, tma=tma, box16=box16, empty=empty, column=column,
                sx0=tsx[..., 0], sy0=tsy[..., 0], thread_live=live.all(-1),
                sx=sx, sy=sy, outside=outside, inside=inside & valid, partial=valid & ~inside)


def warp_classes(w, h, u1, u2):
    """Counts of every path and boundary of k_warp that the flow reaches (tests/test_tilefields.py)"""
    g = warp_geometry(w, h, u1, u2)
    tiles_y, tiles_x = g["rw"].shape
    st = g["staged"]
    # a thread that would be a column thread but for the last-column / last-row limit
    ok = g["thread_live"] & st[:, :, None, None]
    col = g["column"]
    c = {
        "tile_tma16": int(g["box16"].sum()),
        "tile_tma32": int((g["tma"] & ~g["box16"]).sum()),
        "tile_scalar_window": int((st & ~g["tma"]).sum()),
        "tile_global": int((~st & ~g["empty"]).sum()),
        "tile_all_outside": int(g["empty"].sum()),
        "thread_column": int(col.sum()),
        "thread_perpixel_staged": int((ok & ~col).sum()),
        "thread_perpixel_global": int((g["thread_live"] & ~st[:, :, None, None]).sum()),
        "column_sx_w-4": int((col & (g["sx0"] == w - 4)).sum()),
        "column_sy_h-4": int((col & (g["sy0"] + WP_PX - 1 == h - 4)).sum()),
        "column_sx_0": int((col & (g["sx0"] == 0)).sum()),
        "column_sy_0": int((col & (g["sy0"] == 0)).sum()),
        "px_sx_w-3": int((~g["outside"] & (g["sx"] == w - 3)).sum()),
        "px_sy_h-3": int((~g["outside"] & (g["sy"] == h - 3)).sum()),
        "px_outside_sx_w": int((g["sx"] == w).sum()),
        "px_outside_sx+4_0": int((g["sx"] + 4 == 0).sum()),
        "px_outside_far": int((np.abs(g["sx"]) > 5000).sum()),
        "px_partial": int(g["partial"].sum()),
        "px_inside": int(g["inside"].sum()),
    }
    # the window limits, each on the path it decides: a window that fits is copied by TMA (inside the image),
    # one row or column more sends the tile to global loads
    for v in (88, 16, 17, 32):
        c["tile_%s_%d_tma" % ("rw" if v == 88 else "rh", v)] = int((g["tma"] & (g["rw" if v == 88 else "rh"] == v)).sum())
    c["tile_rw_89_global"] = int((~st & ~g["empty"] & (g["rw"] == 89) & (g["rh"] <= WP_RH)).sum())
    c["tile_rh_33_global"] = int((~st & ~g["empty"] & (g["rh"] == 33) & (g["rw"] <= WP_RW)).sum())
    c["tiles"] = tiles_x * tiles_y
    return c


# ---------------------------------------------------------------- k_warp_cuda


def cuda_taps(v):
    """cuda_taps of k_warp_cuda: lo = ceil(v - 2), n = floor(v + 2) - lo + 1 held to 0 .. 5 (fp32 sums)"""
    v = v.astype(F32)
    lo = np.ceil(v - F32(2)).astype(np.int64)
    hi = np.floor(v + F32(2)).astype(np.int64)
    return lo, np.clip(hi - lo + 1, 0, 5)


def warp_cuda_geometry(w, h, u1, u2):
    """The staged box of each k_warp_cuda tile: (width, height, staged) per tile, and the per-pixel tap counts"""
    ys, xs = np.mgrid[0:h, 0:w]
    fx = xs.astype(F32) + u1.astype(F32)
    fy = ys.astype(F32) + u2.astype(F32)
    lx, nx = cuda_taps(fx)
    ly, ny = cuda_taps(fy)
    big = 2 ** 31 - 1
    okx, oky = nx > 0, ny > 0
    bx0 = np.where(okx, np.clip(lx, 0, w - 1) - 1, big)
    bx1 = np.where(okx, np.clip(lx + nx - 1, 0, w - 1) + 1, -1)
    by0 = np.where(oky, np.clip(ly, 0, h - 1) - 1, big)
    by1 = np.where(oky, np.clip(ly + ny - 1, 0, h - 1) + 1, -1)
    rx0 = np.maximum(_tiles(bx0, WC_TH, WC_TW, big).min(axis=(2, 3)), 0)
    ry0 = np.maximum(_tiles(by0, WC_TH, WC_TW, big).min(axis=(2, 3)), 0)
    rx1 = np.minimum(_tiles(bx1, WC_TH, WC_TW, -1).max(axis=(2, 3)), w - 1)
    ry1 = np.minimum(_tiles(by1, WC_TH, WC_TW, -1).max(axis=(2, 3)), h - 1)
    bw, bh = rx1 - rx0 + 1, ry1 - ry0 + 1
    staged = (rx1 >= rx0) & (ry1 >= ry0) & (bw <= WC_RW) & (bh <= WC_RH)
    return dict(bw=bw, bh=bh, staged=staged, nx=nx, ny=ny)


def warp_cuda_classes(w, h, u1, u2):
    g = warp_cuda_geometry(w, h, u1, u2)
    c = {"tile_staged": int(g["staged"].sum()), "tile_global": int((~g["staged"]).sum()),
         "px_5_taps": int(((g["nx"] == 5) | (g["ny"] == 5)).sum()), "tiles": g["staged"].size}
    for v in (64, 65):
        c["tile_bw_%d" % v] = int(((g["bw"] == v) & (g["bh"] <= WC_RH)).sum())
    for v in (48, 49):
        c["tile_bh_%d" % v] = int(((g["bh"] == v) & (g["bw"] <= WC_RW)).sum())
    return c


# ---------------------------------------------------------------- k_median5


def median5_interior(w, h):
    """Per tile (tiles_y, tiles_x): True where k_median5 stages the tile by TMA (no border handling needed)"""
    x0 = np.arange(cdiv(w, MED_TW)) * MED_TW
    y0 = np.arange(cdiv(h, MED_TH)) * MED_TH
    return ((y0[:, None] >= 2) & (y0[:, None] + MED_TH + 2 <= h)) & ((x0[None, :] >= 4) & (x0[None, :] + MED_TW + 4 <= w))


def median5_classes(w, h):
    """Interior tiles, border tiles, and the tiles one row off the interior test (y0 + 17 == h: an off-by-one
    there sends a tile whose last output row needs the replicate border to TMA's zero fill)"""
    inner = median5_interior(w, h)
    x0 = np.arange(cdiv(w, MED_TW)) * MED_TW
    y0 = np.arange(cdiv(h, MED_TH)) * MED_TH
    x_in = (x0 >= 4) & (x0 + MED_TW + 4 <= w)
    return {"tile_tma": int(inner.sum()), "tile_border": int((~inner).sum()),
            "tile_y0+17==h": int(((y0[:, None] + MED_TH + 1 == h) & x_in[None, :]).sum())}


# ---------------------------------------------------------------- sizes

SEED = 20261021
# the small stage sizes of tests/test_gpu_kernels.py, plus widths one below / above a tile
WARP_SMALL = [(16, 16), (37, 53), (65, 125), (97, 249), (130, 500), (41, 191), (57, 257)]
WARP_CUDA_SMALL = [(16, 16), (37, 53), (65, 125), (97, 249), (130, 500), (47, 97)]
# (h, w) of the median tests: h = 1 (mod 16) with w >= 260 puts a tile at y0 + 17 == h
MEDIAN_SIZES = [(16, 16), (37, 53), (65, 125), (97, 249), (130, 500), (33, 260), (49, 261), (65, 389), (34, 259)]


def grid_sizes(sms):
    """Image sizes whose tile count is at least 3 x SMs x (blocks per SM the thread limit allows), so that
    every block of a persistent grid walks at least three tiles whatever the occupancy; none is a multiple of
    its tile.  Returns {kernel: (h, w)}."""
    def size(tw, th, threads, w):
        need = 3 * sms * (2048 // threads)
        tx = cdiv(w, tw)
        return (cdiv(need, tx) - 1) * th + th // 2 + 1, w   # the last tile row is partly filled
    hw, ww = size(WP_TW, WP_TH, 128, 64 * 31 + 19)           # k_warp: 128 threads
    hc, wc = size(WC_TW, WC_TH, 256, 32 * 31 + 9)            # k_warp_cuda: 256 threads
    # k_median5: 256 threads, h = 1 (mod 16) and w >= 260 (the bottom interior test)
    tx = cdiv(128 * 21 + 45, MED_TW)
    hm = cdiv(3 * sms * 8, tx) * MED_TH + 1
    return {"warp": (hw, ww), "warp_cuda": (hc, wc), "median5": (hm, 128 * 21 + 45)}


# ---------------------------------------------------------------- flow fields

# regimes of a k_warp tile
SMOOTH, EDGE_R, EDGE_L, EDGE_B, EDGE_T, STEP, RW88, RW89, RH16, RH17, RH32, RH33, FAR = range(13)
N_REGIMES = 13


def _frac(rng, shape):
    """sub-pixel parts that stay in one 1/32 cell (so that a target integer position is hit exactly)"""
    return (rng.integers(0, 31, shape) + 0.25 + 0.5 * rng.random(shape)) / 32.0


def warp_field(h, w, seed, regimes=None):
    """(u1, u2) float32 for k_warp: every 64 x 8 tile gets a regime drawn at random (so that a block's walk
    meets every kind in every order); `regimes`, if given, restricts the draw.  The positions are built in
    fp64 as target source + 1 + a sub-pixel part and the flow is (position - pixel), rounded to fp32 once."""
    rng = np.random.default_rng(seed)
    ty_n, tx_n = cdiv(h, WP_TH), cdiv(w, WP_TW)
    choice = np.asarray(regimes if regimes is not None else range(N_REGIMES))
    reg = rng.choice(choice, size=(ty_n, tx_n))
    mx = np.zeros((ty_n * WP_TH, tx_n * WP_TW))
    my = np.zeros_like(mx)
    lx = np.arange(WP_TW)[None, :]
    ly = np.arange(WP_TH)[:, None]
    for ty in range(ty_n):
        for tx in range(tx_n):
            r = reg[ty, tx]
            x0, y0 = tx * WP_TW, ty * WP_TH
            X, Y = x0 + lx + 0 * ly, y0 + ly + 0 * lx
            # smooth flow: an integer shift, a sub-pixel part varying across the tile (each thread keeps one
            # part for its four rows, so that its sources stay vertically adjacent)
            sxs, sys_ = rng.integers(-6, 7), rng.integers(-4, 5)
            fx = ((rng.integers(0, 31) + 0.3 + 0.4 * np.sin(0.1 * lx + rng.random() * 6)) / 32.0) + 0 * ly
            fy = ((rng.integers(0, 31) + 0.3 + 0.4 * np.cos(0.1 * lx + rng.random() * 6)) / 32.0) + 0 * ly
            px, py = X + sxs + fx, Y + sys_ + fy
            if r in (EDGE_R, EDGE_L):
                # every column of the tile maps onto one of the seven columns at the edge: sx = w-6 .. w (right)
                # or -6 .. 0 (left), so the sources of the last allowed / first refused register-window column,
                # the partly-outside taps and the exact outside limit all occur
                c = rng.integers(-6, 1, WP_TW)[None, :] + 0 * ly
                px = (w + c if r == EDGE_R else c) + 1 + _frac(rng, (1, WP_TW))
            elif r in (EDGE_B, EDGE_T):
                # each thread's first source row sits at one of h-9 .. h-3 (bottom) or -6 .. 0 (top); its four
                # sources stay vertically adjacent
                c = rng.integers(-9, -2, (2, WP_TW)) if r == EDGE_B else rng.integers(-6, 1, (2, WP_TW))
                first = (h + c) if r == EDGE_B else c
                k = np.arange(WP_PX)[:, None]
                py = np.concatenate([first[0][None, :] + k, first[1][None, :] + k]) + 1 + _frac(rng, (1, WP_TW))
            elif r == STEP:
                # a step inside some threads' four rows: their sources stop being vertically adjacent
                jump = (rng.random((2, WP_TW)) < 0.5) * rng.integers(1, 4, (2, WP_TW))
                at = rng.integers(1, WP_PX, (2, WP_TW))
                k = np.arange(WP_PX)[:, None, None]
                d = (k >= at[None]) * jump[None]
                d = d.transpose(1, 0, 2).reshape(WP_TH, WP_TW)
                if rng.random() < 0.5:
                    py = py + d
                else:
                    px = px + d
            elif r in (RW88, RW89, RH16, RH17, RH32, RH33):
                # one pixel (not in the first column, which holds the leftmost source) far enough from the
                # others to make the window exactly that wide / tall
                px, py = X + sxs + 0.25 / 32 + 0 * fx, Y + sys_ + fy
                sx = X + sxs - 1
                sy = np.floor(py + 1 / 64.0).astype(np.int64) - 1
                i, j = rng.integers(0, WP_TH), rng.integers(1, WP_TW)
                if r in (RW88, RW89):
                    rx0 = ((sx.min() - 1) >> 2) << 2
                    target = (88 if r == RW88 else 89) - 5 + rx0    # rw = x1 + 5 - rx0
                    px[i, j] = target + 1 + 0.25 / 32
                else:
                    want = {RH16: 16, RH17: 17, RH32: 32, RH33: 33}[r]
                    target = sy.min() + want - 6                      # rh = y1 - y0 + 6
                    py[i, j] = target + 1 + fy[i, j]
            elif r == FAR:
                # sources wholly outside, by +-1e4, for a random part of the tile
                far = rng.random((WP_TH, WP_TW)) < rng.choice([0.3, 1.0])
                px = np.where(far, X + rng.choice([-1e4, 1e4]), px)
            mx[y0:y0 + WP_TH, x0:x0 + WP_TW] = px
            my[y0:y0 + WP_TH, x0:x0 + WP_TW] = py
    ys, xs = np.mgrid[0:h, 0:w]
    u1 = (mx[:h, :w] - xs).astype(F32)
    u2 = (my[:h, :w] - ys).astype(F32)
    return u1, u2


def warp_cuda_field(h, w, seed):
    """(u1, u2) float32 for k_warp_cuda: per 32 x 16 tile a smooth flow (integer positions included, which
    have 5 taps), a flow at an image edge, a box made exactly 64 / 65 wide or 48 / 49 tall by one pixel, or
    sources far outside"""
    rng = np.random.default_rng(seed)
    ty_n, tx_n = cdiv(h, WC_TH), cdiv(w, WC_TW)
    mx = np.zeros((ty_n * WC_TH, tx_n * WC_TW))
    my = np.zeros_like(mx)
    lx = np.arange(WC_TW)[None, :]
    ly = np.arange(WC_TH)[:, None]
    for ty in range(ty_n):
        for tx in range(tx_n):
            r = rng.integers(0, 8)
            x0, y0 = tx * WC_TW, ty * WC_TH
            X, Y = x0 + lx + 0 * ly, y0 + ly + 0 * lx
            f = rng.choice([0.0, 0.5, rng.random()])
            px = X + rng.integers(-5, 6) + f + 0.02 * np.sin(0.2 * (lx + ly))
            py = Y + rng.integers(-5, 6) + rng.choice([0.0, rng.random()]) + 0 * lx
            if r == 1:
                px = np.where(rng.random(px.shape) < 0.5, w - 1 + rng.integers(-2, 4, px.shape) + 0.0, rng.integers(-3, 2, px.shape) + 0.25)
            elif r == 2:
                py = np.where(rng.random(py.shape) < 0.5, h - 1 + rng.integers(-2, 4, py.shape) + 0.5, rng.integers(-3, 2, py.shape) + 0.0)
            elif r in (3, 4, 5, 6):
                # base: a pure shift with a non-integer position (4 taps: lo .. lo+3, box lo-1 .. lo+4)
                px = X + 3 + 0.5
                py = Y + 3 + 0.5
                # one pixel (not in the first row / column, which hold the smallest taps) moved so far that
                # the box is exactly that wide / tall: width = (lo + 3 + 1) - (lo_min - 1) + 1 for its lo
                i, j = rng.integers(1, WC_TH), rng.integers(1, WC_TW)
                lo_x, lo_y = np.ceil(px - 2).astype(np.int64), np.ceil(py - 2).astype(np.int64)
                if r in (3, 4):
                    lo = lo_x.min() + (64 if r == 3 else 65) - 6
                    px[i, j] = lo + 1.5   # ceil(lo + 1.5 - 2) = lo
                else:
                    lo = lo_y.min() + (48 if r == 5 else 49) - 6
                    py[i, j] = lo + 1.5
            elif r == 7:
                far = rng.random(px.shape) < 0.5
                px = np.where(far, X + rng.choice([-1e4, 1e4]), px)
            mx[y0:y0 + WC_TH, x0:x0 + WC_TW] = px
            my[y0:y0 + WC_TH, x0:x0 + WC_TW] = py
    ys, xs = np.mgrid[0:h, 0:w]
    return (mx[:h, :w] - xs).astype(F32), (my[:h, :w] - ys).astype(F32)
