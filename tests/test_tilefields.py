"""The flow fields of tests/test_gpu_tile_walk.py reach what they are meant to reach: every path and boundary of
k_warp, k_warp_cuda and k_median5, several times, at the sizes the GPU tests run (CPU only)."""
import numpy as np
import pytest

import tilefields as T
from tilefields import WARP_SMALL, WARP_CUDA_SMALL, MEDIAN_SIZES, SEED

SMS = 148   # the B200; the GPU tests size their grids from the device they run on

MIN_COUNT = 3


def test_geometry_restates_the_kernel_by_hand():
    """A few pixels of k_warp's source() worked out by hand, the window and TMA box choice, the column limits
    and the interior test of k_median5"""
    w, h = 200, 40
    u1 = np.zeros((h, w), np.float32)
    u2 = np.zeros((h, w), np.float32)
    sx, sy, out = T.source(w, h, u1, u2)
    assert sx[5, 7] == 6 and sy[5, 7] == 4 and not out[5, 7]
    u1[0, 0] = np.float32(w - 1 + 1 / 64)     # mx * 32 = 32 w - 31.5: a tie, rounds to even (32 w - 32) -> sx = w - 2
    u1[0, 1] = np.float32(w)                  # mx = w + 1 -> sx = w: outside exactly
    u1[0, 2] = np.float32(-6)                 # mx = -4 -> sx = -5: outside by one
    u1[0, 3] = np.float32(-6 + 1 / 32)        # mx = -3 + 1/32 -> sx = -4: sx + 4 == 0, outside exactly
    sx, sy, out = T.source(w, h, u1, u2)
    assert (sx[0, :4] == [w - 2, w, -5, -4]).all() and out[0, :4].tolist() == [False, True, True, True]
    z = np.zeros((h, w), np.float32)
    g = T.warp_geometry(w, h, z, z)
    # zero flow: sources (x - 1, y - 1).  Tile (0, 0): x0 = y0 = -1 -> rx0 = -4, ry0 = -2: scalar copies
    assert g["rw"][0, 0] == 62 + 4 + 4 + 1 and g["rh"][0, 0] == 6 + 4 + 2 + 1
    assert g["staged"][0, 0] and not g["tma"][0, 0]
    # tile (1, 1): x0 = 63 -> rx0 = 60, y0 = 7 -> ry0 = 6: inside the image, 13 rows -> the 16-row box
    assert g["rw"][1, 1] == 71 and g["rh"][1, 1] == 13 and g["tma"][1, 1] and g["box16"][1, 1]
    # a zero-flow thread is a column thread unless its sources reach x >= w - 3 or y >= h - 3 (or x, y < 0)
    col = g["column"]   # (tiles_y, tiles_x, 2 row groups, 64 columns)
    assert col[1, 0, 0, 5] and not col[0, 0, 0, 5]       # row group 0 of tile row 0 starts at sy = -1
    assert col[1, 3, 0, 5] and not col[1, 3, 0, 6]       # x = 197: sx = w - 4 is allowed; x = 198: w - 3 is not
    assert not T.median5_interior(260, 33).any()          # y0 + 18 <= h fails for the middle tile row ...
    assert T.median5_interior(260, 34)[1, 1] and not T.median5_interior(259, 34)[1, 1]   # ... and x0 + 132 <= w


def test_grid_sizes():
    """every block of a persistent grid walks >= 3 tiles; no size is a tile multiple; the median size has
    h = 1 (mod 16) and w >= 260"""
    s = T.grid_sizes(SMS)
    for k, (tw, th, thr) in {"warp": (64, 8, 128), "warp_cuda": (32, 16, 256), "median5": (128, 16, 256)}.items():
        h, w = s[k]
        assert T.cdiv(h, th) * T.cdiv(w, tw) >= 3 * SMS * (2048 // thr), k
        assert h % th and w % tw, k
    h, w = s["median5"]
    assert h % 16 == 1 and w >= 260


def _check(c, keys):
    low = {k: c[k] for k in keys if c[k] < MIN_COUNT}
    assert not low, "classes the field does not reach (or too rarely): %s of %s" % (low, c)


WARP_KEYS = ["tile_tma16", "tile_tma32", "tile_scalar_window", "tile_global", "tile_all_outside",
             "thread_column", "thread_perpixel_staged", "thread_perpixel_global",
             "column_sx_w-4", "column_sy_h-4", "column_sx_0", "column_sy_0", "px_sx_w-3", "px_sy_h-3",
             "px_outside_sx_w", "px_outside_sx+4_0", "px_outside_far", "px_partial", "px_inside",
             "tile_rw_88_tma", "tile_rw_89_global", "tile_rh_16_tma", "tile_rh_17_tma", "tile_rh_32_tma",
             "tile_rh_33_global"]


def test_warp_field_reaches_every_class():
    h, w = T.grid_sizes(SMS)["warp"]
    u1, u2 = T.warp_field(h, w, SEED)
    _check(T.warp_classes(w, h, u1, u2), WARP_KEYS)


@pytest.mark.parametrize("h,w", WARP_SMALL)
def test_warp_field_small_sizes(h, w):
    """the small sizes reach the paths their tiles allow (every regime needs a few tiles: counted over
    three seeds, the size of the GPU test's draw)"""
    tot = {}
    for s in range(3):
        u1, u2 = T.warp_field(h, w, SEED + s)
        for k, v in T.warp_classes(w, h, u1, u2).items():
            tot[k] = tot.get(k, 0) + v
    _check(tot, ["thread_column", "thread_perpixel_staged", "px_outside_sx_w", "px_outside_sx+4_0", "px_partial",
                 "column_sx_w-4", "px_sx_w-3"])


CUDA_KEYS = ["tile_staged", "tile_global", "px_5_taps", "tile_bw_64", "tile_bw_65", "tile_bh_48", "tile_bh_49"]


def test_warp_cuda_field_reaches_every_class():
    h, w = T.grid_sizes(SMS)["warp_cuda"]
    u1, u2 = T.warp_cuda_field(h, w, SEED)
    _check(T.warp_cuda_classes(w, h, u1, u2), CUDA_KEYS)


@pytest.mark.parametrize("h,w", WARP_CUDA_SMALL)
def test_warp_cuda_field_small_sizes(h, w):
    """5-tap pixels at every size, both window paths once there are enough tiles to draw from (counted over
    the three seeds of the GPU test)"""
    tot = {}
    for s in range(3):
        u1, u2 = T.warp_cuda_field(h, w, SEED + s)
        for k, v in T.warp_cuda_classes(w, h, u1, u2).items():
            tot[k] = tot.get(k, 0) + v
    _check(tot, ["px_5_taps"] + (["tile_staged", "tile_global"] if tot["tiles"] >= 20 else []))


def test_median_sizes_reach_the_bottom_interior_limit():
    h, w = T.grid_sizes(SMS)["median5"]
    c = T.median5_classes(w, h)
    _check(c, ["tile_tma", "tile_border", "tile_y0+17==h"])
    assert any(T.median5_classes(w, h)["tile_y0+17==h"] for h, w in MEDIAN_SIZES)
