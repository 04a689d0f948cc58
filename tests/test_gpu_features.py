"""N4: the feature pre-alignment in front of the flow stage (reference src/features.cpp:46-167,
src/optflow.cpp:366-377, 411-444) against the same pipeline built from the CPU classes of the installed
cv2 (oracle/features_ref.py).  Keypoints and RANSAC draws are not reproducible across implementations, so
the comparison is between TRANSFORMS; the warps are compared with cv2.warpAffine directly."""
import numpy as np
import pytest

from fibsem_optflow_b200 import synth

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")


def moved_pair(h, w, seed, angle_deg, zoom, tx, ty):
    """(frame0, frame1, A): frame1(x) = frame0(A x), i.e. A maps frame1 coordinates to frame0 coordinates"""
    m = 120
    c = synth.to_u8(synth.texture(h + 2 * m, w + 2 * m, seed, 2.0, coarse=8))
    th = np.deg2rad(angle_deg)
    A = np.array([[zoom * np.cos(th), -zoom * np.sin(th), tx], [zoom * np.sin(th), zoom * np.cos(th), ty]])
    M = A.copy()
    M[:, 2] += m                                              # frame0(x) = canvas(x + m)
    f0 = np.ascontiguousarray(c[m:m + h, m:m + w])
    f1 = cv2.warpAffine(c, M, (w, h), flags=cv2.INTER_CUBIC | cv2.WARP_INVERSE_MAP)
    return f0, f1, A


@pytest.mark.parametrize("case", [(0.4, 1.02, 7.3, -4.6), (-1.1, 0.97, -12.0, 9.5), (0.0, 1.0, 3.25, 2.5)])
def test_find_alignment_recovers_transform(gpu, case):
    from oracle import features_ref as F
    h, w = 900, 1100
    f0, f1, A = moved_pair(h, w, 5, *case)
    s = gpu.Solver(gpu.default_params())
    aff, nm, ng = s.find_alignment(f1, f0)                   # as solve_rois calls it: (frame1, frame0)
    ref, rnm, rng_ = F.find_alignment(f1, f0)
    assert ng > 50 and nm > 1000, (nm, ng)
    e_true, e_ref, e_cv = F.corner_error(aff, A, w, h), F.corner_error(aff, ref, w, h), F.corner_error(ref, A, w, h)
    # cv2's own pipeline (ORB + BF + findHomography, top 2x3 of the homography) lands within 0.3 .. 1.5 px of
    # the truth at the frame corners on these pairs (measured: 1.40, 1.51, 0.28); this one must do as well
    assert e_cv < 2.0, e_cv
    assert e_true < max(1.0, e_cv), (e_true, e_cv, aff, A)
    assert e_ref < 2.5, e_ref
    # reproducible run to run (fixed-seed RANSAC, order-independent keypoint selection)
    aff2, _, _ = s.find_alignment(f1, f0)
    assert np.array_equal(aff, aff2)
    s.close()


def test_find_alignment_falls_back_to_identity(gpu):
    rng = np.random.default_rng(2)
    flat = np.full((400, 500), 90, np.uint8)
    noise = rng.integers(0, 255, size=(400, 500), dtype=np.uint8)
    s = gpu.Solver(gpu.default_params())
    aff, nm, ng = s.find_alignment(flat, noise)               # no corners in a flat frame
    assert np.array_equal(aff, np.array([[1, 0, 0], [0, 1, 0]], np.float32)) and ng == 0
    other = rng.integers(0, 255, size=(400, 500), dtype=np.uint8)
    aff, nm, ng = s.find_alignment(noise, other)              # unrelated frames: too few good matches, or rejected
    assert np.array_equal(aff, np.array([[1, 0, 0], [0, 1, 0]], np.float32))
    s.close()


@pytest.mark.parametrize("aff", [[[1.02, -0.007, 7.3], [0.007, 1.02, -4.6]], [[0.95, 0.05, -20.5], [-0.04, 1.1, 13.25]],
                                 [[1, 0, 0], [0, 1, 0]]])
def test_warp_affine_matches_cv2(gpu, aff):
    rng = np.random.default_rng(7)
    img = rng.integers(0, 256, size=(301, 407), dtype=np.uint8)
    A = np.array(aff, np.float32)
    want = cv2.warpAffine(img, A.astype(np.float64), (390, 280), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    got = gpu.warp_affine(img, A, (390, 280))
    assert np.array_equal(got, want), int(np.abs(got.astype(int) - want).max())
    # pitched source and destination (GpuMat rows are padded): the same pixels, the padding neither read nor written
    for sp, dp in [(512, 390), (407, 391), (408, 512)]:
        assert np.array_equal(gpu.warp_affine(img, A, (390, 280), spitch=sp, dpitch=dp), want), (sp, dp)
    plane = (rng.standard_normal((301, 407)) * 100).astype(np.float32)
    want = cv2.warpAffine(plane, A.astype(np.float64), (390, 280), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    got = gpu.warp_affine(plane, A, (390, 280))
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-4)
    for sp, dp in [(416, 390), (407, 393)]:
        assert np.array_equal(gpu.warp_affine(plane, A, (390, 280), spitch=sp, dpitch=dp), got), (sp, dp)


def _composition(orc, f0, f1, aff, output_type, tv):
    """solve_rois + solve_wrapper of the reference (src/optflow.cpp:366-377, 411-444, 471-473) for one
    whole-frame roi, from cv2's warpAffine and the TV-L1 oracle, given the affine"""
    from oracle import features_ref as F
    h, w = f0.shape
    moved = F.warp_affine(f1, aff, (w, h))
    u, v, _, _ = orc.tvl1_calc(f0, moved, **tv)
    mx = u + np.arange(w, dtype=np.float32)[None, :]
    my = v + np.arange(h, dtype=np.float32)[:, None]
    mx, my = F.warp_affine(mx, aff, (w, h)), F.warp_affine(my, aff, (w, h))
    if output_type == "flow":
        mx = mx - np.arange(w, dtype=np.float32)[None, :]
        my = my - np.arange(h, dtype=np.float32)[:, None]
    mx = np.where(moved <= 1, np.float32(0), mx)
    my = np.where(moved <= 1, np.float32(0), my)
    return moved, mx, my


@pytest.mark.parametrize("output_type", ["map", "flow", "random_points"])
def test_solve_rois_with_features(gpu, orc, output_type):
    """api.solve_rois on a pair without roi: the reference forces the pre-alignment (src/optflow.cpp:366).
    Frame1 moved by cv2.warpAffine with the same affine, the oracle's flow, cv2's map warp = the reference's
    composition; the match q's follow the `features` branch of random_points (:544-550)."""
    from fibsem_optflow_b200 import api
    h, w = 420, 560
    f0, f1, A = moved_pair(h, w, 11, 0.5, 1.01, 5.3, -3.6)
    f1[:, :6] = 0                                              # something for the frame1 <= 1 mask
    tv = {"lambda": 0.15, "nscales": 4}
    args = dict(tv, output_type=output_type, scale=1.0, npoints=9, debug=True)
    im = {"pId": "a", "qId": "b", "pGroupId": "1.0", "qGroupId": "2.0"}
    aff = api.find_alignment(f1, f0, im, args)
    assert not np.array_equal(aff, np.array([[1, 0, 0], [0, 1, 0]], np.float32))
    out = api.solve_rois(f0, f1, {"default": [0, 0, w, h]}, im, args, seed=-1)
    gx, gy = out["default"]
    moved, wx, wy = _composition(orc, f0, f1, aff, output_type, tv)
    assert np.array_equal(gpu.warp_affine(f1, aff, (w, h)), moved)
    # cv2's fp32 warpAffine sums its four products in another order (SIMD): a few ulp of a ~500 coordinate
    np.testing.assert_allclose(gx, wx, rtol=0, atol=5e-4)
    np.testing.assert_allclose(gy, wy, rtol=0, atol=5e-4)
    assert np.array_equal(gx == 0, wx == 0)
    if output_type == "random_points":
        rec = args["point_matches"][0]
        assert rec["pId"] == "a" and rec["qGroupId"] == "2.0"
        m = rec["matches"]
        # the debug stream starts as an unseeded process does, i.e. as srand(1); the oracle's own seed=-1 would
        # continue this process's libc rand() state, which earlier tests (test_abi's srand / rand) have moved
        want = orc.random_points(f0, moved, gx, gy, roi0=(0, 0), roi1=(0, 0), scale=1.0, npoints=9, seed=1)
        pos = want[5]
        assert m["p"][0] == want[0].tolist() and m["p"][1] == want[1].tolist()
        # q = (map(pos) + roi1) * inv_scale: no pos term, the planes hold a map
        assert m["q"][0] == [float(gx[y, x]) for x, y in pos] and m["q"][1] == [float(gy[y, x]) for x, y in pos]
        assert m["w"] == [1] * 9
    api.release_solvers()


def test_solve_rois_features_precedence_and_realign(gpu):
    """an explicit false at either level wins over a true at the other (src/optflow.cpp:323-338); with two
    roi keys the second key aligns the already aligned frame again, as the reference's loop does"""
    from fibsem_optflow_b200 import api
    h, w = 420, 560
    f0, f1, A = moved_pair(h, w, 12, 0.0, 1.0, 4.0, 2.0)
    args = {"lambda": 0.15, "nscales": 3, "output_type": "flow", "features": True}
    off = api.solve_rois(f0, f1, {"top": [0, 0, w, 64]}, {"features": False}, dict(args))
    on = api.solve_rois(f0, f1, {"top": [0, 0, w, 64]}, {}, dict(args))
    # without the alignment the strip's flow carries the 4 px shift, with it only the residual
    assert abs(np.median(off["top"][0])) > 3.0 and abs(np.median(on["top"][0][:, 40:-40])) > 3.0
    raw = api.solve_wrapper(f0[:64], gpu.warp_affine(f1, api.find_alignment(f1, f0, {}, args), (w, h))[:64], {},
                            dict(args, output_type="flow"))
    assert abs(np.median(raw[0][:, 40:-40])) < 0.5
    both = api.solve_rois(f0, f1, {"top": [0, 0, w, 64], "bottom": [0, h - 64, w, 64]}, {}, dict(args))
    assert set(both) == {"top", "bottom"}
    api.release_solvers()
