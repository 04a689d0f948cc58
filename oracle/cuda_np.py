"""NumPy restatement of the two stages in which the cv::cuda-semantics mode differs from the CPU class:
cuda::resize(INTER_LINEAR) and warpBackward (SURVEY.md Appendix B).

TEST INFRASTRUCTURE ONLY.  Written from the algorithm, independently of oracle/tvl1_oracle_cuda.c, so that the C
restatement is checked by a second hand (tests/test_cuda_semantics_reference.py).  Every operation is an fp32
NumPy operation in the order the algorithm states (NumPy never contracts to FMA).
"""
import numpy as np

F32 = np.float32


def resize_cuda(src, dw=None, dh=None, inv_scale=0.0):
    """cuda::resize(INTER_LINEAR): dst(x, y) from src_x = x * fx, fx = (float)(1 / f), no half-pixel offset,
    the second tap of each axis clamped to the last row / column, the four taps added to 0 in order."""
    src = np.asarray(src, F32)
    sh, sw = src.shape
    if inv_scale > 0:
        dw, dh = int(np.rint(sw * inv_scale)), int(np.rint(sh * inv_scale))
        fx = fy = F32(1.0 / inv_scale)
    else:
        fx, fy = F32(1.0 / (dw / sw)), F32(1.0 / (dh / sh))
    sx = np.arange(dw, dtype=F32) * fx
    sy = np.arange(dh, dtype=F32) * fy
    x1 = np.floor(sx).astype(np.int64)
    y1 = np.floor(sy).astype(np.int64)
    x2, y2 = x1 + 1, y1 + 1
    x1r, x2r = np.minimum(x1, sw - 1), np.minimum(x2, sw - 1)
    y1r, y2r = np.minimum(y1, sh - 1), np.minimum(y2, sh - 1)
    ax = (x2.astype(F32) - sx)[None, :]
    bx = (sx - x1.astype(F32))[None, :]
    ay = (y2.astype(F32) - sy)[:, None]
    by = (sy - y1.astype(F32))[:, None]
    out = np.zeros((dh, dw), F32)
    out = out + src[y1r][:, x1r] * (ax * ay)
    out = out + src[y1r][:, x2r] * (bx * ay)
    out = out + src[y2r][:, x1r] * (ax * by)
    out = out + src[y2r][:, x2r] * (bx * by)
    return out.astype(F32)


def bicubic_coeff(t):
    """OpenCV's bicubicCoeff, A = -0.5"""
    x = np.abs(np.asarray(t, F32))
    near = x * x * (F32(1.5) * x - F32(2.5)) + F32(1.0)
    far = x * (x * (F32(-0.5) * x + F32(2.5)) - F32(4.0)) + F32(2.0)
    return np.where(x <= F32(1.0), near, np.where(x < F32(2.0), far, F32(0.0))).astype(F32)


def _taps(v):
    lo = np.ceil(v - F32(2.0))
    hi = np.floor(v + F32(2.0))
    return lo.astype(np.int64), np.clip(hi.astype(np.int64) - lo.astype(np.int64) + 1, 0, 5)


def warp_cuda(I0, I1, u1, u2):
    """warpBackward + calcGradRho: (I1w, I1wx, I1wy, grad, rho_c).  Taps ceil(w - 2) .. floor(w + 2) per axis, rows
    outer, columns inner, zero-weight taps included; every read clamped into the image, the centred gradients of
    the taps from clamped neighbours; each sum times 1 / (sum of weights).  Flows must be finite."""
    I0, I1, u1, u2 = (np.asarray(a, F32) for a in (I0, I1, u1, u2))
    h, w = I0.shape
    P = np.pad(I1, 1, mode="edge")
    I1x = (F32(0.5) * (P[1:-1, 2:] - P[1:-1, :-2])).astype(F32)
    I1y = (F32(0.5) * (P[2:, 1:-1] - P[:-2, 1:-1])).astype(F32)
    wx = (np.arange(w, dtype=F32)[None, :] + u1).astype(F32)
    wy = (np.arange(h, dtype=F32)[:, None] + u2).astype(F32)
    x0, nx = _taps(wx)
    y0, ny = _taps(wy)
    s = np.zeros((h, w), F32)
    sx = np.zeros((h, w), F32)
    sy = np.zeros((h, w), F32)
    ws = np.zeros((h, w), F32)
    for a in range(5):
        cy = y0 + a
        ky = bicubic_coeff(wy - cy.astype(F32))
        yc = np.clip(cy, 0, h - 1)
        for b in range(5):
            on = (a < ny) & (b < nx)
            cx = x0 + b
            wgt = (bicubic_coeff(wx - cx.astype(F32)) * ky).astype(F32)
            xc = np.clip(cx, 0, w - 1)
            s = np.where(on, s + wgt * I1[yc, xc], s)
            sx = np.where(on, sx + wgt * I1x[yc, xc], sx)
            sy = np.where(on, sy + wgt * I1y[yc, xc], sy)
            ws = np.where(on, ws + wgt, ws)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = (F32(1.0) / ws).astype(F32)
    iw, iwx, iwy = (s * c).astype(F32), (sx * c).astype(F32), (sy * c).astype(F32)
    grad = (iwx * iwx + iwy * iwy).astype(F32)
    rho_c = (((iw - iwx * u1) - iwy * u2) - I0).astype(F32)
    return iw, iwx, iwy, grad, rho_c
