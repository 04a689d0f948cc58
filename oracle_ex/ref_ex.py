"""Second-hand restatements of fp32 frames and the initial flow (SURVEY.md A.2a, Appendix B), written independently
of oracle_ex/tvl1_oracle_ex.c so that the C restatement is checked by a second hand.

TEST INFRASTRUCTURE ONLY, same rules as oracle/tvl1_ref.py.  tvl1_calc_ex is the cv2 composition of the CPU class
(oracle/tvl1_ref.py's stages) with an fp32 frame's convertTo and the initial flow's pyramid through the real
cv2.resize + cv2.multiply.  flow_down_cuda is cv::cuda's step of that pyramid on oracle/cuda_np.py's resize.
"""
import numpy as np

from oracle import cuda_np
from oracle.tvl1_ref import FLT_MAX, _need_cv2, centered_gradient, iterate, iterate_gamma, warp

F32 = np.float32


def level0(frame):
    """convertTo(CV_32F): 8-bit frames as they are, fp32 frames times 255 (one fp32 rounding)"""
    frame = np.asarray(frame)
    if frame.dtype == np.uint8:
        return frame.astype(F32)
    if frame.dtype == np.float32:
        with np.errstate(over="ignore"):   # beyond FLT_MAX / 255: inf, as in OpenCV
            return (frame * F32(255.0)).astype(F32)
    raise ValueError("frames must be uint8 or float32")


def flow_down(u, step):
    """resize(u, Size(), step, step) then multiply(u, Scalar::all(step)), with cv2"""
    import cv2
    _need_cv2()
    return cv2.multiply(cv2.resize(u, None, fx=step, fy=step, interpolation=cv2.INTER_LINEAR), step)


def flow_down_cuda(u, step):
    """cuda::resize(u, Size(), step, step) then multiply by the float scalar: fp32 products"""
    return (cuda_np.resize_cuda(u, inv_scale=step) * F32(step)).astype(F32)


def tvl1_calc_ex(I0, I1, init=None, tau=0.25, lambda_=0.15, theta=0.3, nscales=5, warps=5, epsilon=0.01,
                 inner_iterations=30, outer_iterations=10, scale_step=0.8, median_filtering=5, gamma=0.0):
    """oracle/tvl1_ref.tvl1_calc for uint8 or float32 frames, starting from init = (u0, v0) (None: zero flow).
    Returns (u, v, iters[levels][warps])."""
    import cv2
    _need_cv2()
    I0s, I1s = [level0(I0)], [level0(I1)]
    u1s = u2s = None
    if init is not None:
        u1s, u2s = [np.asarray(init[0], F32)], [np.asarray(init[1], F32)]
    for s in range(1, nscales):
        a = cv2.resize(I0s[s - 1], None, fx=scale_step, fy=scale_step, interpolation=cv2.INTER_LINEAR)
        b = cv2.resize(I1s[s - 1], None, fx=scale_step, fy=scale_step, interpolation=cv2.INTER_LINEAR)
        if a.shape[1] < 16 or a.shape[0] < 16:
            nscales = s
            break
        I0s.append(a)
        I1s.append(b)
        if init is not None:
            u1s.append(flow_down(u1s[s - 1], scale_step))
            u2s.append(flow_down(u2s[s - 1], scale_step))
    l_t = F32(lambda_ * theta)
    taut = F32(tau / theta)
    th = F32(theta)
    if init is not None:
        u1, u2 = u1s[-1].copy(), u2s[-1].copy()
    else:
        u1, u2 = np.zeros_like(I0s[-1]), np.zeros_like(I0s[-1])
    u3 = np.zeros_like(I0s[-1])          # gamma != 0 only; zero whatever the initial flow
    iters = np.full((nscales, warps), -1, np.int32)
    for s in range(nscales - 1, -1, -1):
        I0, I1 = I0s[s], I1s[s]
        h, w = I0.shape
        scaled_eps = F32(epsilon * epsilon * (w * h))
        I1x, I1y = centered_gradient(I1)
        p11, p12, p21, p22, p31, p32 = (np.zeros_like(I0) for _ in range(6))
        for wi in range(warps):
            _, I1wx, I1wy, grad, rho_c = warp(I0, I1, I1x, I1y, u1, u2)
            error = FLT_MAX
            count = 0
            no = 0
            while error > scaled_eps and no < outer_iterations:
                if median_filtering > 1:
                    u1 = cv2.medianBlur(u1, median_filtering)
                    u2 = cv2.medianBlur(u2, median_filtering)
                ni = 0
                while error > scaled_eps and ni < inner_iterations:
                    if gamma != 0.0:
                        u1, u2, u3, p11, p12, p21, p22, p31, p32, e = iterate_gamma(
                            I1wx, I1wy, grad, rho_c, u1, u2, u3, p11, p12, p21, p22, p31, p32, l_t, th, taut, gamma)
                    else:
                        u1, u2, p11, p12, p21, p22, e = iterate(I1wx, I1wy, grad, rho_c, u1, u2,
                                                                p11, p12, p21, p22, l_t, th, taut)
                    error = F32(e)
                    count += 1
                    ni += 1
                no += 1
            iters[s, wi] = count
        if s == 0:
            break
        ph, pw = I0s[s - 1].shape
        up = F32(1 / scale_step)
        u1 = cv2.resize(u1, (pw, ph), interpolation=cv2.INTER_LINEAR) * up
        u2 = cv2.resize(u2, (pw, ph), interpolation=cv2.INTER_LINEAR) * up
        if gamma != 0.0:
            u3 = cv2.resize(u3, (pw, ph), interpolation=cv2.INTER_LINEAR)
    return u1, u2, iters
