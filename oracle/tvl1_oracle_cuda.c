/*
 * tvl1_oracle_cuda.c -- CPU restatement of the TVL1_SEMANTICS_CUDA mode of the flow stage: the algorithm of
 * cv::cuda::OpticalFlowDual_TVL1 (OpenCV 3.4.1, modules/cudaoptflow/src/tvl1flow.cpp and cuda/tvl1flow.cu) as
 * SURVEY.md Appendix B recalls it.  TEST INFRASTRUCTURE ONLY, same rules as tvl1_oracle.h.
 *
 * It shares everything the two classes share -- the pyramid sizes, the per-pixel iteration (estimateU +
 * estimateDualVariables = A.5, the fp32 error terms summed in fp64: iterate_ws with error_sum_mode 0) -- with
 * the CPU-class restatement by including it, and adds what differs:
 *   orc_resize_cuda  cuda::resize(INTER_LINEAR): no half-pixel offset, clamped reads of the second tap
 *   orc_warp_cuda    warpBackward: A = -0.5 cubic over ceil(w - 2) .. floor(w + 2), clamped reads, normalised
 *   orc_tvl1_calc_cuda  the flat loop with the sparse stop test, no median
 * Build flags as for libtvl1_oracle.so (-ffp-contract=off, no -ffast-math).
 */
#include "tvl1_oracle.c"

#include <limits.h>

#include "tvl1_oracle_cuda.h"

/* cuda::resize(src, dst, dsize, f, f, INTER_LINEAR): fx = (float)(1 / f) source pixels per destination pixel;
 * f = inv_scale when > 0, else dw / sw (and dh / sh) in fp64.  x1 is clamped like x2 so that no size reads
 * outside the source; the pyramid's sizes never need it. */
void orc_resize_cuda(const float* src, int sw, int sh, float* dst, int dw, int dh, double inv_scale)
{
    const double f_x = inv_scale > 0 ? inv_scale : (double)dw / sw;
    const double f_y = inv_scale > 0 ? inv_scale : (double)dh / sh;
    const float fx = (float)(1.0 / f_x), fy = (float)(1.0 / f_y);
#pragma omp parallel for schedule(static)
    for (int dy = 0; dy < dh; dy++) {
        const float src_y = (float)dy * fy;
        const int y1 = (int)floorf(src_y), y2 = y1 + 1;
        const int y1r = y1 < sh - 1 ? y1 : sh - 1, y2r = y2 < sh - 1 ? y2 : sh - 1;
        for (int dx = 0; dx < dw; dx++) {
            const float src_x = (float)dx * fx;
            const int x1 = (int)floorf(src_x), x2 = x1 + 1;
            const int x1r = x1 < sw - 1 ? x1 : sw - 1, x2r = x2 < sw - 1 ? x2 : sw - 1;
            float out = 0.f;
            out = out + src[(size_t)y1r * sw + x1r] * (((float)x2 - src_x) * ((float)y2 - src_y));
            out = out + src[(size_t)y1r * sw + x2r] * ((src_x - (float)x1) * ((float)y2 - src_y));
            out = out + src[(size_t)y2r * sw + x1r] * (((float)x2 - src_x) * (src_y - (float)y1));
            out = out + src[(size_t)y2r * sw + x2r] * ((src_x - (float)x1) * (src_y - (float)y1));
            dst[(size_t)dy * dw + dx] = out;
        }
    }
}

/* OpenCV's bicubicCoeff (A = -0.5), written as OpenCV writes it */
static inline float bicubic_coeff(float t)
{
    const float x = fabsf(t);
    if (x <= 1.0f) return x * x * (1.5f * x - 2.5f) + 1.0f;
    if (x < 2.0f) return x * (x * (-0.5f * x + 2.5f) - 4.0f) + 2.0f;
    return 0.0f;
}

/* float -> int, truncating, saturating, NaN -> 0 (the device's cvt.rzi.s32.f32) */
static inline int sat_int(float v)
{
    if (v != v) return 0;
    if (v >= 2147483648.0f) return INT_MAX;
    if (v <= -2147483648.0f) return INT_MIN;
    return (int)v;
}

static inline void taps(float v, int* lo, int* n)
{
    *lo = sat_int(ceilf(v - 2.0f));
    const long long k = (long long)sat_int(floorf(v + 2.0f)) - *lo + 1;
    *n = (int)(k < 0 ? 0 : (k > 5 ? 5 : k));
}

static inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

void orc_warp_cuda(const float* I0, const float* I1, const float* u1, const float* u2, int w, int h,
                   float* I1w, float* I1wx, float* I1wy, float* grad, float* rho_c)
{
    /* the I1x / I1y planes (A.3), read at clamped taps like the other plane */
    float* I1x = (float*)malloc(sizeof(float) * (size_t)w * h);
    float* I1y = (float*)malloc(sizeof(float) * (size_t)w * h);
    orc_centered_gradient(I1, w, h, I1x, I1y);
#pragma omp parallel for schedule(static)
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const size_t i = (size_t)y * w + x;
            const float wx = (float)x + u1[i], wy = (float)y + u2[i];
            int x0, nx, y0, ny;
            taps(wx, &x0, &nx);
            taps(wy, &y0, &ny);
            float sum = 0.0f, sumx = 0.0f, sumy = 0.0f, wsum = 0.0f;
            for (int a = 0; a < ny; a++) {
                const int cy = y0 + a;
                for (int b = 0; b < nx; b++) {
                    const int cx = x0 + b;
                    const float wgt = bicubic_coeff(wx - (float)cx) * bicubic_coeff(wy - (float)cy);
                    const size_t t = (size_t)clampi(cy, 0, h - 1) * w + clampi(cx, 0, w - 1);
                    sum += wgt * I1[t];
                    sumx += wgt * I1x[t];
                    sumy += wgt * I1y[t];
                    wsum += wgt;
                }
            }
            const float c = 1.0f / wsum;
            const float iw = sum * c, iwx = sumx * c, iwy = sumy * c;
            const float Ix2 = iwx * iwx;
            const float Iy2 = iwy * iwy;
            if (I1w) I1w[i] = iw;
            I1wx[i] = iwx;
            I1wy[i] = iwy;
            grad[i] = Ix2 + Iy2;
            rho_c[i] = ((iw - iwx * u1[i]) - iwy * u2[i]) - I0[i];
        }
    free(I1x);
    free(I1y);
}

int orc_tvl1_calc_cuda(const orc_params* p, int iterations, const unsigned char* I0, long pitch0,
                       const unsigned char* I1, long pitch1, int w, int h, float* u_out, float* v_out,
                       int* iters_out)
{
    if (!p || p->nscales <= 0 || p->nscales > ORC_MAX_LEVELS || w <= 0 || h <= 0) return -1;
    if (p->gamma != 0.0) return -3;
#ifdef _OPENMP
    if (p->nthreads > 0) omp_set_num_threads(p->nthreads);
#endif
    const int N = iterations > 0 ? iterations : 300;
    int ws[ORC_MAX_LEVELS + 1], hs[ORC_MAX_LEVELS + 1];
    float *I0s[ORC_MAX_LEVELS], *I1s[ORC_MAX_LEVELS], *u1s[ORC_MAX_LEVELS], *u2s[ORC_MAX_LEVELS];
    memset(I0s, 0, sizeof(I0s)); memset(I1s, 0, sizeof(I1s));
    memset(u1s, 0, sizeof(u1s)); memset(u2s, 0, sizeof(u2s));
    if (iters_out)
        for (int i = 0; i < p->nscales * p->warps; i++) iters_out[i] = -1;

    const size_t n0 = (size_t)w * h;
    int nscales = p->nscales;
    ws[0] = w; hs[0] = h;
    I0s[0] = (float*)malloc(n0 * 4); I1s[0] = (float*)malloc(n0 * 4);
    orc_convert_u8(I0, pitch0, w, h, I0s[0]);
    orc_convert_u8(I1, pitch1, w, h, I1s[0]);
    /* the level that falls below 16 px is built, then dropped (as in the CPU class) */
    for (int s = 1; s < nscales; s++) {
        ws[s] = orc_scaled_size(ws[s - 1], p->scale_step);
        hs[s] = orc_scaled_size(hs[s - 1], p->scale_step);
        if (ws[s] < 1 || hs[s] < 1) { nscales = s; break; }
        const size_t n = (size_t)ws[s] * hs[s];
        I0s[s] = (float*)malloc(n * 4); I1s[s] = (float*)malloc(n * 4);
        orc_resize_cuda(I0s[s - 1], ws[s - 1], hs[s - 1], I0s[s], ws[s], hs[s], p->scale_step);
        orc_resize_cuda(I1s[s - 1], ws[s - 1], hs[s - 1], I1s[s], ws[s], hs[s], p->scale_step);
        if (ws[s] < 16 || hs[s] < 16) { nscales = s; break; }
    }
    for (int s = 0; s < nscales; s++) {
        const size_t n = (size_t)ws[s] * hs[s];
        u1s[s] = (float*)calloc(n, 4); u2s[s] = (float*)calloc(n, 4);
    }
    float* I1wx = (float*)malloc(n0 * 4); float* I1wy = (float*)malloc(n0 * 4);
    float* grad = (float*)malloc(n0 * 4); float* rho_c = (float*)malloc(n0 * 4);
    float* p11 = (float*)malloc(n0 * 4); float* p12 = (float*)malloc(n0 * 4);
    float* p21 = (float*)malloc(n0 * 4); float* p22 = (float*)malloc(n0 * 4);
    iter_ws wsb;
    memset(&wsb, 0, sizeof(wsb));
    ws_reserve(&wsb, w, h);

    const float l_t = (float)(p->lambda * p->theta);
    const float taut = (float)(p->tau / p->theta);
    const float theta = (float)p->theta;

    for (int s = nscales - 1; s >= 0; --s) {
        const int lw = ws[s], lh = hs[s];
        const size_t n = (size_t)lw * lh;
        float *u1 = u1s[s], *u2 = u2s[s];
        const double eps = p->epsilon * p->epsilon * (double)(lw * lh);
        memset(p11, 0, n * 4); memset(p12, 0, n * 4);
        memset(p21, 0, n * 4); memset(p22, 0, n * 4);
        for (int warpings = 0; warpings < p->warps; ++warpings) {
            orc_warp_cuda(I0s[s], I1s[s], u1, u2, lw, lh, NULL, I1wx, I1wy, grad, rho_c);
            double error = DBL_MAX, prev = 0.0;
            int it = 0;
            for (; error > eps && it < N; ++it) {
                const int calc = p->epsilon > 0 && (it & 1) && prev < eps;
                const double e = iterate_ws(&wsb, I1wx, I1wy, grad, rho_c, u1, u2, p11, p12, p21, p22, lw, lh,
                                            l_t, theta, taut, 0);
                if (calc) { error = e; prev = error; }
                else { error = DBL_MAX; prev -= eps; }
            }
            if (iters_out) iters_out[s * p->warps + warpings] = it;
        }
        if (s == 0) break;
        const float up = (float)(1 / p->scale_step);
        orc_resize_cuda(u1, lw, lh, u1s[s - 1], ws[s - 1], hs[s - 1], 0.0);
        orc_resize_cuda(u2, lw, lh, u2s[s - 1], ws[s - 1], hs[s - 1], 0.0);
        const size_t nn = (size_t)ws[s - 1] * hs[s - 1];
        float *a = u1s[s - 1], *b = u2s[s - 1];
#pragma omp parallel for schedule(static)
        for (long i = 0; i < (long)nn; i++) { a[i] = a[i] * up; b[i] = b[i] * up; }
    }
    memcpy(u_out, u1s[0], n0 * 4);
    memcpy(v_out, u2s[0], n0 * 4);
    for (int s = 0; s < ORC_MAX_LEVELS; s++) { free(I0s[s]); free(I1s[s]); free(u1s[s]); free(u2s[s]); }
    free(I1wx); free(I1wy); free(grad); free(rho_c);
    free(p11); free(p12); free(p21); free(p22);
    ws_free(&wsb);
    return nscales;
}
