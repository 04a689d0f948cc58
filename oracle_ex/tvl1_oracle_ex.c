/*
 * tvl1_oracle_ex.c -- fp32 frames and an initial flow for both restatements (see tvl1_oracle_ex.h).  TEST
 * INFRASTRUCTURE ONLY.  It includes the cv::cuda restatement (which includes the CPU-class one) and reuses their
 * stages; the two drivers below are orc_tvl1_calc and orc_tvl1_calc_cuda with level 0 and the coarsest flow set up
 * as calc(I0, I1, flow) with useInitialFlow does it (SURVEY.md A.2a and Appendix B).  The iteration, warp and median
 * are theirs.  Build flags as for libtvl1_oracle.so (-ffp-contract=off, no -ffast-math).
 */
#include "../oracle/tvl1_oracle_cuda.c"

#include "tvl1_oracle_ex.h"

void orc_convert_f32(const float* src, long pitch, int w, int h, float* dst)
{
    /* convertTo(CV_32F, 255.0): saturate_cast<float>(x * 255.0); the fp64 product is exact */
#pragma omp parallel for schedule(static)
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            dst[(size_t)y * w + x] = (float)((double)src[(size_t)y * pitch + x] * 255.0);
}

void orc_flow_down(const float* src, int sw, int sh, float* dst, int dw, int dh, double step)
{
    orc_resize_linear(src, sw, sh, dst, dw, dh, step);
    for (size_t i = 0; i < (size_t)dw * dh; i++) dst[i] = (float)((double)dst[i] * step);
}

void orc_flow_down_cuda(const float* src, int sw, int sh, float* dst, int dw, int dh, double step)
{
    orc_resize_cuda(src, sw, sh, dst, dw, dh, step);
    const float f = (float)step;
    for (size_t i = 0; i < (size_t)dw * dh; i++) dst[i] = dst[i] * f;
}

/* level 0 of both frames (by frame type), the image pyramid (cuda: cuda::resize) and the flow of every level: the
 * initial flow's pyramid, or zero at the coarsest level.  Returns the levels used. */
static int build_levels(const orc_params* p, int cuda, int frame_type, const void* I0, long pitch0, const void* I1,
                        long pitch1, int w, int h, const float* u0, const float* v0, int* ws, int* hs, float** I0s,
                        float** I1s, float** u1s, float** u2s)
{
    const size_t n0 = (size_t)w * h;
    int nscales = p->nscales;
    ws[0] = w; hs[0] = h;
    I0s[0] = (float*)malloc(n0 * 4); I1s[0] = (float*)malloc(n0 * 4);
    if (frame_type == ORC_FRAME_F32) {
        orc_convert_f32((const float*)I0, pitch0, w, h, I0s[0]);
        orc_convert_f32((const float*)I1, pitch1, w, h, I1s[0]);
    } else {
        orc_convert_u8((const unsigned char*)I0, pitch0, w, h, I0s[0]);
        orc_convert_u8((const unsigned char*)I1, pitch1, w, h, I1s[0]);
    }
    u1s[0] = (float*)calloc(n0, 4); u2s[0] = (float*)calloc(n0, 4);
    if (u0) { memcpy(u1s[0], u0, n0 * 4); memcpy(u2s[0], v0, n0 * 4); }
    /* the level that falls below 16 px is built, then dropped; the flow is resized after that test */
    for (int s = 1; s < nscales; s++) {
        ws[s] = orc_scaled_size(ws[s - 1], p->scale_step);
        hs[s] = orc_scaled_size(hs[s - 1], p->scale_step);
        if (ws[s] < 1 || hs[s] < 1) { nscales = s; break; }
        const size_t n = (size_t)ws[s] * hs[s];
        I0s[s] = (float*)malloc(n * 4); I1s[s] = (float*)malloc(n * 4);
        void (*rs)(const float*, int, int, float*, int, int, double) = cuda ? orc_resize_cuda : orc_resize_linear;
        rs(I0s[s - 1], ws[s - 1], hs[s - 1], I0s[s], ws[s], hs[s], p->scale_step);
        rs(I1s[s - 1], ws[s - 1], hs[s - 1], I1s[s], ws[s], hs[s], p->scale_step);
        if (ws[s] < 16 || hs[s] < 16) { nscales = s; break; }
        u1s[s] = (float*)calloc(n, 4); u2s[s] = (float*)calloc(n, 4);
        if (u0) {
            void (*fd)(const float*, int, int, float*, int, int, double) = cuda ? orc_flow_down_cuda : orc_flow_down;
            fd(u1s[s - 1], ws[s - 1], hs[s - 1], u1s[s], ws[s], hs[s], p->scale_step);
            fd(u2s[s - 1], ws[s - 1], hs[s - 1], u2s[s], ws[s], hs[s], p->scale_step);
        }
    }
    return nscales;
}

int orc_tvl1_calc_ex(const orc_params* p, int frame_type, const void* I0, long pitch0, const void* I1, long pitch1,
                     int w, int h, const float* u0, const float* v0, float* u_out, float* v_out, int* iters_out)
{
    if (!p || p->nscales <= 0 || p->nscales > ORC_MAX_LEVELS || w <= 0 || h <= 0) return -1;
    if (frame_type != ORC_FRAME_U8 && frame_type != ORC_FRAME_F32) return -1;
    if ((u0 == NULL) != (v0 == NULL)) return -1;
    if (p->median_filtering != 1 && p->median_filtering != 3 && p->median_filtering != 5) return -3;
#ifdef _OPENMP
    if (p->nthreads > 0) omp_set_num_threads(p->nthreads);
#endif
    cubic_tab_init();

    int ws[ORC_MAX_LEVELS + 1], hs[ORC_MAX_LEVELS + 1];
    float *I0s[ORC_MAX_LEVELS], *I1s[ORC_MAX_LEVELS], *u1s[ORC_MAX_LEVELS], *u2s[ORC_MAX_LEVELS];
    memset(I0s, 0, sizeof(I0s)); memset(I1s, 0, sizeof(I1s));
    memset(u1s, 0, sizeof(u1s)); memset(u2s, 0, sizeof(u2s));
    if (iters_out)
        for (int i = 0; i < p->nscales * p->warps; i++) iters_out[i] = -1;
    const size_t n0 = (size_t)w * h;
    const int nscales = build_levels(p, 0, frame_type, I0, pitch0, I1, pitch1, w, h, u0, v0, ws, hs, I0s, I1s, u1s, u2s);

    float* I1x = (float*)malloc(n0 * 4); float* I1y = (float*)malloc(n0 * 4);
    float* I1wx = (float*)malloc(n0 * 4); float* I1wy = (float*)malloc(n0 * 4);
    float* grad = (float*)malloc(n0 * 4); float* rho_c = (float*)malloc(n0 * 4);
    float* p11 = (float*)malloc(n0 * 4); float* p12 = (float*)malloc(n0 * 4);
    float* p21 = (float*)malloc(n0 * 4); float* p22 = (float*)malloc(n0 * 4);
    float* med = (float*)malloc(n0 * 4);
    /* gamma != 0: u3 starts at zero whatever the initial flow (it is not part of calc's flow argument) */
    const int use_gamma = p->gamma != 0.0;
    const float gamma = (float)p->gamma;
    float* u3s[ORC_MAX_LEVELS];
    memset(u3s, 0, sizeof(u3s));
    float *p31 = NULL, *p32 = NULL;
    if (use_gamma) {
        for (int s = 0; s < nscales; s++) u3s[s] = (float*)calloc((size_t)ws[s] * hs[s], 4);
        p31 = (float*)malloc(n0 * 4); p32 = (float*)malloc(n0 * 4);
    }
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
        const float scaledEpsilon = (float)(p->epsilon * p->epsilon * (double)(lw * lh));
        orc_centered_gradient(I1s[s], lw, lh, I1x, I1y);
        memset(p11, 0, n * 4); memset(p12, 0, n * 4);
        memset(p21, 0, n * 4); memset(p22, 0, n * 4);
        if (use_gamma) { memset(p31, 0, n * 4); memset(p32, 0, n * 4); }
        for (int warpings = 0; warpings < p->warps; ++warpings) {
            orc_warp(I0s[s], I1s[s], I1x, I1y, u1, u2, lw, lh, NULL, I1wx, I1wy, grad, rho_c);
            float error = FLT_MAX;
            int count = 0;
            for (int n_outer = 0; error > scaledEpsilon && n_outer < p->outer_iterations; ++n_outer) {
                if (p->median_filtering == 5) {
                    orc_median5(u1, lw, lh, med); memcpy(u1, med, n * 4);
                    orc_median5(u2, lw, lh, med); memcpy(u2, med, n * 4);
                } else if (p->median_filtering == 3) {
                    orc_median3(u1, lw, lh, med); memcpy(u1, med, n * 4);
                    orc_median3(u2, lw, lh, med); memcpy(u2, med, n * 4);
                }
                for (int n_inner = 0; error > scaledEpsilon && n_inner < p->inner_iterations; ++n_inner) {
                    const double e = use_gamma
                        ? iterate_ws_g(&wsb, I1wx, I1wy, grad, rho_c, u1, u2, u3s[s], p11, p12, p21, p22,
                                       p31, p32, lw, lh, l_t, theta, taut, gamma, p->error_sum_mode)
                        : iterate_ws(&wsb, I1wx, I1wy, grad, rho_c, u1, u2, p11, p12, p21, p22, lw, lh, l_t, theta,
                                     taut, p->error_sum_mode);
                    error = (float)e;
                    ++count;
                }
            }
            if (iters_out) iters_out[s * p->warps + warpings] = count;
        }
        if (s == 0) break;
        const float up = (float)(1 / p->scale_step);
        orc_resize_linear(u1, lw, lh, u1s[s - 1], ws[s - 1], hs[s - 1], 0.0);
        orc_resize_linear(u2, lw, lh, u2s[s - 1], ws[s - 1], hs[s - 1], 0.0);
        if (use_gamma) orc_resize_linear(u3s[s], lw, lh, u3s[s - 1], ws[s - 1], hs[s - 1], 0.0);
        const size_t nn = (size_t)ws[s - 1] * hs[s - 1];
        float *a = u1s[s - 1], *b = u2s[s - 1];
#pragma omp parallel for schedule(static)
        for (long i = 0; i < (long)nn; i++) { a[i] = a[i] * up; b[i] = b[i] * up; }
    }
    memcpy(u_out, u1s[0], n0 * 4);
    memcpy(v_out, u2s[0], n0 * 4);

    for (int s = 0; s < ORC_MAX_LEVELS; s++) { free(I0s[s]); free(I1s[s]); free(u1s[s]); free(u2s[s]); free(u3s[s]); }
    free(I1x); free(I1y); free(I1wx); free(I1wy); free(grad); free(rho_c);
    free(p11); free(p12); free(p21); free(p22); free(med);
    free(p31); free(p32);
    ws_free(&wsb);
    return nscales;
}

int orc_tvl1_calc_cuda_ex(const orc_params* p, int iterations, int frame_type, const void* I0, long pitch0,
                          const void* I1, long pitch1, int w, int h, const float* u0, const float* v0, float* u_out,
                          float* v_out, int* iters_out)
{
    if (!p || p->nscales <= 0 || p->nscales > ORC_MAX_LEVELS || w <= 0 || h <= 0) return -1;
    if (frame_type != ORC_FRAME_U8 && frame_type != ORC_FRAME_F32) return -1;
    if ((u0 == NULL) != (v0 == NULL)) return -1;
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
    const int nscales = build_levels(p, 1, frame_type, I0, pitch0, I1, pitch1, w, h, u0, v0, ws, hs, I0s, I1s, u1s, u2s);

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
