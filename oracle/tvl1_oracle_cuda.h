/*
 * tvl1_oracle_cuda.h -- CPU restatement of the TVL1_SEMANTICS_CUDA mode (cv::cuda::OpticalFlowDual_TVL1's
 * algorithm, SURVEY.md Appendix B).  TEST INFRASTRUCTURE ONLY, same rules as tvl1_oracle.h.  Built into
 * libtvl1_oracle_cuda.so together with the CPU-class restatement it shares its iteration with.
 */
#ifndef TVL1_ORACLE_CUDA_H
#define TVL1_ORACLE_CUDA_H

#include "tvl1_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* cuda::resize(INTER_LINEAR).  inv_scale > 0: by that factor (dw, dh = orc_scaled_size); else to dw x dh. */
void orc_resize_cuda(const float* src, int sw, int sh, float* dst, int dw, int dh, double inv_scale);

/* warpBackward + calcGradRho.  I1w may be NULL. */
void orc_warp_cuda(const float* I0, const float* I1, const float* u1, const float* u2, int w, int h,
                   float* I1w, float* I1wx, float* I1wy, float* grad, float* rho_c);

/* Whole solve in cv::cuda's algorithm.  Reads tau, lambda, theta, epsilon, scale_step, gamma (must be 0),
 * nscales, warps, nthreads of p; `iterations` (<= 0: 300) is the flat count per (level, warp).  iters_out as
 * for orc_tvl1_calc.  Returns levels used, or < 0 on error. */
int orc_tvl1_calc_cuda(const orc_params* p, int iterations, const unsigned char* I0, long pitch0,
                       const unsigned char* I1, long pitch1, int w, int h, float* u, float* v,
                       int* iters_out);

#ifdef __cplusplus
}
#endif
#endif
