/*
 * tvl1_oracle_ex.h -- CPU restatement of the rest of the classes' calc(I0, I1, flow): fp32 frames and
 * useInitialFlow, in both semantics (tvl1_calc_ex of include/tvl1_b200.h).  TEST INFRASTRUCTURE ONLY, same rules
 * as oracle/tvl1_oracle.h.  Built into libtvl1_oracle_ex.so together with the restatements under oracle/, whose
 * stages it reuses; those files and their entry points are left as they are, so the tests that pin them keep
 * checking the same code.
 */
#ifndef TVL1_ORACLE_EX_H
#define TVL1_ORACLE_EX_H

#include "../oracle/tvl1_oracle_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

#define ORC_FRAME_U8 0    /* TVL1_FRAME_U8 */
#define ORC_FRAME_F32 1   /* TVL1_FRAME_F32 */

/* A.2 for a CV_32FC1 frame: I.convertTo(CV_32F, 255.0), computed in fp64 and rounded once.  pitch in elements. */
void orc_convert_f32(const float* src, long pitch, int w, int h, float* dst);

/* One level of the initial flow's pyramid (SURVEY.md A.2a): resize(src, dst, Size(), step, step) -- INTER_AREA's
 * fast path at 0.5 -- then multiply(dst, Scalar::all(step)): RN_f32(x * (double)step). */
void orc_flow_down(const float* src, int sw, int sh, float* dst, int dw, int dh, double step);

/* The same in cv::cuda (SURVEY.md Appendix B): cuda::resize, then x * (float)step in fp32. */
void orc_flow_down_cuda(const float* src, int sw, int sh, float* dst, int dw, int dh, double step);

/* orc_tvl1_calc / orc_tvl1_calc_cuda with a frame type (pitches in elements of that type) and an initial flow
 * (u0, v0: dense w*h planes, both or neither; NULL: zero).  Return as those. */
int orc_tvl1_calc_ex(const orc_params* p, int frame_type, const void* I0, long pitch0, const void* I1, long pitch1,
                     int w, int h, const float* u0, const float* v0, float* u, float* v, int* iters_out);
int orc_tvl1_calc_cuda_ex(const orc_params* p, int iterations, int frame_type, const void* I0, long pitch0,
                          const void* I1, long pitch1, int w, int h, const float* u0, const float* v0, float* u,
                          float* v, int* iters_out);

#ifdef __cplusplus
}
#endif
#endif
