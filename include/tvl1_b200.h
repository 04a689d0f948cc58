/*
 * tvl1_b200.h -- C ABI of the B200-native TV-L1 flow stage.
 *
 * Drop-in boundary for fibsem-optflow's flow stage.  The reference has no FFI of
 * its own; the seam is two C++ functions, and every entry point below names the
 * reference interface it replaces (paths relative to the reference repo):
 *
 *   tvl1_default_params / tvl1_params   <- generate_TV_args   src/optflow.cpp:500-514
 *   tvl1_create / tvl1_destroy          <- OpticalFlowDual_TVL1::create, called per
 *                                          solve in TVL1_solve   src/optflow.cpp:518
 *   tvl1_calc_u8 / tvl1_calc_u8_host    <- TVL1_solve (solver->calc)
 *                                          src/optflow.h:31, src/optflow.cpp:516-520
 *   tvl1_mask_flow_u8                   <- threshold + setTo in solve_wrapper
 *                                          src/optflow.cpp:471-473
 *   tvl1_sample_matches[_host]          <- mask build src/optflow.cpp:488-493 and
 *                                          random_points src/optflow.h:33,
 *                                          src/optflow.cpp:522-572
 *
 *   tvl1_finish_flow_u8                 <- map grid + mask of solve_wrapper   src/optflow.cpp:445-473
 *   tvl1_find_alignment                 <- find_alignment   src/features.cpp:46-167
 *   tvl1_warp_affine_u8 / _f32          <- cv::cuda::warpAffine   src/optflow.cpp:374, 431-432
 *   tvl1_prescale_u8                    <- the loader's cv::resize   src/optflow.cpp:111,124
 *   tvl1_stack_run                      <- the pair loop of from_file   src/optflow.cpp:75-178
 *
 * NUMERICS: the solver computes what OpenCV's CPU class cv::DualTVL1OpticalFlow computes (cubic
 * 1/32-px remap, 5x5 median per outer iteration, stop test every iteration), bit for bit against
 * the CPU restatement in oracle/.  The reference BINARY calls cv::cuda::OpticalFlowDual_TVL1
 * (src/optflow.cpp:518: flat loop, no median, another bicubic, fast-math), so outputs are not
 * bit-comparable with that binary's for the same job; see DESIGN.md section 1.
 *
 * Conventions: plain pointers and sizes, no C++ or torch types.  "d_" pointers are
 * device memory on the handle's device, "h_" pointers are host memory.  8-bit images
 * are single channel rows with a byte pitch (the reference passes GpuMat ROI views,
 * src/optflow.cpp:362,382).  Flow is returned PLANAR (u then v), fp32, with a byte
 * pitch -- the reference splits OpenCV's interleaved result immediately
 * (src/optflow.cpp:404).  All functions return TVL1_OK (0) or a negative status and
 * never throw; tvl1_last_error() describes the last failure on the calling thread.
 * A handle is bound to one device and must be used by one host thread at a time.
 */
#ifndef TVL1_B200_H
#define TVL1_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TVL1_OK 0
#define TVL1_ERR_INVALID (-1)   /* bad argument */
#define TVL1_ERR_CUDA (-2)      /* CUDA runtime error, see tvl1_last_error() */
#define TVL1_ERR_UNSUPPORTED (-3)
#define TVL1_ERR_NOMEM (-4)

#define TVL1_MAX_LEVELS 32
#define TVL1_MAX_WARPS 64

typedef struct tvl1_handle tvl1_handle;

/* The ten keys of generate_TV_args (src/optflow.cpp:503-512) plus the CPU-class
 * parameters OpenCV's DualTVL1 has and the cv::cuda API lacks (SURVEY.md T3/T4). */
typedef struct tvl1_params {
    double tau;             /* 0.25 */
    double lambda;          /* reference wrapper default 0.05 (OpenCV 0.15) */
    double theta;           /* 0.3 */
    double epsilon;         /* 0.01 */
    double scale_step;      /* "scaleStep", 0.8 */
    double gamma;           /* 0; != 0 adds OpenCV's third channel (u3, p31, p32): supported, on a plain two-launch iteration */
    int nscales;            /* reference wrapper default 10 (OpenCV 5) */
    int warps;              /* 5 */
    int iterations;         /* 300; used when inner/outer are <= 0:
                               inner = 30, outer = ceil(iterations / 30) */
    int inner_iterations;   /* <= 0: derive from iterations */
    int outer_iterations;   /* <= 0: derive from iterations */
    int median_filtering;   /* 5 (CPU class); 3; 1 = off */
    int use_initial_flow;   /* read by the reference but never forwarded
                               (src/optflow.cpp:512,518); must be 0 */
    int reserved[3];
} tvl1_params;

/* Iteration counts and stage times of the last calc. */
typedef struct tvl1_stats {
    int levels;                                     /* pyramid levels actually used */
    int warps;
    int width[TVL1_MAX_LEVELS], height[TVL1_MAX_LEVELS];
    int iters[TVL1_MAX_LEVELS * TVL1_MAX_WARPS];    /* [level * warps + warp], level 0 = finest */
    int outer[TVL1_MAX_LEVELS * TVL1_MAX_WARPS];    /* outer iterations (median passes) run */
    long long total_iterations;
    long long px_iterations;                        /* sum over (level,warp) of px * iters */
    double algorithmic_bytes;                       /* BASELINE.md section 4 byte model */
    float ms_total, ms_pyramid, ms_warp, ms_iterate, ms_median, ms_other;  /* CUDA events on
                                                       the solve's stream */
    float ms_iterate_level[TVL1_MAX_LEVELS];        /* ms_iterate split by level */
    long long launches;                             /* kernels launched by the last calc */
} tvl1_stats;

const char* tvl1_version(void);
const char* tvl1_last_error(void);

/* Reference-wrapper defaults of generate_TV_args (src/optflow.cpp:503-512). */
void tvl1_default_params(tvl1_params* p);

int tvl1_create(const tvl1_params* p, int device, tvl1_handle** out);
void tvl1_destroy(tvl1_handle* h);
int tvl1_set_params(tvl1_handle* h, const tvl1_params* p);
/* Tuning knobs that never change results.  "fused_min_px": pyramid levels with at least this
 * many pixels run the temporally blocked two-iteration passes (default 0 = always;
 * 1e18 = never).  "multi_iter": smaller levels run all inner iterations of an outer iteration in one
 * cooperative launch (default 1; 0 = one launch per iteration).  "coop_outer": the larger levels run
 * the inner loop of an outer iteration (two-iteration and single passes) in one cooperative launch
 * (default 1; 0 = host-driven launch slots). */
int tvl1_set_option(tvl1_handle* h, const char* key, double value);
/* per-stage CUDA-event timing (ms_pyramid, ms_warp, ms_iterate[_level], ms_median, ms_other of
 * tvl1_stats; two events per stage span).  Default off: only ms_total is measured. */
int tvl1_set_timing(tvl1_handle* h, int enabled);

/* Flow from frame0 to frame1 (device pointers).  stream is a cudaStream_t (may be 0).
 * Returns after the result is complete on `stream` and the stop test has been resolved
 * (the call synchronises the stream: the iteration count is data dependent). */
int tvl1_calc_u8(tvl1_handle* h, const uint8_t* d_frame0, size_t pitch0,
                 const uint8_t* d_frame1, size_t pitch1, int width, int height,
                 float* d_u, float* d_v, size_t pitch_out, void* stream, tvl1_stats* stats);

/* Same with host buffers: H2D of both frames, solve, D2H of both planes. */
int tvl1_calc_u8_host(tvl1_handle* h, const uint8_t* h_frame0, size_t pitch0,
                      const uint8_t* h_frame1, size_t pitch1, int width, int height,
                      float* h_u, float* h_v, size_t pitch_out, tvl1_stats* stats);

/* flow = 0 where frame1 <= 1 (src/optflow.cpp:471-473). */
int tvl1_mask_flow_u8(tvl1_handle* h, const uint8_t* d_frame1, size_t pitch1, int width,
                      int height, float* d_u, float* d_v, size_t pitch_out, void* stream);

/* The post-processing of solve_wrapper in one pass (src/optflow.cpp:445-473): with add_grid != 0
 * ("output_type": "map") the coordinate grid is added to the flow, u += x, v += y -- the reference
 * builds that grid in a host double loop and uploads it (:451-465) --, then flow = 0 where
 * frame1 <= 1 (:471-473).  add_grid == 0 is tvl1_mask_flow_u8; add_grid < 0 SUBTRACTS the grid (the "flow"
 * output after a feature pre-alignment, :434-438); d_frame1 == NULL skips the mask. */
int tvl1_finish_flow_u8(tvl1_handle* h, const uint8_t* d_frame1, size_t pitch1, int width,
                        int height, float* d_u, float* d_v, size_t pitch_out, int add_grid,
                        void* stream);

/* random_points (features == false path).  mask = (frame0 > 1) | (frame1 > 1); the mask's
 * non-zero pixels in row-major order are shuffled exactly as libstdc++'s
 * std::random_shuffle driven by glibc rand() does: seed < 0 reproduces the reference's
 * debug mode (no srand), seed >= 0 reproduces srand(seed) (the reference uses time(0)).
 * The first min(npoints, count) entries are returned:
 *   p = (pos + roi0) * inv_scale,  q = (pos + roi1 + flow(pos)) * inv_scale   in fp32,
 * widened to double as jsoncpp stores them; w = 1.  An empty mask yields the single dummy
 * entry (-1,-1,-1,-1, w = 0).  out arrays are HOST memory with room for max(npoints,1)
 * entries; positions (may be NULL) receives npoints (x,y) int pairs.  *n_out = entries. */
int tvl1_sample_matches(tvl1_handle* h, const uint8_t* d_frame0, size_t pitch0,
                        const uint8_t* d_frame1, size_t pitch1,
                        const float* d_u, const float* d_v, size_t pitch_flow,
                        int width, int height, int roi0_x, int roi0_y, int roi1_x, int roi1_y,
                        float scale, int npoints, long long seed,
                        double* px, double* py, double* qx, double* qy, double* w,
                        int* positions, int* n_out, void* stream);

/* Same, for a process that keeps drawing from one rand() stream (the reference's debug mode
 * never calls srand, so pair k starts where pair k-1 stopped): rand_skip = rand() calls already
 * made since the (implicit) srand(seed); *rand_used (may be NULL) receives the calls this
 * shuffle makes (mask pixels - 1). */
int tvl1_sample_matches_skip(tvl1_handle* h, const uint8_t* d_frame0, size_t pitch0,
                             const uint8_t* d_frame1, size_t pitch1,
                             const float* d_u, const float* d_v, size_t pitch_flow,
                             int width, int height, int roi0_x, int roi0_y, int roi1_x, int roi1_y,
                             float scale, int npoints, long long seed, long long rand_skip,
                             double* px, double* py, double* qx, double* qy, double* w,
                             int* positions, int* n_out, long long* rand_used, void* stream);

/* Same with the `features` branch of random_points (src/optflow.cpp:544-550): with q_is_map != 0 the planes
 * hold a MAP (flow + coordinate grid, as solve_wrapper leaves them after a feature pre-alignment) and
 * q = (map(pos) + roi1) * inv_scale, without the pos term. */
int tvl1_sample_matches_ex(tvl1_handle* h, const uint8_t* d_frame0, size_t pitch0,
                           const uint8_t* d_frame1, size_t pitch1,
                           const float* d_u, const float* d_v, size_t pitch_flow,
                           int width, int height, int roi0_x, int roi0_y, int roi1_x, int roi1_y,
                           float scale, int npoints, long long seed, long long rand_skip, int q_is_map,
                           double* px, double* py, double* qx, double* qy, double* w,
                           int* positions, int* n_out, long long* rand_used, void* stream);

/* ---- feature pre-alignment (N4): find_alignment, src/features.cpp:46-167, called by solve_rois whenever
 * a job asks for `features`, has no roi, or pairs frames of different size (src/optflow.cpp:366-377).
 * Keypoints + 256-bit binary descriptors on both frames (FAST-9 / Harris ranking / intensity-centroid
 * orientation / steered BRIEF over an ORB-style pyramid), Hamming 2-NN + ratio test, RANSAC homography,
 * the reference's +-20 % zoom sanity check; the top 2x3 of the homography is the affine that maps
 * `moving` (the pair's frame1) coordinates to `fixed` (frame0) coordinates.  Identity when there are not
 * more than 10 good matches or the check fails, as in the reference.  Not OpenCV's ORB bit for bit (its
 * learned test pattern is part of OpenCV's source): tests compare transforms.  SURF (features type 2,
 * the reference's default, non-free) takes the same path. */
typedef struct tvl1_feature_params {
    int nfeatures;          /* 5000   orb_defaults, src/features.cpp:19-32 */
    float scale_factor;     /* 1.2 */
    int nlevels;            /* 8 */
    int edge_threshold;     /* 31 */
    int first_level;        /* 0 (only 0) */
    int patch_size;         /* 31 */
    int fast_threshold;     /* 20 */
    float ratio;            /* 0.8    src/features.cpp:107 */
    double ransac;          /* 5.0    reprojection threshold, src/features.cpp:133 */
    int homo;               /* 8 = cv::RANSAC (4, 16 are served by RANSAC too), 0 = least squares on all matches */
    int debug;              /* prints the counts and the homography like the reference's debug mode */
    int reserved[4];
} tvl1_feature_params;
void tvl1_default_feature_params(tvl1_feature_params* p);
int tvl1_find_alignment(tvl1_handle* h, const uint8_t* d_moving, size_t pitch_moving, int w_moving, int h_moving,
                        const uint8_t* d_fixed, size_t pitch_fixed, int w_fixed, int h_fixed,
                        const tvl1_feature_params* prm, float* affine /* [6], row-major 2x3 */,
                        int* n_matches, int* n_good, void* stream);
/* cv::cuda::warpAffine(src, dst, affine, dsize, INTER_LINEAR, BORDER_CONSTANT, 0) of src/optflow.cpp:374
 * (8-bit frame) and :431-432 (fp32 map planes), computed as cv::warpAffine does: dst(x) = src(A^-1 x),
 * source coordinates in 1/32 px.  Pitches in bytes. */
int tvl1_warp_affine_u8(const uint8_t* d_src, size_t spitch, int sw, int sh, const float* affine,
                        uint8_t* d_dst, size_t dpitch, int dw, int dh, void* stream);
int tvl1_warp_affine_f32(const float* d_src, size_t spitch, int sw, int sh, const float* affine,
                         float* d_dst, size_t dpitch, int dw, int dh, void* stream);

/* A stack of adjacent slices: pairs (k, k+1), k = 0 .. n_slices-2, solved in order on one GPU
 * (the pair loop of from_file, src/optflow.cpp:86-176, incl. its re-use of the previous pair's
 * q frame as the next p, :97-103).  Every slice is uploaded once; the upload of slice k+2 and
 * the download of pair k-1's result run on copy streams while pair k is being solved, so host
 * buffers should be pinned.  Multi-GPU jobs give each rank a contiguous block of the stack. */
typedef struct tvl1_stack_io {
    const uint8_t* const* h_slices;   /* n_slices host pointers, 8-bit rows with byte pitch */
    size_t pitch;
    int n_slices, width, height;
    int apply_mask;                   /* flow = 0 where slice k+1 <= 1 (src/optflow.cpp:471-473) */
    float* const* h_u;                /* n_slices-1 host planes each, or NULL: no flow download */
    float* const* h_v;
    size_t pitch_out;
    int npoints;                      /* < 0: no match sampling */
    float scale;
    long long seed;                   /* >= 0: srand(seed) before every pair; < 0: one unseeded
                                         stream across the stack (the reference's debug mode) */
    double *px, *py, *qx, *qy, *w;    /* [(n_slices-1) * max(npoints,1)], or NULL if npoints < 0 */
    int* n_out;                       /* [n_slices-1] entries written per pair */
    tvl1_stats* stats;                /* [n_slices-1] or NULL */
    double prescale;                  /* 0 or 1: slices are used as given.  Otherwise every slice is
                                         shrunk on the device by this factor right after its upload,
                                         exactly like the loader's cv::resize (src/optflow.cpp:111,124);
                                         width/height/pitch describe the slices as given, the flow
                                         planes have tvl1_prescaled_size(width, height, prescale) */
    const int* pair_p;                /* NULL: pairs (k, k+1).  Otherwise n_pairs explicit pairs            */
    const int* pair_q;                /* (slices[pair_p[k]], slices[pair_q[k]]) -- the "images" list of a  */
    int n_pairs;                      /* job (src/optflow.cpp:86-94); outputs are indexed by pair.  A slice */
                                      /* consecutive pairs share stays on the device; the next pair's frames */
                                      /* go up while the current pair is solved                              */
} tvl1_stack_io;

int tvl1_stack_run(tvl1_handle* h, const tvl1_stack_io* io, float* ms_total);

/* ---- 8-bit prescale: the reference's loader shrinks every decoded frame with
 * cv::resize(frame, frame, cv::Size(), scale, scale) before anything else (src/optflow.cpp:111,124;
 * `scale` is a float job key, default 0.5).  Same result bit for bit (OpenCV's 11-bit fixed-point
 * bilinear, its 2x2 area path for scale == 0.5), computed on the device.  Output size:
 * cvRound(w * scale) x cvRound(h * scale).  Pitches in bytes. ---- */
int tvl1_prescaled_size(int w, int h, double scale, int* dw, int* dh);
int tvl1_prescale_u8(const uint8_t* d_src, size_t spitch, int w, int h, double scale,
                     uint8_t* d_dst, size_t dpitch, void* stream);
/* host buffers: upload, prescale, download (blocking; device scratch is kept per device and only grows) */
int tvl1_prescale_u8_host(int device, const uint8_t* src, size_t spitch, int w, int h, double scale,
                          uint8_t* dst, size_t dpitch);

/* ---- stage-level entry points: the individual kernels, exposed so that each can be
 * checked against the oracle on its own (tests/) and profiled on its own (bench.py).
 * Planes are fp32 with a pitch in ELEMENTS; pointers are device memory. ---- */
int tvl1_k_convert_u8(const uint8_t* d_src, size_t pitch_bytes, int w, int h, float* d_dst,
                      int pitch, void* stream);
int tvl1_k_resize(const float* d_src, int sw, int sh, int spitch, float* d_dst, int dw, int dh,
                  int dpitch, double inv_scale /* <= 0: explicit size */, float mul, void* stream);
int tvl1_k_centered_gradient(const float* d_src, int w, int h, int pitch, float* d_dx,
                             float* d_dy, void* stream);
/* warp step; I1's centred gradients are formed inside (A.3 fused into A.4).  d_I1w and d_grad
 * may be NULL. */
int tvl1_k_warp(const float* d_I0, const float* d_I1, const float* d_u1, const float* d_u2,
                int w, int h, int pitch, float* d_I1w, float* d_I1wx, float* d_I1wy,
                float* d_grad, float* d_rho_c, void* stream);
/* n inner iterations with no stop test; state planes are updated in place (the result
 * is copied back if it ends in the internal twin buffers).  errors (host, may be NULL)
 * receives the n per-iteration error sums. */
int tvl1_k_iterate(const float* d_I1wx, const float* d_I1wy, const float* d_grad,
                   const float* d_rho_c, float* d_u1, float* d_u2, float* d_p11, float* d_p12,
                   float* d_p21, float* d_p22, int w, int h, int pitch,
                   float l_t, float theta, float taut, int n, double* errors, void* stream);
/* n inner iterations of the three-channel form (gamma != 0: u3, p31, p32 join), in place, no stop test */
int tvl1_k_iterate_gamma(const float* d_I1wx, const float* d_I1wy, const float* d_rho_c,
                         float* d_u1, float* d_u2, float* d_u3, float* d_p11, float* d_p12,
                         float* d_p21, float* d_p22, float* d_p31, float* d_p32, int w, int h,
                         int pitch, float l_t, float theta, float taut, float gamma, int n,
                         double* errors, void* stream);
/* same through the temporally blocked kernel (two iterations per launch); n must be even */
int tvl1_k_iterate_fused2(const float* d_I1wx, const float* d_I1wy, const float* d_grad,
                          const float* d_rho_c, float* d_u1, float* d_u2, float* d_p11, float* d_p12,
                          float* d_p21, float* d_p22, int w, int h, int pitch,
                          float l_t, float theta, float taut, int n, double* errors, void* stream);
/* same through k_outer, the kernel the solver ships: all n iterations (any n >= 0) in ONE cooperative
 * launch -- two-iteration passes and, for odd n, a final single pass */
int tvl1_k_outer(const float* d_I1wx, const float* d_I1wy, const float* d_grad,
                 const float* d_rho_c, float* d_u1, float* d_u2, float* d_p11, float* d_p12,
                 float* d_p21, float* d_p22, int w, int h, int pitch,
                 float l_t, float theta, float taut, int n, double* errors, void* stream);
int tvl1_k_median5(const float* d_src, int w, int h, int pitch, float* d_dst, void* stream);
/* medianBlur(src, 3): the other fp32 aperture (medianFiltering = 3) */
int tvl1_k_median3(const float* d_src, int w, int h, int pitch, float* d_dst, void* stream);
/* The feature pre-alignment's kernels (8-bit images, pitches in BYTES; the score plane's in elements).
 * Candidates are {float harris; uint16_t x, y} (8 bytes), keypoints {float x, y, angle; int level}
 * (16 bytes, x and y in level-0 pixels), descriptors 8 uint32 words (byte l = tests 8l .. 8l+7, bit k = test 8l+k).
 * tvl1_k_gauss7_u8: 7x7 Gaussian (sigma 2), reflect-101 border, rounded to 8 bits. */
int tvl1_k_gauss7_u8(const uint8_t* d_src, size_t spitch, int w, int h, uint8_t* d_dst, size_t dpitch, void* stream);
/* FAST-9 score plane (0 within `border` of the frame), then 3x3 non-maximum suppression and the Harris response
 * of the survivors: up to `cap` candidates in d_cand, in any order.  *d_count and the 2048-bin histogram of the
 * responses' float bits >> 20 are ADDED to (the caller zeroes them) and count every survivor, listed or not. */
int tvl1_k_fast_corners(const uint8_t* d_img, size_t pitch, int w, int h, int border, int t, float* d_score, int spitch,
                        void* d_cand, int cap, int* d_count, int* d_hist, void* stream);
/* intensity-centroid angle on d_img and the 256 steered tests on d_blur (its own pitch) for n candidates;
 * keypoint x, y = candidate position * scale */
int tvl1_k_describe(const uint8_t* d_img, size_t pitch, const uint8_t* d_blur, size_t bpitch, const void* d_cand, int n,
                    float scale, int level, void* d_kp, uint32_t* d_desc, void* stream);
/* Hamming 2-NN of nq query descriptors among nt >= 1 train descriptors: nearest index (first on ties), its
 * distance and the second smallest distance (1 << 30 when nt == 1) */
int tvl1_k_knn2(const uint32_t* d_q, int nq, const uint32_t* d_t, int nt, int* d_idx1, int* d_d1, int* d_d2, void* stream);
/* one frame through the keypoint + descriptor stage of tvl1_find_alignment: *n_out <= nfeatures keypoints and
 * descriptors, level by level, each level's strongest first; cap (entries of d_kp / d_desc) >= nfeatures */
int tvl1_features_extract(tvl1_handle* h, const uint8_t* d_img, size_t pitch, int width, int height,
                          const tvl1_feature_params* prm, void* d_kp, uint32_t* d_desc, int cap, int* n_out,
                          void* stream);
/* CUDA-event time of the kernel launches of the calling thread's most recent tvl1_k_warp /
 * tvl1_k_iterate / tvl1_k_median5 call (waits for them). */
int tvl1_k_last_ms(float* ms);

/* Self-test of the kernels' exact fast paths (reciprocal-sharing division, fused hypot) against
 * the IEEE operators on n pseudo-random operand triples with binary exponents in [elo, ehi];
 * *mismatches receives the number of differing results (must be 0). */
int tvl1_selftest_arith(long long n, unsigned seed, int elo, int ehi, long long* mismatches,
                        long long* unvouched /* may be NULL: operand pairs the fp32 hypot handed to the exact path */);

/* pyramid level sizes for (w, h): returns levels used (A.2 stop rule) */
int tvl1_pyramid_sizes(int w, int h, int nscales, double scale_step, int* ws, int* hs);

/* glibc-compatible rand() stream used by the sampler: fills out[0..n) with the values
 * rand() returns at calls skip .. skip+n-1 after srand(seed) (seed < 0: unseeded). */
int tvl1_glibc_rand(long long seed, long long skip, int n, int* out);

/* minimal device-memory helpers so that C / ctypes callers need no other CUDA binding */
int tvl1_dev_count(void);
int tvl1_dev_alloc(int device, size_t bytes, void** out);
int tvl1_dev_free(int device, void* p);
int tvl1_dev_memset(void* d_dst, int value, size_t bytes);
int tvl1_dev_h2d(void* d_dst, const void* h_src, size_t bytes);
int tvl1_dev_d2h(void* h_dst, const void* d_src, size_t bytes);
int tvl1_dev_sync(int device);
/* streams and asynchronous copies for callers that overlap I/O with the solves (the job driver):
 * streams are created non-blocking; host buffers of the async copies must be pinned. */
int tvl1_set_device(int device);                        /* binds the calling host thread to the device */
int tvl1_stream_create(int device, void** out_stream);
int tvl1_stream_destroy(void* stream);
int tvl1_stream_sync(void* stream);
int tvl1_stream_query(void* stream);                    /* 1: all work done, 0: still running, < 0: error */
int tvl1_stream_wait(void* waiter, void* signaller);    /* waiter's later work runs after signaller's earlier work */
int tvl1_dev_h2d_async(void* d_dst, const void* h_src, size_t bytes, void* stream);
int tvl1_dev_d2h_async(void* h_dst, const void* d_src, size_t bytes, void* stream);
int tvl1_host_alloc_pinned(size_t bytes, void** out);
int tvl1_host_free_pinned(void* p);

#ifdef __cplusplus
}
#endif
#endif /* TVL1_B200_H */
