// tvl1_engine.cu -- per-device solver handle, the pair-level driver loop and the C ABI
// declared in include/tvl1_b200.h.  Replaces TVL1_solve (reference src/optflow.cpp:516-520),
// which builds a fresh cv::cuda::OpticalFlowDual_TVL1 -- and all its buffers -- per call: here
// the handle keeps one arena per device and re-uses it across pairs of the same size.
//
// There is no CPU fallback: every entry point runs CUDA kernels or fails with a status.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <mutex>
#include <vector>

#include "tvl1_kernels.cuh"
#include "tvl1_batch.cuh"
#include "tvl1_internal.h"

namespace tvl1 {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(TVL1_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                              \
    } while (0)

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------- cubic table (A.4)

static void cubic_coeffs(float x, float* c)
{
    // Keys bicubic, A = -0.75, evaluated in fp32 exactly as OpenCV's interpolateCubic does
    const float A = -0.75f;
    c[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
    c[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
    c[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
    c[3] = 1.f - c[0] - c[1] - c[2];
}

static int upload_cubic_table(int device)
{
    static bool done[64] = {false};
    if (device >= 0 && device < 64 && done[device]) return TVL1_OK;
    float tab[128];
    const float scale = 1.f / 32;
    for (int i = 0; i < 32; i++) cubic_coeffs(i * scale, tab + 4 * i);
    CK(cudaMemcpyToSymbol(c_cubic_tab, tab, sizeof(tab)));
    if (device >= 0 && device < 64) done[device] = true;
    return TVL1_OK;
}

int copy_words(const void* src, void* dst, int n32, cudaStream_t st)
{
    if (n32 <= 0) return TVL1_OK;
    const int blocks = n32 <= 256 ? 1 : (n32 + 1023) / 1024 < 32 ? (n32 + 1023) / 1024 : 32;
    k_copy_words<<<blocks, n32 < 256 ? 32 : 256, 0, st>>>((const int*)src, (int*)dst, n32);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// ---------------------------------------------------------------- tensor maps (TMA)

// cuTensorMapEncodeTiled through the runtime's driver entry point: the library keeps linking the CUDA
// runtime only (statically), never libcuda
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// an fp32 plane {pitch x h} as a 2-D tensor whose box is one staged tile (box_w x box_h elements, dense rows)
int make_plane_map(CUtensorMap* tm, const float* base, int pitch, int h, int box_w, int box_h)
{
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return fail(TVL1_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[2] = {(cuuint64_t)pitch, (cuuint64_t)h};
    const cuuint64_t strides[1] = {(cuuint64_t)pitch * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h}, es[2] = {1, 1};
    const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(TVL1_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for a %dx%d plane", (int)r, pitch, h);
    return TVL1_OK;
}

// n fp32 planes {pitch x h} at equal distances as a 3-D tensor {x, y, plane}; the box is one 128-px row of every plane
static int make_section_map(CUtensorMap* tm, const float* base, int pitch, int h, int n, size_t plane_stride_bytes)
{
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return fail(TVL1_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[3] = {(cuuint64_t)pitch, (cuuint64_t)h, (cuuint64_t)n};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * sizeof(float), (cuuint64_t)plane_stride_bytes};
    const cuuint32_t box[3] = {128u, 1u, (cuuint32_t)n}, es[3] = {1, 1, 1};
    const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(TVL1_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for %d planes of %dx%d", (int)r, n, pitch, h);
    return TVL1_OK;
}

// the tensor maps the two-iteration pass fills its ring through (IterMaps), from the plane pointers of `a`:
// the planes of each section must sit at equal, 16-byte aligned distances
static int make_section(CUtensorMap* tm, const float* const* planes, int n, int pitch, int h)
{
    const ptrdiff_t d = (const char*)planes[1] - (const char*)planes[0];
    bool even = d > 0 && d % 16 == 0 && (size_t)d >= (size_t)pitch * h * sizeof(float) && !((uintptr_t)planes[0] & 15);
    for (int k = 2; k < n && even; k++) even = (const char*)planes[k] - (const char*)planes[k - 1] == d;
    if (!even) return fail(TVL1_ERR_INVALID, "the planes of a ring section must sit at equal 16-byte aligned distances");
    return make_section_map(tm, planes[0], pitch, h, n, (size_t)d);
}

int make_iter_maps(IterArgs& a)
{
    int rc;
    const float* c[3] = {a.I1wx, a.I1wy, a.rho_c};
    if ((rc = make_section(&a.tm.c, c, 3, a.pitch, a.h))) return rc;
    for (int t = 0; t < 2; t++) {
        const float* u[2] = {a.u1[t], a.u2[t]};
        const float* p[4] = {a.p11[t], a.p12[t], a.p21[t], a.p22[t]};
        if ((rc = make_section(&a.tm.u[t], u, 2, a.pitch, a.h))) return rc;
        if ((rc = make_section(&a.tm.p[t], p, 4, a.pitch, a.h))) return rc;
    }
    return TVL1_OK;
}

// ---------------------------------------------------------------- pyramid geometry (A.2)

static int scaled_size(int n, double f) { return (int)lrint((double)n * f); }   // round half even

int pyramid_sizes(int w, int h, int nscales, double scale_step, int* ws, int* hs)
{
    if (nscales > TVL1_MAX_LEVELS) nscales = TVL1_MAX_LEVELS;
    ws[0] = w;
    hs[0] = h;
    int used = nscales;
    for (int s = 1; s < nscales; s++) {
        ws[s] = scaled_size(ws[s - 1], scale_step);
        hs[s] = scaled_size(hs[s - 1], scale_step);
        if (ws[s] < 16 || hs[s] < 16) { used = s; break; }   // that level is built then dropped
    }
    return used;
}

// ---------------------------------------------------------------- launch helpers

static inline dim3 grid2d(int w, int h, dim3 b) { return dim3(cdiv(w, b.x), cdiv(h, b.y)); }

int launch_convert(const uint8_t* src, size_t pitch, int w, int h, float* dst, int dpitch, cudaStream_t st)
{
    dim3 b(32, 8);
    dim3 g(cdiv(cdiv(w, 4), 32), cdiv(h, 8));
    k_convert_u8<<<g, b, 0, st>>>(src, pitch, w, h, dst, dpitch);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// fp32 frame (byte pitch, a multiple of 4) -> level 0, x 255
int launch_convert_f32(const float* src, size_t pitch_bytes, int w, int h, float* dst, int dpitch, cudaStream_t st)
{
    dim3 b(32, 8);
    dim3 g(cdiv(cdiv(w, 4), 32), cdiv(h, 8));
    k_convert_f32<<<g, b, 0, st>>>(src, pitch_bytes / 4, w, h, dst, dpitch);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// one or two planes (srcB / dstB null: one) of one pair, the source in twin 0
static ResizeArgs resize_args(const float* srcA, const float* srcB, int sw, int sh, int sp, float* dstA, float* dstB, int dw,
                              int dh, int dp)
{
    ResizeArgs a = {};
    a.src[0][0] = srcA; a.src[1][0] = srcB; a.dst[0] = dstA; a.dst[1] = dstB;
    a.sw = sw; a.sh = sh; a.sp = sp; a.dw = dw; a.dh = dh; a.dp = dp;
    return a;
}

// gridDim.z of a resize of a's planes of n pairs.  One plane (dst[1] null) of n > 1 pairs, without a ctrl: pair k's
// plane is taken as plane k & 1 of pair k >> 1 at twice the stride
static unsigned resize_z(ResizeArgs& a, int n)
{
    if (a.dst[1]) return 2 * n;
    if (n == 1) return 1;
    a.src[1][0] = (const float*)((const char*)a.src[0][0] + a.stride);
    a.dst[1] = (float*)((char*)a.dst[0] + a.stride);
    a.stride *= 2;
    return n;
}

// a's planes of n pairs (two planes each, or one: see resize_z) resized alike in one launch.  inv_scale > 0:
// resize(src, Size(), inv_scale, inv_scale); otherwise the explicit size dw x dh.  apply_mul: see scale_px
int launch_resize(ResizeArgs a, int n, double inv_scale, double mul, int apply_mul, cudaStream_t st)
{
    double inv_x, inv_y;
    if (inv_scale > 0) { inv_x = inv_scale; inv_y = inv_scale; }
    else { inv_x = (double)a.dw / a.sw; inv_y = (double)a.dh / a.sh; }
    a.scale_x = 1. / inv_x; a.scale_y = 1. / inv_y; a.mul = mul; a.apply_mul = apply_mul;
    const unsigned nz = resize_z(a, n);
    dim3 b(32, 8);
    // resize(src, Size(), 0.5, 0.5): OpenCV's INTER_AREA fast path.  The fp32 multiply (tvl1_k_resize with mul != 1)
    // has always taken the bilinear kernel at 0.5 and keeps doing so; the fp64 one (an initial flow's downscale) is
    // cv::resize followed by cv::multiply and so takes the area path like the image pyramid
    if (inv_scale == 0.5 && apply_mul != 1) k_resize_half<<<dim3(cdiv(a.dw, 32), cdiv(a.dh, 8), nz), b, 0, st>>>(a);
    else k_resize<<<dim3(cdiv(cdiv(a.dw, 4), 32), cdiv(a.dh, 8), nz), b, 0, st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// cv::cuda semantics: cuda::resize(INTER_LINEAR) of a's planes of n pairs, as launch_resize.  inv_scale > 0:
// resize(src, Size(), inv_scale, inv_scale); otherwise the explicit size dw x dh (factor dw / sw in fp64).  The
// source step fx = (float)(1 / factor) and the multiply by (float)mul (apply_mul != 0) are fp32.
int launch_resize_cuda(ResizeArgs a, int n, double inv_scale, double mul, int apply_mul, cudaStream_t st)
{
    const double f_x = inv_scale > 0 ? inv_scale : (double)a.dw / a.sw;
    const double f_y = inv_scale > 0 ? inv_scale : (double)a.dh / a.sh;
    a.scale_x = 1.0 / f_x; a.scale_y = 1.0 / f_y; a.mul = mul; a.apply_mul = apply_mul;
    dim3 b(32, 8);
    dim3 g(cdiv(a.dw, 32), cdiv(a.dh, 8), resize_z(a, n));
    k_resize_cuda<<<g, b, 0, st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int launch_gradient(const float* src, int w, int h, int pitch, float* dx, float* dy, cudaStream_t st)
{
    dim3 b(32, 8);
    k_centered_gradient<<<grid2d(w, h, b), b, 0, st>>>(src, w, h, pitch, dx, dy);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int launch_warp(const WarpArgs& a, cudaStream_t st)
{
    // persistent blocks: one grid of resident blocks walks the tile list
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int& resident = cached[dev & 63];
    if (!resident) {
        int sms = 148, occ = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_warp, TVL1_WP_THREADS, 0) != cudaSuccess || occ < 1) occ = 2;
        resident = sms * occ;
    }
    const long long ntiles = (long long)cdiv(a.w, TVL1_WP_TW) * cdiv(a.h, TVL1_WP_TH);
    dim3 b(32, TVL1_WP_NW);
    k_warp<<<(unsigned)(ntiles < resident ? ntiles : resident), b, 0, st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// cv::cuda semantics: warpBackward (persistent blocks over the 32 x 16 tiles)
int launch_warp_cuda(const WarpArgs& a, cudaStream_t st)
{
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int& resident = cached[dev & 63];
    if (!resident) {
        int sms = 148, occ = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_warp_cuda<false>, 256, 0) != cudaSuccess || occ < 1) occ = 2;
        resident = sms * occ;
    }
    const long long ntiles = (long long)cdiv(a.w, TVL1_WC_TW) * cdiv(a.h, TVL1_WC_TH);
    k_warp_cuda<false><<<(unsigned)(ntiles < resident ? ntiles : resident), dim3(32, 8), 0, st>>>(a, 0);
    CK(cudaGetLastError());
    return TVL1_OK;
}

static const int ITER_NW = 4;   // warps per block of the iteration kernels

// resident blocks of the iteration kernels on the current device (SMs x occupancy), queried once
// per device; the fused kernel's shared-memory ring needs the opt-in limit raised first
enum { KI_SMALL = 0, KI_LARGE = 1, KI_FUSED = 2, KI_MULTI = 3, KI_OUTER = 4 };   // k_iterate<.,5>, k_iterate<.,4>, k_iterate2, k_iterate_multi
static const long long ITER_LARGE_PX = 16000000;     // levels at least this large: 4 blocks per SM

// CS: the instantiation with the cv::cuda stop schedule (TVL1_SEMANTICS_CUDA)
template <bool CS>
static int resident_blocks(int which)
{
    static int cached[5][64] = {};
    int dev = 0, sms = 148, occ = 0;
    cudaGetDevice(&dev);
    int& c = cached[which][dev & 63];
    if (c) return c;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e;
    if (which == KI_FUSED) {
        // the shared-memory ring needs the opt-in limit raised first
        cudaFuncSetAttribute(k_iterate2<ITER_NW, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, TVL1_RING_BYTES(ITER_NW));
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_iterate2<ITER_NW, CS>, 32 * ITER_NW, TVL1_RING_BYTES(ITER_NW));
    } else if (which == KI_OUTER) {
        cudaFuncSetAttribute(k_outer<ITER_NW, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, TVL1_RING_BYTES(ITER_NW));
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_outer<ITER_NW, CS>, 32 * ITER_NW, TVL1_RING_BYTES(ITER_NW));
    } else if (which == KI_MULTI) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_iterate_multi<ITER_NW, 4, CS>, 32 * ITER_NW, 0);
    } else if (which == KI_LARGE) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_iterate<ITER_NW, 4, CS>, 32 * ITER_NW, 0);
    } else {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_iterate<ITER_NW, 5, CS>, 32 * ITER_NW, 0);
    }
    if (e != cudaSuccess || occ < 1) occ = (which == KI_FUSED || which == KI_OUTER) ? 3 : 4;
    c = sms * occ;
    return c;
}

static int resident_blocks(int which, bool cs) { return cs ? resident_blocks<true>(which) : resident_blocks<false>(which); }

// upper bound of the grid of any iteration kernel (blocks resident on the device), for the
// per-block partial sums: SMs x the 32-blocks-per-SM hardware limit, two slabs
size_t iterate_max_blocks()
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (size_t)sms * 32 * 2;
}

// Rows per tile and grid size.  A tile is one warp's strip x R rows and every resident warp walks
// the tile list with a grid stride: tall tiles amortise the halo rows (R / (R + halo)), but the
// tile count has to spread evenly over the resident warps (no nearly empty last round).
static int tile_rows_search(int w, int h, int strip, int halo, int rmin, int resident_blocks, int* grid)
{
    const long long ns = cdiv(w, strip);
    const long long slots = (long long)resident_blocks * ITER_NW;
    double best = -1.0;
    int best_r = rmin;
    long long best_g = 1;
    for (int R = rmin; R <= 64; ++R) {
        const long long ntiles = ns * cdiv(h, R);
        const long long G = ntiles < slots ? ntiles : slots;   // warps that get work
        const long long rounds = (ntiles + G - 1) / G;
        double eff = (double)ntiles / (double)(rounds * G) * (double)R / (double)(R + halo);
        if (G < slots) eff *= (double)G / (double)slots;       // not even one tile per warp
        if (eff >= best) { best = eff; best_r = R; best_g = G; }
    }
    *grid = (int)((best_g + ITER_NW - 1) / ITER_NW);
    return best_r;
}

// the search runs once per (size, kernel): a solve launches the same few shapes hundreds of times
static int tile_rows(int w, int h, int strip, int halo, int rmin, int resident_blocks, int* grid)
{
    struct Entry { int w, h, strip, resident, rows, grid; };
    static thread_local Entry cache[32];
    static thread_local int used = 0, next = 0;
    for (int i = 0; i < used; i++) {
        const Entry& e = cache[i];
        if (e.w == w && e.h == h && e.strip == strip && e.resident == resident_blocks) { *grid = e.grid; return e.rows; }
    }
    Entry e = {w, h, strip, resident_blocks, 0, 0};
    e.rows = tile_rows_search(w, h, strip, halo, rmin, resident_blocks, &e.grid);
    cache[next] = e;
    next = (next + 1) % 32;
    if (used < 32) used++;
    *grid = e.grid;
    return e.rows;
}

int launch_iterate(IterArgs& a, cudaStream_t st, bool cs = false)
{
    int grid = 1;
    const bool large = (long long)a.w * a.h >= ITER_LARGE_PX;
    a.rows = tile_rows(a.w, a.h, TVL1_STRIP, 1, 4, resident_blocks(large ? KI_LARGE : KI_SMALL, cs), &grid);
    dim3 b(32, ITER_NW);
    if (cs) {
        if (large) k_iterate<ITER_NW, 4, true><<<grid, b, 0, st>>>(a);
        else k_iterate<ITER_NW, 5, true><<<grid, b, 0, st>>>(a);
    } else if (large) k_iterate<ITER_NW, 4><<<grid, b, 0, st>>>(a);
    else k_iterate<ITER_NW, 5><<<grid, b, 0, st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// several iterations in one cooperative launch (small levels); the grid must be co-resident
int launch_iterate_multi(IterArgs& a, cudaStream_t st, bool cs = false)
{
    // these levels are bound by latency, not by throughput: the shortest tiles that still give every
    // tile its own warp (one round) make an iteration a chain of R + 1 dependent row steps only
    const int resident = resident_blocks(KI_MULTI, cs);
    const long long slots = (long long)resident * ITER_NW, ns = cdiv(a.w, TVL1_STRIP);
    int grid = 1, R = 0;
    for (int r = 1; r <= 8 && !R; ++r)
        if (ns * cdiv(a.h, r) <= slots) R = r;
    if (R) {
        a.rows = R;
        grid = (int)((ns * cdiv(a.h, R) + ITER_NW - 1) / ITER_NW);
    } else {
        a.rows = tile_rows(a.w, a.h, TVL1_STRIP, 1, 4, resident, &grid);
    }
    dim3 b(32, ITER_NW), g(grid);
    void* args[] = {(void*)&a};
    const void* fn = cs ? (const void*)k_iterate_multi<ITER_NW, 4, true> : (const void*)k_iterate_multi<ITER_NW, 4>;
    cudaError_t e = cudaLaunchCooperativeKernel(fn, g, b, args, 0, st);
    if (e != cudaSuccess) return fail(TVL1_ERR_CUDA, "cooperative launch of k_iterate_multi failed: %s", cudaGetErrorString(e));
    return TVL1_OK;
}

// the inner loop of one outer iteration (fused + single passes) in one cooperative launch
int launch_outer(IterArgs& a, cudaStream_t st, bool cs = false)
{
    int grid = 1, g1 = 1;
    const int resident = resident_blocks(KI_OUTER, cs);
    const long long slots = (long long)resident * ITER_NW;
    const long long ns2 = cdiv(a.w, TVL1_STRIP2), ns1 = cdiv(a.w, TVL1_STRIP);
    int R2 = 0, R1 = 0;
    // small levels are bound by latency: the shortest tiles that still give every tile its own warp
    for (int r = 1; r <= 8 && !R2; ++r)
        if (ns2 * cdiv(a.h, r) <= slots) R2 = r;
    for (int r = 1; r <= 8 && !R1; ++r)
        if (ns1 * cdiv(a.h, r) <= slots) R1 = r;
    if (R2) {
        a.rows = R2;
        grid = (int)((ns2 * cdiv(a.h, R2) + ITER_NW - 1) / ITER_NW);
    } else {
        a.rows = tile_rows(a.w, a.h, TVL1_STRIP2, 3, 8, resident, &grid);
    }
    a.rows1 = R1 ? R1 : tile_rows(a.w, a.h, TVL1_STRIP, 1, 4, resident, &g1);   // single passes stride over the same grid
    dim3 b(32, ITER_NW), g(grid);
    void* args[] = {(void*)&a};
    const void* fn = cs ? (const void*)k_outer<ITER_NW, true> : (const void*)k_outer<ITER_NW>;
    cudaError_t e = cudaLaunchCooperativeKernel(fn, g, b, args, TVL1_RING_BYTES(ITER_NW), st);
    if (e != cudaSuccess) return fail(TVL1_ERR_CUDA, "cooperative launch of k_outer failed: %s", cudaGetErrorString(e));
    return TVL1_OK;
}

int launch_iterate2(IterArgs& a, cudaStream_t st, bool cs = false)
{
    int grid = 1;
    a.rows = tile_rows(a.w, a.h, TVL1_STRIP2, 3, 8, resident_blocks(KI_FUSED, cs), &grid);   // 3 halo rows per tile
    dim3 b(32, ITER_NW);
    if (cs) k_iterate2<ITER_NW, true><<<grid, b, TVL1_RING_BYTES(ITER_NW), st>>>(a);
    else k_iterate2<ITER_NW><<<grid, b, TVL1_RING_BYTES(ITER_NW), st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// gamma != 0: one inner iteration = k_plain_u<3> + k_plain_p<3> (persistent blocks over row segments)
int launch_gamma_iteration(const PlainIterArgs& a, cudaStream_t st)
{
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int& resident = cached[dev & 63];
    if (!resident) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        resident = sms * 8;
    }
    const long long ntiles = (long long)cdiv(a.w, 128) * a.h;
    const long long want = (ntiles + TVL1_PLAIN_NW - 1) / TVL1_PLAIN_NW;
    const unsigned grid = (unsigned)(want < resident ? want : resident);
    dim3 b(32, TVL1_PLAIN_NW);
    k_plain_u<3><<<grid, b, 0, st>>>(a);
    k_plain_p<3><<<grid, b, 0, st>>>(a);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int launch_median3(const MedianArgs& a, int planes, cudaStream_t st)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long n = (long long)cdiv(a.w, 4) * a.h * planes;
    const long long want = (n + 255) / 256;
    k_median3<<<(unsigned)(want < sms * 8 ? want : sms * 8), 256, 0, st>>>(a, planes, 0);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int launch_median(const MedianArgs& a, int planes, cudaStream_t st)
{
    // persistent blocks: one grid of resident blocks walks the tile list of both planes
    static int cached[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int& resident = cached[dev & 63];
    if (!resident) {
        int sms = 148, occ = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_median5, 256, 0) != cudaSuccess || occ < 1) occ = 2;
        resident = sms * occ;
    }
    const long long ntiles = (long long)cdiv(a.w, TVL1_MED_TW) * cdiv(a.h, TVL1_MED_TH) * planes;
    dim3 b(32, 8);
    k_median5<<<(unsigned)(ntiles < resident ? ntiles : resident), b, 0, st>>>(a, planes);
    CK(cudaGetLastError());
    return TVL1_OK;
}

// ---------------------------------------------------------------- handle

struct Level {
    alignas(64) CUtensorMap tm_med[2][2];   // median tiles of [u1 | u2][twin] (built with the arena)
    CUtensorMap tm_I1[2];                   // warp windows of I1: RW x 16 and RW x RH boxes
    IterMaps tm_iter;                       // ring rows of the two-iteration pass
    int w, h, pitch;
    float *I0, *I1, *u1, *u2;   // u1/u2: buffer [0] of the twin pair; [1] is shared scratch
};

// Byte offsets of one pair's state in the batch arena (tvl1_calc_batch_ex); pair b's copy is at + b * stride.
// u3, p31, p32: only in an arena made for gamma != 0
struct BatchLayout {
    size_t I0[TVL1_MAX_LEVELS], I1[TVL1_MAX_LEVELS], u1[TVL1_MAX_LEVELS], u2[TVL1_MAX_LEVELS], u3[TVL1_MAX_LEVELS];
    size_t u1x, u2x, I1wx, I1wy, rho, p[4], p31, p32, part, ctrl;
};

}  // namespace tvl1

using namespace tvl1;

#define TVL1_STACK_SLOTS 4   // slice slots of tvl1_stack_run: two for the pair being solved, two for the next pair's frames

struct tvl1_handle {
    int device = 0;
    tvl1_params prm;
    int inner = 30, outer = 10;
    bool timing = false;
 bool coop_outer = true;             // fused levels: the inner loop of an outer iteration in ONE cooperative launch
    bool multi_iter = true;             // levels below fused_min_px: all inner iterations of an outer one in ONE cooperative launch
    long long fused_min_px = 0;         // levels at least this large use the two-iteration passes (with the cooperative loop they win at every size)
    // arena
    char* arena = nullptr;
    size_t arena_bytes = 0;
    int cap_w = 0, cap_h = 0, cap_scales = 0;
    double cap_step = 0;
    int nlevels = 0;
    Level lv[TVL1_MAX_LEVELS];
    float *I1wx = nullptr, *I1wy = nullptr, *rho = nullptr;   // warp outputs (I1x, I1y, grad never exist as planes)
    float *u1x = nullptr, *u2x = nullptr;   // twin [1] of u, shared by all levels
    float* p[4][2] = {{nullptr}};           // p11,p12,p21,p22 twins
    // gamma != 0 only: u3 per level, p31, p32 (their own allocation, made on first use)
    char* garena = nullptr;
    float* u3[TVL1_MAX_LEVELS] = {};
    float *p31 = nullptr, *p32 = nullptr;
    Ctrl* d_ctrl = nullptr;
    Ctrl* h_ctrl = nullptr;                 // pinned
    double* d_partials = nullptr;
    size_t partials_cap = 0;
    // staging for the host-buffer entry points: frames (rows of stage_pitch bytes, u8 or fp32), flow out, and the
    // initial flow (allocated on first use); reallocated when the size changes or fp32 rows need more room
    void *d_f0 = nullptr, *d_f1 = nullptr;
    float *d_uo = nullptr, *d_vo = nullptr, *d_ui = nullptr, *d_vi = nullptr;
    size_t stage_pitch = 0;
    int stage_w = 0, stage_h = 0;
    cudaStream_t own_stream = nullptr;
    std::vector<cudaEvent_t> events;
    size_t ev_used = 0;
    // sampler scratch (tvl1_sampler.cu), feature scratch (tvl1_features.cu)
    void* samp = nullptr;
    void* feat = nullptr;
    // stack runner (tvl1_stack_run): 3 slice slots, 2 flow buffers, copy streams
    uint8_t* st_slice[TVL1_STACK_SLOTS] = {};
    uint8_t* st_raw[2] = {nullptr, nullptr};   // raw slices awaiting the device prescale
    size_t st_raw_bytes = 0;
    float* st_flow[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
    size_t st_pitch8 = 0;
    int st_w = 0, st_h = 0;
    cudaStream_t st_in = nullptr, st_out = nullptr;
    cudaEvent_t st_up[TVL1_STACK_SLOTS] = {}, st_ready[2] = {nullptr, nullptr}, st_down[2] = {nullptr, nullptr};
    // batch arena (tvl1_calc_batch_ex), apart from the single-pair one: bcap_n copies of a pair's state at
    // bstride bytes, then the 4 * bcap_n pointers of the frames and initial flows; pinned: bcap_n Ctrl read-backs,
    // then those pointers.  bcap_gamma: the pairs' state includes the planes of the third channel
    char* barena = nullptr;
    char* bhost = nullptr;
    size_t bstride = 0;
    int bcap_n = 0, bcap_w = 0, bcap_h = 0, bcap_scales = 0;
    bool bcap_gamma = false;
    double bcap_step = 0;
    BatchLayout bl;
    long long readbacks = 0;   // host read-backs of the stop state by the last calc
};

namespace tvl1 {

int handle_device(const tvl1_handle* h) { return h->device; }
void** handle_sampler_slot(tvl1_handle* h) { return &h->samp; }
void** handle_feature_slot(tvl1_handle* h) { return &h->feat; }

static int get_event(tvl1_handle* H, cudaEvent_t* out)
{
    if (H->ev_used == H->events.size()) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        H->events.push_back(e);
    }
    *out = H->events[H->ev_used++];
    return TVL1_OK;
}

static void release_arena(tvl1_handle* H)
{
    if (H->garena) cudaFree(H->garena);
    H->garena = nullptr;
    if (H->arena) cudaFree(H->arena);
    H->arena = nullptr;
    H->arena_bytes = 0;
    H->cap_w = H->cap_h = 0;
}

static int ensure_capacity(tvl1_handle* H, int w, int h, cudaStream_t st)
{
    if (H->arena && H->cap_w == w && H->cap_h == h && H->cap_scales == H->prm.nscales &&
        H->cap_step == H->prm.scale_step)
        return TVL1_OK;
    release_arena(H);
    int ws[TVL1_MAX_LEVELS + 1], hs[TVL1_MAX_LEVELS + 1];
    const int L = pyramid_sizes(w, h, H->prm.nscales, H->prm.scale_step, ws, hs);
    // carve: 256-byte aligned planes
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    struct Plan { size_t I0, I1, u1, u2; } plan[TVL1_MAX_LEVELS];
    for (int s = 0; s < L; s++) {
        const int pitch = round_up(ws[s], 32);
        const size_t b = (size_t)pitch * hs[s] * sizeof(float);
        plan[s].I0 = carve(b); plan[s].I1 = carve(b); plan[s].u1 = carve(b); plan[s].u2 = carve(b);
    }
    const int pitch0 = round_up(w, 32);
    const size_t b0 = (size_t)pitch0 * h * sizeof(float);
    size_t o_scr[5], o_p[8];
    for (int i = 0; i < 5; i++) o_scr[i] = carve(b0);   // I1wx I1wy rho u1x u2x
    for (int i = 0; i < 8; i++) o_p[i] = carve(b0);
    const size_t nb = iterate_max_blocks();
    const size_t o_part = carve(nb * sizeof(double));
    const size_t o_ctrl = carve(sizeof(Ctrl));
    cudaError_t e = cudaMalloc(&H->arena, off);
    if (e != cudaSuccess) {
        H->arena = nullptr;
        return fail(TVL1_ERR_NOMEM, "cudaMalloc(%zu bytes) for a %dx%d pair failed: %s", off, w, h,
                    cudaGetErrorString(e));
    }
    H->arena_bytes = off;
    for (int s = 0; s < L; s++) {
        H->lv[s].w = ws[s]; H->lv[s].h = hs[s]; H->lv[s].pitch = round_up(ws[s], 32);
        H->lv[s].I0 = (float*)(H->arena + plan[s].I0); H->lv[s].I1 = (float*)(H->arena + plan[s].I1);
        H->lv[s].u1 = (float*)(H->arena + plan[s].u1); H->lv[s].u2 = (float*)(H->arena + plan[s].u2);
    }
    H->nlevels = L;
    float** scr[5] = {&H->I1wx, &H->I1wy, &H->rho, &H->u1x, &H->u2x};
    for (int i = 0; i < 5; i++) *scr[i] = (float*)(H->arena + o_scr[i]);
    for (int i = 0; i < 8; i++) H->p[i / 2][i % 2] = (float*)(H->arena + o_p[i]);
    H->d_partials = (double*)(H->arena + o_part);
    H->partials_cap = nb;
    H->d_ctrl = (Ctrl*)(H->arena + o_ctrl);
    for (int s = 0; s < L; s++) {   // tensor maps of the planes TMA reads, once per arena
        Level& lv = H->lv[s];
        const float* planes[2][2] = {{lv.u1, H->u1x}, {lv.u2, H->u2x}};
        for (int z = 0; z < 2; z++)
            for (int t = 0; t < 2; t++) {
                const int r = make_plane_map(&lv.tm_med[z][t], planes[z][t], lv.pitch, lv.h, TVL1_MED_SW, TVL1_MED_SH);
                if (r) { release_arena(H); return r; }
            }
        for (int k = 0; k < 2; k++) {
            const int r = make_plane_map(&lv.tm_I1[k], lv.I1, lv.pitch, lv.h, TVL1_WP_RW, k == 0 ? 16 : TVL1_WP_RH);
            if (r) { release_arena(H); return r; }
        }
        {
            IterArgs ia;
            ia.I1wx = H->I1wx; ia.I1wy = H->I1wy; ia.rho_c = H->rho;
            ia.u1[0] = lv.u1; ia.u1[1] = H->u1x; ia.u2[0] = lv.u2; ia.u2[1] = H->u2x;
            for (int k = 0; k < 2; k++) { ia.p11[k] = H->p[0][k]; ia.p12[k] = H->p[1][k]; ia.p21[k] = H->p[2][k]; ia.p22[k] = H->p[3][k]; }
            ia.w = lv.w; ia.h = lv.h; ia.pitch = lv.pitch;
            const int r = make_iter_maps(ia);
            if (r) { release_arena(H); return r; }
            lv.tm_iter = ia.tm;
        }
    }
    H->cap_w = w; H->cap_h = h; H->cap_scales = H->prm.nscales; H->cap_step = H->prm.scale_step;
    // pad columns are read (never used) by the vectorised kernels: give them defined contents.  On the
    // solve's own stream: a non-blocking stream does not order itself after the legacy default stream
    CK(cudaMemsetAsync(H->arena, 0, off, st));
    return TVL1_OK;
}

// planes of the third channel (gamma != 0): sized like the arena they accompany, released with it
static int ensure_gamma(tvl1_handle* H, cudaStream_t st)
{
    if (H->prm.gamma == 0.0 || H->garena) return TVL1_OK;
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    size_t o3[TVL1_MAX_LEVELS];
    for (int s = 0; s < H->nlevels; s++) o3[s] = carve((size_t)H->lv[s].pitch * H->lv[s].h * sizeof(float));
    const size_t b0 = (size_t)H->lv[0].pitch * H->lv[0].h * sizeof(float);
    const size_t o31 = carve(b0), o32 = carve(b0);
    cudaError_t e = cudaMalloc(&H->garena, off);
    if (e != cudaSuccess) {
        H->garena = nullptr;
        return fail(TVL1_ERR_NOMEM, "cudaMalloc(%zu bytes) for the gamma planes failed: %s", off, cudaGetErrorString(e));
    }
    for (int s = 0; s < H->nlevels; s++) H->u3[s] = (float*)(H->garena + o3[s]);
    H->p31 = (float*)(H->garena + o31);
    H->p32 = (float*)(H->garena + o32);
    CK(cudaMemsetAsync(H->garena, 0, off, st));
    return TVL1_OK;
}

static int resolve_iterations(tvl1_handle* H)
{
    const tvl1_params& p = H->prm;
    if (p.semantics == TVL1_SEMANTICS_CUDA) {
        // cv::cuda's flat loop: `iterations` iterations per (level, warp), no outer iterations
        H->inner = p.iterations > 0 ? p.iterations : 300;
        H->outer = 1;
        return TVL1_OK;
    }
    if (p.inner_iterations > 0 && p.outer_iterations > 0) {
        H->inner = p.inner_iterations;
        H->outer = p.outer_iterations;
    } else {
        // SURVEY.md T3: the cv::cuda API's flat `iterations` = inner 30 x outer ceil(N/30)
        H->inner = p.inner_iterations > 0 ? p.inner_iterations : 30;
        const int n = p.iterations > 0 ? p.iterations : 300;
        H->outer = p.outer_iterations > 0 ? p.outer_iterations : (n + H->inner - 1) / H->inner;
    }
    return TVL1_OK;
}

static int check_params(const tvl1_params* p)
{
    if (!p) return fail(TVL1_ERR_INVALID, "params is null");
    if (p->nscales <= 0) return fail(TVL1_ERR_INVALID, "nscales must be > 0");   // CV_Assert(nscales > 0)
    if (p->nscales > TVL1_MAX_LEVELS) return fail(TVL1_ERR_INVALID, "nscales > %d", TVL1_MAX_LEVELS);
    if (p->warps <= 0 || p->warps > TVL1_MAX_WARPS) return fail(TVL1_ERR_INVALID, "warps out of range");
    if (!(p->scale_step > 0.0 && p->scale_step < 1.0)) return fail(TVL1_ERR_INVALID, "scaleStep must be in (0,1)");
    if (!(p->gamma == p->gamma)) return fail(TVL1_ERR_INVALID, "gamma is not a number");
    if (p->use_initial_flow) return fail(TVL1_ERR_UNSUPPORTED, "useInitialFlow is not supported (the reference never forwards it)");
    if (p->semantics != TVL1_SEMANTICS_CPU && p->semantics != TVL1_SEMANTICS_CUDA)
        return fail(TVL1_ERR_INVALID, "semantics must be TVL1_SEMANTICS_CPU (0) or TVL1_SEMANTICS_CUDA (1)");
    if (p->semantics == TVL1_SEMANTICS_CUDA) {   // medianFiltering is not read in this mode
        if (p->inner_iterations > 0 || p->outer_iterations > 0)
            return fail(TVL1_ERR_INVALID, "cuda semantics has one flat loop of `iterations`: inner/outer iterations must be <= 0");
        if (p->gamma != 0.0) return fail(TVL1_ERR_UNSUPPORTED, "gamma != 0 is not supported with cuda semantics");
        if (!(p->theta > 0.0)) return fail(TVL1_ERR_INVALID, "theta must be > 0");
        if (!(p->lambda >= 0.0)) return fail(TVL1_ERR_INVALID, "lambda must be >= 0");
        return TVL1_OK;
    }
    if (p->median_filtering != 1 && p->median_filtering != 3 && p->median_filtering != 5)   // cv::medianBlur's fp32 apertures
        return fail(TVL1_ERR_UNSUPPORTED, "medianFiltering must be 1 (off), 3 or 5");
    if (!(p->theta > 0.0)) return fail(TVL1_ERR_INVALID, "theta must be > 0");
    if (!(p->lambda >= 0.0)) return fail(TVL1_ERR_INVALID, "lambda must be >= 0");   // the threshold step assumes l_t * grad >= 0
    return TVL1_OK;
}

// frame type, row pitches and initial-flow planes of tvl1_calc_ex[_host]
static int check_frames(int frame_type, size_t pitch0, size_t pitch1, int w, int h, const float* u0, const float* v0,
                        size_t pitch_init, size_t pitch_out)
{
    if (w <= 0 || h <= 0) return fail(TVL1_ERR_INVALID, "empty image (%dx%d)", w, h);
    if (frame_type != TVL1_FRAME_U8 && frame_type != TVL1_FRAME_F32)
        return fail(TVL1_ERR_INVALID, "frame_type must be TVL1_FRAME_U8 (0) or TVL1_FRAME_F32 (1)");
    const size_t row = (size_t)w * (frame_type == TVL1_FRAME_F32 ? 4 : 1);
    if (pitch0 < row || pitch1 < row || pitch_out < (size_t)w * 4) return fail(TVL1_ERR_INVALID, "pitch smaller than a row");
    if (frame_type == TVL1_FRAME_F32 && (pitch0 % 4 || pitch1 % 4))
        return fail(TVL1_ERR_INVALID, "fp32 frame pitches must be multiples of 4 bytes");
    if ((u0 == nullptr) != (v0 == nullptr)) return fail(TVL1_ERR_INVALID, "the initial flow needs both planes (or neither)");
    if (u0 && (pitch_init % 4 || pitch_init < (size_t)w * 4))
        return fail(TVL1_ERR_INVALID, "initial-flow pitch must be a multiple of 4 bytes and at least a row");
    return TVL1_OK;
}

// stats from a pair's final Ctrl: level sizes, iteration counts, totals and the byte model (zeroes the rest)
static void stats_counts(tvl1_stats* stats, const Ctrl& c, int L, int W, const int* ws, const int* hs)
{
    memset(stats, 0, sizeof(*stats));
    stats->levels = L;
    stats->warps = W;
    double bytes = 70.0 * (double)ws[0] * hs[0];
    for (int s = 0; s < L; s++) {
        stats->width[s] = ws[s];
        stats->height[s] = hs[s];
        const double px = (double)ws[s] * hs[s];
        double per_px = 12.0;
        for (int wi = 0; wi < W; wi++) {
            const int n = c.iters[s * W + wi], o = c.outer[s * W + wi];
            stats->iters[s * W + wi] = n;
            stats->outer[s * W + wi] = o;
            stats->total_iterations += n;
            stats->px_iterations += (long long)px * n;
            per_px += 40.0 + 64.0 * n + 16.0 * o;
        }
        bytes += px * per_px;
    }
    stats->algorithmic_bytes = bytes;
}

// the solve proper; everything is enqueued on `st`.  u0 / v0 (both or neither): the initial flow (useInitialFlow),
// which may be d_u / d_v themselves
static int calc_device(tvl1_handle* H, int frame_type, const void* f0, size_t pitch0, const void* f1, size_t pitch1,
                       int w, int h, const float* u0, const float* v0, size_t pitch_init,
                       float* d_u, float* d_v, size_t pitch_out, cudaStream_t st, tvl1_stats* stats)
{
    if (!f0 || !f1 || !d_u || !d_v) return fail(TVL1_ERR_INVALID, "null image or flow pointer");
    int rc = check_frames(frame_type, pitch0, pitch1, w, h, u0, v0, pitch_init, pitch_out);
    if (rc) return rc;
    if (w > 32767 || h > 32767) return fail(TVL1_ERR_INVALID, "image side > 32767 (remap uses int16 coordinates)");
    CK(cudaSetDevice(H->device));
    if ((rc = ensure_capacity(H, w, h, st))) return rc;
    if ((rc = ensure_gamma(H, st))) return rc;
    if ((rc = upload_cubic_table(H->device))) return rc;
    const tvl1_params& P = H->prm;
    const int L = H->nlevels, W = P.warps;
    const float l_t = (float)(P.lambda * P.theta);
    const float taut = (float)(P.tau / P.theta);
    const float theta = (float)P.theta;
    // TVL1_SEMANTICS_CUDA: cv::cuda's resize, warp and flat loop with its sparse stop test, no median
    const bool cs = P.semantics == TVL1_SEMANTICS_CUDA;
    long long launches = 0;
    H->ev_used = 0;
    H->readbacks = 0;

    cudaEvent_t ev_begin, ev_pyr, ev_end;
    if ((rc = get_event(H, &ev_begin)) || (rc = get_event(H, &ev_pyr)) || (rc = get_event(H, &ev_end))) return rc;
    struct Span { cudaEvent_t a, b; int kind, level; };
    std::vector<Span> spans;
    // per-stage events only when the caller asked for them (tvl1_set_timing): thousands of
    // cudaEventRecord calls per pair otherwise
    const bool timed = stats != nullptr && H->timing;
    auto span_begin = [&](int kind, int level) -> int {
        if (!timed) return TVL1_OK;
        Span s; s.kind = kind; s.level = level;
        int r = get_event(H, &s.a); if (r) return r;
        r = get_event(H, &s.b); if (r) return r;
        cudaEventRecord(s.a, st);
        spans.push_back(s);
        return TVL1_OK;
    };
    auto span_end = [&]() { if (timed) cudaEventRecord(spans.back().b, st); };

    CK(cudaEventRecord(ev_begin, st));
    CK(cudaMemsetAsync(H->d_ctrl, 0, sizeof(Ctrl), st));
    // (1) pyramid: convert, then resize level by level
    if (frame_type == TVL1_FRAME_F32) {
        if ((rc = launch_convert_f32((const float*)f0, pitch0, w, h, H->lv[0].I0, H->lv[0].pitch, st))) return rc;
        if ((rc = launch_convert_f32((const float*)f1, pitch1, w, h, H->lv[0].I1, H->lv[0].pitch, st))) return rc;
    } else {
        if ((rc = launch_convert((const uint8_t*)f0, pitch0, w, h, H->lv[0].I0, H->lv[0].pitch, st))) return rc;
        if ((rc = launch_convert((const uint8_t*)f1, pitch1, w, h, H->lv[0].I1, H->lv[0].pitch, st))) return rc;
    }
    launches += 2;
    for (int s = 1; s < L; s++) {
        const Level &a = H->lv[s - 1], &b = H->lv[s];
        const ResizeArgs ra = resize_args(a.I0, a.I1, a.w, a.h, a.pitch, b.I0, b.I1, b.w, b.h, b.pitch);
        if ((rc = cs ? launch_resize_cuda(ra, 1, P.scale_step, 1.f, 0, st) : launch_resize(ra, 1, P.scale_step, 1.f, 0, st)))
            return rc;
        launches += 1;
    }
    if (u0) {
        // useInitialFlow: level 0 is the caller's flow, each coarser level the image pyramid's resize of the finer
        // one, then times scaleStep as a rounding of its own -- cv::multiply by a double Scalar in the CPU class,
        // an fp32 product in cv::cuda (SURVEY.md A.2a, Appendix B).  Into twin 0, which ucur names after the Ctrl
        // memset; the coarsest level is not zeroed, the finer ones are overwritten by the upsample as usual.
        const Level& l0 = H->lv[0];
        CK(cudaMemcpy2DAsync(l0.u1, (size_t)l0.pitch * 4, u0, pitch_init, (size_t)w * 4, h, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpy2DAsync(l0.u2, (size_t)l0.pitch * 4, v0, pitch_init, (size_t)w * 4, h, cudaMemcpyDeviceToDevice, st));
        for (int s = 1; s < L; s++) {
            const Level &a = H->lv[s - 1], &b = H->lv[s];
            const ResizeArgs ra = resize_args(a.u1, a.u2, a.w, a.h, a.pitch, b.u1, b.u2, b.w, b.h, b.pitch);
            rc = cs ? launch_resize_cuda(ra, 1, P.scale_step, (float)P.scale_step, 1, st)
                    : launch_resize(ra, 1, P.scale_step, P.scale_step, 2, st);
            if (rc) return rc;
            launches += 1;
        }
    }
    {
        const Level& c = H->lv[L - 1];
        const size_t b = (size_t)c.pitch * c.h * sizeof(float);
        if (!u0) {
            CK(cudaMemsetAsync(c.u1, 0, b, st));
            CK(cudaMemsetAsync(c.u2, 0, b, st));
        }
        if (P.gamma != 0.0) CK(cudaMemsetAsync(H->u3[L - 1], 0, b, st));
    }
    CK(cudaEventRecord(ev_pyr, st));

    const size_t hdr = offsetof(Ctrl, iters);
    std::vector<int> counts((size_t)L * W, 0);   // iterations each (level, warp) needed
    for (int s = L - 1; s >= 0; --s) {
        const Level& lv = H->lv[s];
        const size_t pb = (size_t)lv.pitch * lv.h * sizeof(float);
        const float scaled_eps = (float)(P.epsilon * P.epsilon * (double)(lv.w * lv.h));
        if ((rc = span_begin(3, s))) return rc;
        // p11 .. p22 start a level at zero: the level's first warp kernel writes the zeros (WarpArgs::pz)
        if (P.gamma != 0.0) { CK(cudaMemsetAsync(H->p31, 0, pb, st)); CK(cudaMemsetAsync(H->p32, 0, pb, st)); }
        span_end();

        IterArgs ia;
        ia.I1wx = H->I1wx; ia.I1wy = H->I1wy; ia.rho_c = H->rho;
        ia.u1[0] = lv.u1; ia.u1[1] = H->u1x; ia.u2[0] = lv.u2; ia.u2[1] = H->u2x;
        for (int k = 0; k < 2; k++) { ia.p11[k] = H->p[0][k]; ia.p12[k] = H->p[1][k]; ia.p21[k] = H->p[2][k]; ia.p22[k] = H->p[3][k]; }
        ia.w = lv.w; ia.h = lv.h; ia.pitch = lv.pitch;
        ia.l_t = l_t; ia.theta = theta; ia.taut = taut; ia.scaled_eps = scaled_eps; ia.one = 1.0f;
        ia.level = s; ia.ctrl = H->d_ctrl; ia.partials = H->d_partials; ia.errlog = nullptr;
        ia.mode = 0; ia.inner_max = H->inner;
        ia.tm = lv.tm_iter;
        ia.eps_d = P.epsilon * P.epsilon * (double)(lv.w * lv.h);
        ia.err_on = P.epsilon > 0.0;
        const bool with_gamma = P.gamma != 0.0;
        PlainIterArgs ga = {};
        if (with_gamma) {
            ga.I1wx = H->I1wx; ga.I1wy = H->I1wy; ga.rho_c = H->rho;
            ga.u1[0] = ia.u1[0]; ga.u1[1] = ia.u1[1]; ga.u2[0] = ia.u2[0]; ga.u2[1] = ia.u2[1]; ga.u3 = H->u3[s];
            // in place in H->p[k][0], the planes the level's first warp zeroes: only the k_iterate* / k_outer kernels
            // flip pcur, so this solve never leaves them
            ga.p11 = H->p[0][0]; ga.p12 = H->p[1][0]; ga.p21 = H->p[2][0]; ga.p22 = H->p[3][0];
            ga.p31 = H->p31; ga.p32 = H->p32;
            ga.w = lv.w; ga.h = lv.h; ga.pitch = lv.pitch;
            ga.l_t = l_t; ga.theta = theta; ga.taut = taut; ga.gamma = (float)P.gamma; ga.scaled_eps = scaled_eps;
            ga.level = s; ga.slot = 0; ga.inner_max = H->inner;
            ga.ctrl = H->d_ctrl; ga.partials = H->d_partials; ga.errlog = nullptr;
        }
        const bool fused = (long long)lv.w * lv.h >= H->fused_min_px && H->inner >= 2;
        const bool multi = !fused && H->multi_iter && H->inner >= 2;
        MedianArgs ma;
        ma.u1[0] = lv.u1; ma.u1[1] = H->u1x; ma.u2[0] = lv.u2; ma.u2[1] = H->u2x;
        ma.w = lv.w; ma.h = lv.h; ma.pitch = lv.pitch; ma.level = s; ma.ctrl = H->d_ctrl;
        memcpy(ma.tm, lv.tm_med, sizeof(ma.tm));
        WarpArgs wa;
        wa.I0 = lv.I0; wa.I1 = lv.I1;
        wa.u1[0] = lv.u1; wa.u1[1] = H->u1x; wa.u2[0] = lv.u2; wa.u2[1] = H->u2x;
        wa.I1w = nullptr; wa.I1wx = H->I1wx; wa.I1wy = H->I1wy; wa.grad = nullptr; wa.rho_c = H->rho;
        wa.w = lv.w; wa.h = lv.h; wa.pitch = lv.pitch; wa.level = s; wa.ctrl = H->d_ctrl; wa.one = 1.0f;
        memcpy(wa.tmI1, lv.tm_I1, sizeof(wa.tmI1));

        for (int wi = 0; wi < W; ++wi) {
            const int slot = s * W + wi;
            ia.slot = slot;
            ma.slot = slot;
            // (2) warp I1 by the current flow; also re-arms the stop test (error = FLT_MAX)
            if ((rc = span_begin(1, s))) return rc;
            for (int k = 0; k < 4; k++) wa.pz[k] = wi == 0 ? H->p[k][0] : nullptr;
            if ((rc = cs ? launch_warp_cuda(wa, st) : launch_warp(wa, st))) return rc;
            launches++;
            span_end();
            // (3) outer iterations: median + up to `inner` primal-dual iterations.  Every kernel is a
            // no-op once the device-side stop flag is set, so iterations are enqueued in chunks without
            // knowing how many will really run; the first chunk is sized by the count the previous
            // warp (or, for the first warp, the coarser level) needed, and one 32-byte read-back per
            // chunk tells the host whether more are wanted.  The stop iteration is exactly the
            // oracle's; a wrong guess costs a few no-op launches or one extra host round trip.
            const int pred_total = wi > 0 ? counts[slot - 1] : (s < L - 1 ? counts[(s + 1) * W] : H->inner);
            int done_total = 0;
            for (int no = 0; no < H->outer; ++no) {
                if (P.median_filtering > 1 && !cs) {
                    if ((rc = span_begin(2, s))) return rc;
                    if ((rc = P.median_filtering == 3 ? launch_median3(ma, 2, st) : launch_median(ma, 2, st))) return rc;
                    launches++;
                    span_end();
                }
                if ((rc = span_begin(0, s))) return rc;
                // a new outer iteration: no inner iteration done yet
                CK(cudaMemsetAsync(&H->d_ctrl->inner, 0, sizeof(int), st));
                int done_inner = 0, want = 0;
                for (;;) {
                    const int left_pred = pred_total - done_total - done_inner;
                    want = want == 0 ? (left_pred + 1 > 4 ? left_pred + 1 : 4) : 2 * want;
                    if (want > H->inner - done_inner) want = H->inner - done_inner;
                    if (with_gamma) {
                        // the three-channel iteration: two plain launches each, no-ops once the stop flag is set
                        ga.slot = slot;
                        for (int k = 0; k < want; ++k)
                            if ((rc = launch_gamma_iteration(ga, st))) return rc;
                        launches += 2 * want;
                    } else if (fused && H->coop_outer) {
                        // the whole inner loop of this outer iteration in one cooperative launch
                        IterArgs io = ia;
                        io.mode = 2;
                        if ((rc = launch_outer(io, st, cs))) return rc;
                        launches += 1;
                    } else if (fused) {
                        // temporally blocked schedule: [fused pair | single] slot pairs.  Which slot
                        // of a pair really runs is decided on the device: the pair while the stop is
                        // not imminent and two iterations still fit, the single after an overshoot
                        // (replay), near the stop, or for the last iteration.
                        IterArgs i2 = ia, i1 = ia;
                        i2.mode = 2; i1.mode = 1;
                        const int groups = (want + 1) / 2;
                        for (int k = 0; k < groups; ++k) {
                            if ((rc = launch_iterate2(i2, st, cs))) return rc;
                            if ((rc = launch_iterate(i1, st, cs))) return rc;
                        }
                        launches += 2 * groups;
                    } else if (multi) {
                        // small level: one cooperative launch runs the rest of this outer iteration
                        IterArgs im = ia;
                        im.mode = 3;
                        if ((rc = launch_iterate_multi(im, st, cs))) return rc;
                        launches += 1;
                    } else {
                        IterArgs i3 = ia;
                        i3.mode = 3;
                        for (int k = 0; k < want; ++k)
                            if ((rc = launch_iterate(i3, st, cs))) return rc;
                        launches += want;
                    }
                    if ((rc = copy_words(H->d_ctrl, H->h_ctrl, (int)(hdr / 4), st))) return rc;   // no copy engine: see copy_words
                    CK(cudaStreamSynchronize(st));
                    H->readbacks++;
                    done_inner = H->h_ctrl->inner;
                    if (H->h_ctrl->done || done_inner >= H->inner) break;
                }
                span_end();
                done_total += done_inner;
                if (H->h_ctrl->done) break;
            }
            counts[slot] = done_total;
        }
        if (s == 0) break;
        // flow upsample to the next finer level (A.2): resize to its size, times 1/scaleStep
        const Level& up = H->lv[s - 1];
        const int uc = H->h_ctrl->ucur[s];
        const float mul = (float)(1 / P.scale_step);
        if ((rc = span_begin(3, s))) return rc;
        const ResizeArgs ra = resize_args(uc ? H->u1x : lv.u1, uc ? H->u2x : lv.u2, lv.w, lv.h, lv.pitch, up.u1, up.u2, up.w,
                                          up.h, up.pitch);
        if ((rc = cs ? launch_resize_cuda(ra, 1, 0.0, mul, 1, st) : launch_resize(ra, 1, 0.0, mul, 1, st))) return rc;
        launches += 1;
        if (with_gamma) {   // u3 is zoomed like the flow but not scaled
            if ((rc = launch_resize(resize_args(H->u3[s], nullptr, lv.w, lv.h, lv.pitch, H->u3[s - 1], nullptr, up.w, up.h,
                                                up.pitch), 1, 0.0, 1.f, 0, st))) return rc;
            launches += 1;
        }
        span_end();
    }
    // A.8: planar output
    {
        const int uc = H->h_ctrl->ucur[0];
        const Level& l0 = H->lv[0];
        CK(cudaMemcpy2DAsync(d_u, pitch_out, uc ? H->u1x : l0.u1, (size_t)l0.pitch * 4, (size_t)w * 4, h, cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpy2DAsync(d_v, pitch_out, uc ? H->u2x : l0.u2, (size_t)l0.pitch * 4, (size_t)w * 4, h, cudaMemcpyDeviceToDevice, st));
    }
    CK(cudaEventRecord(ev_end, st));
    if ((rc = copy_words(H->d_ctrl, H->h_ctrl, (int)(sizeof(Ctrl) / 4), st))) return rc;
    CK(cudaStreamSynchronize(st));
    H->readbacks++;

    if (stats) {
        int ws[TVL1_MAX_LEVELS], hs[TVL1_MAX_LEVELS];
        for (int s = 0; s < L; s++) { ws[s] = H->lv[s].w; hs[s] = H->lv[s].h; }
        stats_counts(stats, *H->h_ctrl, L, W, ws, hs);
        stats->launches = launches;
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev_begin, ev_end);
        stats->ms_total = ms;
        cudaEventElapsedTime(&ms, ev_begin, ev_pyr);
        stats->ms_pyramid = ms;
        for (const Span& sp : spans) {
            cudaEventElapsedTime(&ms, sp.a, sp.b);
            switch (sp.kind) {
                case 0: stats->ms_iterate += ms; stats->ms_iterate_level[sp.level] += ms; break;
                case 1: stats->ms_warp += ms; break;
                case 2: stats->ms_median += ms; break;
                default: stats->ms_other += ms; break;
            }
        }
    }
    return TVL1_OK;
}

// ---------------------------------------------------------------- batches of equal-size pairs

static void release_batch(tvl1_handle* H)
{
    if (H->barena) cudaFree(H->barena);
    if (H->bhost) cudaFreeHost(H->bhost);
    H->barena = nullptr;
    H->bhost = nullptr;
    H->bcap_n = H->bcap_w = H->bcap_h = 0;
}

// the batch arena for n pairs of w x h: kept while it has room for n pairs of this size and pyramid, and the planes of
// the third channel when gamma != 0
static int ensure_batch(tvl1_handle* H, int n, int w, int h, cudaStream_t st)
{
    const bool gamma = H->prm.gamma != 0.0;
    if (H->barena && H->bcap_n >= n && H->bcap_w == w && H->bcap_h == h && H->bcap_scales == H->prm.nscales &&
        H->bcap_step == H->prm.scale_step && (H->bcap_gamma || !gamma))
        return TVL1_OK;
    release_batch(H);
    int ws[TVL1_MAX_LEVELS + 1], hs[TVL1_MAX_LEVELS + 1];
    const int L = pyramid_sizes(w, h, H->prm.nscales, H->prm.scale_step, ws, hs);
    BatchLayout& B = H->bl;
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    for (int s = 0; s < L; s++) {
        const size_t b = (size_t)round_up(ws[s], 32) * hs[s] * sizeof(float);
        B.I0[s] = carve(b); B.I1[s] = carve(b); B.u1[s] = carve(b); B.u2[s] = carve(b);
    }
    const size_t b0 = (size_t)round_up(w, 32) * h * sizeof(float);
    B.u1x = carve(b0); B.u2x = carve(b0);
    B.I1wx = carve(b0); B.I1wy = carve(b0); B.rho = carve(b0);
    for (int k = 0; k < 4; k++) B.p[k] = carve(b0);
    if (gamma) {
        for (int s = 0; s < L; s++) B.u3[s] = carve((size_t)round_up(ws[s], 32) * hs[s] * sizeof(float));
        B.p31 = carve(b0); B.p32 = carve(b0);
    }
    B.part = carve(TVL1_BATCH_MAX_BLOCKS * sizeof(double));
    B.ctrl = carve(sizeof(Ctrl));
    const size_t ptrs = ((size_t)4 * n * sizeof(void*) + 255) / 256 * 256;
    if (off > (SIZE_MAX - ptrs) / (size_t)n)
        return fail(TVL1_ERR_NOMEM, "a batch of %d pairs of %dx%d does not fit in the address space", n, w, h);
    const size_t total = off * (size_t)n + ptrs;
    cudaError_t e = cudaMalloc(&H->barena, total);
    if (e != cudaSuccess) {
        cudaGetLastError();   // an allocation failure is reported here, not by the next launch check
        H->barena = nullptr;
        return fail(TVL1_ERR_NOMEM, "cudaMalloc(%zu bytes) for a batch of %d pairs of %dx%d failed: %s", total, n, w, h,
                    cudaGetErrorString(e));
    }
    e = cudaMallocHost(&H->bhost, (size_t)n * sizeof(Ctrl) + (size_t)4 * n * sizeof(void*));
    if (e != cudaSuccess) {
        cudaGetLastError();
        H->bhost = nullptr;
        release_batch(H);
        return fail(TVL1_ERR_NOMEM, "cudaMallocHost for a batch of %d pairs failed: %s", n, cudaGetErrorString(e));
    }
    H->bstride = off;
    H->bcap_n = n; H->bcap_w = w; H->bcap_h = h; H->bcap_scales = H->prm.nscales; H->bcap_step = H->prm.scale_step;
    H->bcap_gamma = gamma;
    CK(cudaMemsetAsync(H->barena, 0, total, st));   // pad columns are read (never used): defined contents
    return TVL1_OK;
}

// blocks per pair of a batched launch over `units` work items of `per_block` each: enough to fill the device
// together with the other pairs, at most TVL1_BATCH_MAX_BLOCKS (the per-pair partial sums)
static int batch_blocks(long long units, int per_block, int n)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long cap = ((long long)sms * 16 + n - 1) / n;
    if (cap > TVL1_BATCH_MAX_BLOCKS) cap = TVL1_BATCH_MAX_BLOCKS;
    const long long want = (units + per_block - 1) / per_block;
    return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

// calc_device's loop in lockstep over n pairs of one size: the same (level, warp, outer iteration) for every pair,
// each with its own stop state, so that every pair sees the kernel sequence of its own solve.  Its choices are
// calc_device's: in cuda semantics cv::cuda's resize and warp, no median and one outer iteration of `iterations`;
// with gamma != 0 the three-channel iteration.  u0 / v0 (both or neither): each pair's initial flow, whose entries
// may be those of d_u / d_v
static int calc_batch(tvl1_handle* H, int n, int frame_type, const void* const* f0, size_t pitch0, const void* const* f1,
                      size_t pitch1, int w, int h, const float* const* u0, const float* const* v0, size_t pitch_init,
                      float* const* d_u, float* const* d_v, size_t pitch_out, cudaStream_t st, tvl1_stats* stats)
{
    const tvl1_params& P = H->prm;
    if (n < 1 || n > TVL1_BATCH_MAX_PAIRS) return fail(TVL1_ERR_INVALID, "n must be in 1 .. %d, not %d", TVL1_BATCH_MAX_PAIRS, n);
    if (!f0 || !f1 || !d_u || !d_v) return fail(TVL1_ERR_INVALID, "null pointer array");
    if ((u0 == nullptr) != (v0 == nullptr))
        return fail(TVL1_ERR_INVALID, "the initial flow needs both pointer arrays (or neither)");
    for (int k = 0; k < n; k++) {
        if (!f0[k] || !f1[k] || !d_u[k] || !d_v[k]) return fail(TVL1_ERR_INVALID, "null image or flow pointer in entry %d", k);
        if (u0 && (!u0[k] || !v0[k])) return fail(TVL1_ERR_INVALID, "null initial-flow pointer in entry %d", k);
    }
    int rc = check_frames(frame_type, pitch0, pitch1, w, h, u0 ? u0[0] : nullptr, v0 ? v0[0] : nullptr, pitch_init, pitch_out);
    if (rc) return rc;
    if (w > 32767 || h > 32767) return fail(TVL1_ERR_INVALID, "image side > 32767 (remap uses int16 coordinates)");
    CK(cudaSetDevice(H->device));
    if ((rc = ensure_batch(H, n, w, h, st))) return rc;
    if ((rc = upload_cubic_table(H->device))) return rc;
    int ws[TVL1_MAX_LEVELS + 1], hs[TVL1_MAX_LEVELS + 1];
    const int L = pyramid_sizes(w, h, P.nscales, P.scale_step, ws, hs), W = P.warps;
    int pitch[TVL1_MAX_LEVELS];
    for (int s = 0; s < L; s++) pitch[s] = round_up(ws[s], 32);
    const float l_t = (float)(P.lambda * P.theta), taut = (float)(P.tau / P.theta), theta = (float)P.theta;
    const bool cs = P.semantics == TVL1_SEMANTICS_CUDA, with_gamma = P.gamma != 0.0;
    const BatchLayout& B = H->bl;
    const size_t S = H->bstride;
    char* const base = H->barena;
    auto plane = [&](size_t o) { return (float*)(base + o); };
    Ctrl* const ctrl = (Ctrl*)(base + B.ctrl);
    Ctrl* const hc = (Ctrl*)H->bhost;                                          // pair b's read-back: hc[b]
    const void** const hptr = (const void**)(H->bhost + (size_t)n * sizeof(Ctrl));   // f0[], f1[], u0[], v0[]
    const void** const dptr = (const void**)(base + (size_t)H->bcap_n * S);
    const size_t hdr = offsetof(Ctrl, iters);
    long long launches = 0;
    H->ev_used = 0;
    H->readbacks = 0;
    auto read_ctrl = [&](size_t bytes) -> int {   // every pair's first `bytes` of Ctrl -> hc[], then wait for them
        const int words = (int)(bytes / 4);
        const long long total = (long long)n * words;
        k_bctrl_read<<<(unsigned)(total < 256 * 32 ? (total + 255) / 256 : 32), 256, 0, st>>>(ctrl, S, words, n, (int*)hc);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(st));
        H->readbacks++;
        return TVL1_OK;
    };

    cudaEvent_t ev_begin, ev_end;
    if ((rc = get_event(H, &ev_begin)) || (rc = get_event(H, &ev_end))) return rc;
    CK(cudaEventRecord(ev_begin, st));
    CK(cudaMemset2DAsync(ctrl, S, 0, sizeof(Ctrl), n, st));
    // (1) pyramid of every pair
    const int nptr = u0 ? 4 * n : 2 * n;
    for (int k = 0; k < n; k++) {
        hptr[k] = f0[k]; hptr[n + k] = f1[k];
        if (u0) { hptr[2 * n + k] = u0[k]; hptr[3 * n + k] = v0[k]; }
    }
    CK(cudaMemcpyAsync(dptr, hptr, (size_t)nptr * sizeof(void*), cudaMemcpyHostToDevice, st));
    const dim3 gc(cdiv(cdiv(w, 4), 32), cdiv(h, 8), 2 * n);
    if (frame_type == TVL1_FRAME_F32)
        k_bconvert_f32<<<gc, dim3(32, 8), 0, st>>>((const float* const*)dptr, pitch0 / 4, pitch1 / 4, w, h, plane(B.I0[0]),
                                                   plane(B.I1[0]), pitch[0], S);
    else
        k_bconvert_u8<<<gc, dim3(32, 8), 0, st>>>((const uint8_t* const*)dptr, pitch0, pitch1, w, h, plane(B.I0[0]),
                                                  plane(B.I1[0]), pitch[0], S);
    CK(cudaGetLastError());
    launches += 1;
    for (int s = 1; s < L; s++) {
        ResizeArgs ra = resize_args(plane(B.I0[s - 1]), plane(B.I1[s - 1]), ws[s - 1], hs[s - 1], pitch[s - 1], plane(B.I0[s]),
                                    plane(B.I1[s]), ws[s], hs[s], pitch[s]);
        ra.stride = S;
        if ((rc = cs ? launch_resize_cuda(ra, n, P.scale_step, 1.f, 0, st) : launch_resize(ra, n, P.scale_step, 1.f, 0, st)))
            return rc;
        launches += 1;
    }
    if (u0) {
        // useInitialFlow, as calc_device: level 0 is each pair's flow, each coarser level the finer one resized and
        // times scaleStep (fp64 in the CPU class, fp32 in cv::cuda).  Into twin 0; the coarsest level is not zeroed
        k_bload_flow<<<dim3(cdiv(w, 32), cdiv(h, 8), 2 * n), dim3(32, 8), 0, st>>>(
            (const float* const*)(dptr + 2 * n), pitch_init / 4, w, h, plane(B.u1[0]), plane(B.u2[0]), pitch[0], S);
        CK(cudaGetLastError());
        launches += 1;
        for (int s = 1; s < L; s++) {
            ResizeArgs ra = resize_args(plane(B.u1[s - 1]), plane(B.u2[s - 1]), ws[s - 1], hs[s - 1], pitch[s - 1],
                                        plane(B.u1[s]), plane(B.u2[s]), ws[s], hs[s], pitch[s]);
            ra.stride = S;
            rc = cs ? launch_resize_cuda(ra, n, P.scale_step, (float)P.scale_step, 1, st)
                    : launch_resize(ra, n, P.scale_step, P.scale_step, 2, st);
            if (rc) return rc;
            launches += 1;
        }
    }
    {   // the coarsest level starts from zero flow (without an initial one), u3 from zero
        const size_t b = (size_t)pitch[L - 1] * hs[L - 1] * sizeof(float);
        if (!u0) {
            CK(cudaMemset2DAsync(plane(B.u1[L - 1]), S, 0, b, n, st));
            CK(cudaMemset2DAsync(plane(B.u2[L - 1]), S, 0, b, n, st));
        }
        if (with_gamma) CK(cudaMemset2DAsync(plane(B.u3[L - 1]), S, 0, b, n, st));
    }

    std::vector<int> counts((size_t)L * W, 0);   // the most iterations any pair needed per (level, warp)
    std::vector<int> total(n);
    for (int s = L - 1; s >= 0; --s) {
        const int lw = ws[s], lh = hs[s];
        PlainIterArgs ia = {};
        ia.I1wx = plane(B.I1wx); ia.I1wy = plane(B.I1wy); ia.rho_c = plane(B.rho);
        ia.u1[0] = plane(B.u1[s]); ia.u1[1] = plane(B.u1x); ia.u2[0] = plane(B.u2[s]); ia.u2[1] = plane(B.u2x);
        ia.p11 = plane(B.p[0]); ia.p12 = plane(B.p[1]); ia.p21 = plane(B.p[2]); ia.p22 = plane(B.p[3]);
        ia.w = lw; ia.h = lh; ia.pitch = pitch[s];
        ia.l_t = l_t; ia.theta = theta; ia.taut = taut;
        ia.scaled_eps = (float)(P.epsilon * P.epsilon * (double)(lw * lh));
        ia.level = s; ia.inner_max = H->inner; ia.ctrl = ctrl; ia.partials = (double*)(base + B.part); ia.stride = S;
        ia.eps_d = P.epsilon * P.epsilon * (double)(lw * lh);
        ia.err_on = P.epsilon > 0.0;
        if (with_gamma) {
            ia.u3 = plane(B.u3[s]); ia.p31 = plane(B.p31); ia.p32 = plane(B.p32); ia.gamma = (float)P.gamma;
            // p31 / p32 start the level at zero (the warp zeroes p11 .. p22)
            const size_t pb = (size_t)pitch[s] * lh * sizeof(float);
            CK(cudaMemset2DAsync(ia.p31, S, 0, pb, n, st));
            CK(cudaMemset2DAsync(ia.p32, S, 0, pb, n, st));
        }
        const dim3 gi(batch_blocks((long long)cdiv(lw, 128) * lh, TVL1_PLAIN_NW, n), 1, n);
        MedianArgs ma = {};
        ma.u1[0] = ia.u1[0]; ma.u1[1] = ia.u1[1]; ma.u2[0] = ia.u2[0]; ma.u2[1] = ia.u2[1];
        ma.ctrl = ctrl; ma.w = lw; ma.h = lh; ma.pitch = pitch[s]; ma.level = s;
        const int per_thread = P.median_filtering == 3 ? 4 : 8;
        const dim3 gm(batch_blocks(2LL * cdiv(lw, per_thread) * lh, 256, n), 1, n);
        BWarpArgs wa;
        wa.I0 = plane(B.I0[s]); wa.I1 = plane(B.I1[s]);
        wa.u1[0] = ia.u1[0]; wa.u1[1] = ia.u1[1]; wa.u2[0] = ia.u2[0]; wa.u2[1] = ia.u2[1];
        wa.I1wx = plane(B.I1wx); wa.I1wy = plane(B.I1wy); wa.rho_c = plane(B.rho);
        wa.ctrl = ctrl; wa.w = lw; wa.h = lh; wa.pitch = pitch[s]; wa.level = s; wa.stride = S;
        const dim3 gw(cdiv(lw, 32), cdiv(lh, 8), n);
        WarpArgs wc;   // cuda semantics: k_warp_cuda, persistent blocks per pair over its 32 x 16 tiles
        memset(wc.tmI1, 0, sizeof(wc.tmI1));   // not read by k_warp_cuda
        wc.I0 = wa.I0; wc.I1 = wa.I1;
        wc.u1[0] = ia.u1[0]; wc.u1[1] = ia.u1[1]; wc.u2[0] = ia.u2[0]; wc.u2[1] = ia.u2[1];
        wc.I1w = nullptr; wc.I1wx = wa.I1wx; wc.I1wy = wa.I1wy; wc.grad = nullptr; wc.rho_c = wa.rho_c;
        wc.w = lw; wc.h = lh; wc.pitch = pitch[s]; wc.level = s; wc.one = 1.0f; wc.ctrl = ctrl;
        const dim3 gwc(batch_blocks((long long)cdiv(lw, TVL1_WC_TW) * cdiv(lh, TVL1_WC_TH), 1, n), 1, n);

        for (int wi = 0; wi < W; ++wi) {
            const int slot = s * W + wi;
            ia.slot = slot;
            ma.slot = slot;
            // (2) warp; the level's first warp also zeroes p11 .. p22 and every warp re-arms the stop test
            for (int k = 0; k < 4; k++) wa.pz[k] = wc.pz[k] = wi == 0 ? plane(B.p[k]) : nullptr;
            if (cs) k_warp_cuda<true><<<gwc, dim3(32, 8), 0, st>>>(wc, S);
            else k_bwarp<<<gw, dim3(32, 8), 0, st>>>(wa);
            CK(cudaGetLastError());
            launches++;
            // (3) outer iterations, as calc_device: chunks of iterations enqueued without knowing how many run,
            // sized from the count the previous (level, warp) needed, one read-back of all pairs per chunk.  An
            // outer iteration ends when every pair is done or has used its inner budget.
            const int pred_total = wi > 0 ? counts[slot - 1] : (s < L - 1 ? counts[(s + 1) * W] : H->inner);
            std::fill(total.begin(), total.end(), 0);
            int least_total = 0;   // fewest iterations any pair not yet done has made in this (level, warp)
            for (int no = 0; no < H->outer; ++no) {
                if (P.median_filtering > 1 && !cs) {
                    if (P.median_filtering == 3) k_median3<<<gm, 256, 0, st>>>(ma, 2, S);
                    else k_bmedian5<<<gm, 256, 0, st>>>(ma, S);
                    CK(cudaGetLastError());
                    launches++;
                }
                CK(cudaMemset2DAsync(&ctrl->inner, S, 0, sizeof(int), n, st));
                int least_inner = 0, want = 0;   // fewest inner iterations of a pair still iterating
                for (;;) {
                    const int left_pred = pred_total - least_total - least_inner;
                    want = want == 0 ? (left_pred + 1 > 4 ? left_pred + 1 : 4) : 2 * want;
                    if (want > H->inner - least_inner) want = H->inner - least_inner;
                    for (int k = 0; k < want; ++k) {
                        if (cs) k_plain_u<2, true><<<gi, dim3(32, TVL1_PLAIN_NW), 0, st>>>(ia);
                        else if (with_gamma) k_plain_u<3><<<gi, dim3(32, TVL1_PLAIN_NW), 0, st>>>(ia);
                        else k_plain_u<2><<<gi, dim3(32, TVL1_PLAIN_NW), 0, st>>>(ia);
                        if (with_gamma) k_plain_p<3><<<gi, dim3(32, TVL1_PLAIN_NW), 0, st>>>(ia);
                        else k_plain_p<2><<<gi, dim3(32, TVL1_PLAIN_NW), 0, st>>>(ia);
                    }
                    CK(cudaGetLastError());
                    launches += 2 * want;
                    if ((rc = read_ctrl(hdr))) return rc;
                    least_inner = H->inner;
                    for (int b = 0; b < n; b++)
                        if (!hc[b].done && hc[b].inner < least_inner) least_inner = hc[b].inner;
                    if (least_inner >= H->inner) break;
                }
                bool all_done = true;
                least_total = INT32_MAX;
                for (int b = 0; b < n; b++) {
                    total[b] += hc[b].inner;   // 0 for a pair that was done before this outer iteration
                    if (!hc[b].done) { all_done = false; if (total[b] < least_total) least_total = total[b]; }
                }
                if (all_done) break;
            }
            counts[slot] = *std::max_element(total.begin(), total.end());
        }
        if (s == 0) break;
        // flow upsample to the next finer level, from the twin that holds each pair's flow, times 1/scaleStep
        ResizeArgs ra = resize_args(ia.u1[0], ia.u2[0], lw, lh, pitch[s], plane(B.u1[s - 1]), plane(B.u2[s - 1]), ws[s - 1],
                                    hs[s - 1], pitch[s - 1]);
        ra.src[0][1] = ia.u1[1]; ra.src[1][1] = ia.u2[1];
        ra.ctrl = ctrl; ra.level = s; ra.stride = S;
        const float mul = (float)(1 / P.scale_step);
        if ((rc = cs ? launch_resize_cuda(ra, n, 0.0, mul, 1, st) : launch_resize(ra, n, 0.0, mul, 1, st))) return rc;
        launches += 1;
        if (with_gamma) {   // u3 is zoomed like the flow but not scaled (one buffer: no ctrl)
            ResizeArgs r3 = resize_args(ia.u3, nullptr, lw, lh, pitch[s], plane(B.u3[s - 1]), nullptr, ws[s - 1], hs[s - 1],
                                        pitch[s - 1]);
            r3.stride = S;
            if ((rc = launch_resize(r3, n, 0.0, 1.f, 0, st))) return rc;
            launches += 1;
        }
    }
    // A.8: planar output of every pair, from the twin its final Ctrl names
    if ((rc = read_ctrl(sizeof(Ctrl)))) return rc;
    for (int b = 0; b < n; b++) {
        const size_t o = (size_t)b * S;
        const int uc = hc[b].ucur[0];
        CK(cudaMemcpy2DAsync(d_u[b], pitch_out, base + (uc ? B.u1x : B.u1[0]) + o, (size_t)pitch[0] * 4, (size_t)w * 4, h,
                             cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpy2DAsync(d_v[b], pitch_out, base + (uc ? B.u2x : B.u2[0]) + o, (size_t)pitch[0] * 4, (size_t)w * 4, h,
                             cudaMemcpyDeviceToDevice, st));
    }
    CK(cudaEventRecord(ev_end, st));
    CK(cudaStreamSynchronize(st));
    if (stats) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev_begin, ev_end);
        for (int b = 0; b < n; b++) {
            stats_counts(&stats[b], hc[b], L, W, ws, hs);
            stats[b].ms_total = ms;
            stats[b].launches = launches;
        }
    }
    return TVL1_OK;
}

}  // namespace tvl1

// =================================================================== C ABI

extern "C" {

const char* tvl1_version(void) { return "fibsem-optflow_b200 0.1 (sm_100a)"; }
const char* tvl1_last_error(void) { return tvl1::g_err; }

void tvl1_default_params(tvl1_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    // generate_TV_args defaults, reference src/optflow.cpp:503-512
    p->tau = 0.25; p->lambda = 0.05; p->theta = 0.3; p->nscales = 10; p->warps = 5;
    p->epsilon = 0.01; p->iterations = 300; p->scale_step = 0.8; p->gamma = 0.0;
    p->use_initial_flow = 0;
    p->inner_iterations = 0; p->outer_iterations = 0;   // derived from iterations
    p->median_filtering = 5;                             // CPU-class semantics (SURVEY.md T4)
}

int tvl1_create(const tvl1_params* p, int device, tvl1_handle** out)
{
    if (!out) return fail(TVL1_ERR_INVALID, "out is null");
    *out = nullptr;
    int rc = check_params(p);
    if (rc) return rc;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(TVL1_ERR_CUDA, "no CUDA device (%s); this library has no CPU path",
                    e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(TVL1_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    CK(cudaSetDevice(device));
    tvl1_handle* H = new tvl1_handle();
    H->device = device;
    H->prm = *p;
    resolve_iterations(H);
    e = cudaMallocHost(&H->h_ctrl, sizeof(Ctrl));
    if (e != cudaSuccess) { delete H; return fail(TVL1_ERR_CUDA, "cudaMallocHost: %s", cudaGetErrorString(e)); }
    memset(H->h_ctrl, 0, sizeof(Ctrl));
    e = cudaStreamCreateWithFlags(&H->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { cudaFreeHost(H->h_ctrl); delete H; return fail(TVL1_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    rc = upload_cubic_table(device);
    if (rc) { tvl1_destroy(H); return rc; }
    *out = H;
    return TVL1_OK;
}

void tvl1_destroy(tvl1_handle* H)
{
    if (!H) return;
    cudaSetDevice(H->device);
    tvl1::release_arena(H);
    tvl1::release_batch(H);
    if (H->h_ctrl) cudaFreeHost(H->h_ctrl);
    if (H->d_f0) cudaFree(H->d_f0);
    if (H->d_f1) cudaFree(H->d_f1);
    if (H->d_uo) cudaFree(H->d_uo);
    if (H->d_vo) cudaFree(H->d_vo);
    if (H->d_ui) cudaFree(H->d_ui);
    if (H->d_vi) cudaFree(H->d_vi);
    tvl1::sampler_release(H->samp);
    tvl1::features_release(H->feat);
    for (int i = 0; i < TVL1_STACK_SLOTS; i++) { if (H->st_slice[i]) cudaFree(H->st_slice[i]); if (H->st_up[i]) cudaEventDestroy(H->st_up[i]); }
    for (int i = 0; i < 2; i++) if (H->st_raw[i]) cudaFree(H->st_raw[i]);
    for (int i = 0; i < 2; i++) {
        for (int j = 0; j < 2; j++) if (H->st_flow[i][j]) cudaFree(H->st_flow[i][j]);
        if (H->st_ready[i]) cudaEventDestroy(H->st_ready[i]);
        if (H->st_down[i]) cudaEventDestroy(H->st_down[i]);
    }
    if (H->st_in) cudaStreamDestroy(H->st_in);
    if (H->st_out) cudaStreamDestroy(H->st_out);
    for (cudaEvent_t e : H->events) cudaEventDestroy(e);
    if (H->own_stream) cudaStreamDestroy(H->own_stream);
    delete H;
}

int tvl1_set_params(tvl1_handle* H, const tvl1_params* p)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    int rc = check_params(p);
    if (rc) return rc;
    H->prm = *p;
    return resolve_iterations(H);
}

int tvl1_set_option(tvl1_handle* H, const char* key, double value)
{
    if (!H || !key) return fail(TVL1_ERR_INVALID, "null handle or key");
    if (!strcmp(key, "fused_min_px")) { H->fused_min_px = value < 0 ? 0 : (long long)value; return TVL1_OK; }
    if (!strcmp(key, "multi_iter")) { H->multi_iter = value != 0; return TVL1_OK; }
    if (!strcmp(key, "coop_outer")) { H->coop_outer = value != 0; return TVL1_OK; }
    return fail(TVL1_ERR_INVALID, "unknown option '%s'", key);
}

int tvl1_set_timing(tvl1_handle* H, int enabled)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    H->timing = enabled != 0;
    return TVL1_OK;
}

int tvl1_calc_ex(tvl1_handle* H, int frame_type, const void* d_frame0, size_t pitch0, const void* d_frame1,
                 size_t pitch1, int width, int height, const float* d_u0, const float* d_v0, size_t pitch_init,
                 float* d_u, float* d_v, size_t pitch_out, void* stream, tvl1_stats* stats)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    return calc_device(H, frame_type, d_frame0, pitch0, d_frame1, pitch1, width, height, d_u0, d_v0, pitch_init, d_u, d_v,
                       pitch_out, (cudaStream_t)stream, stats);
}

int tvl1_calc_u8(tvl1_handle* H, const uint8_t* d_frame0, size_t pitch0, const uint8_t* d_frame1, size_t pitch1,
                 int width, int height, float* d_u, float* d_v, size_t pitch_out, void* stream, tvl1_stats* stats)
{
    return tvl1_calc_ex(H, TVL1_FRAME_U8, d_frame0, pitch0, d_frame1, pitch1, width, height, nullptr, nullptr, 0, d_u, d_v,
                        pitch_out, stream, stats);
}

int tvl1_calc_ex_host(tvl1_handle* H, int frame_type, const void* h_frame0, size_t pitch0, const void* h_frame1,
                      size_t pitch1, int width, int height, const float* h_u0, const float* h_v0, size_t pitch_init,
                      float* h_u, float* h_v, size_t pitch_out, tvl1_stats* stats)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    if (!h_frame0 || !h_frame1 || !h_u || !h_v) return fail(TVL1_ERR_INVALID, "null image or flow pointer");
    int rc = check_frames(frame_type, pitch0, pitch1, width, height, h_u0, h_v0, pitch_init, pitch_out);
    if (rc) return rc;
    CK(cudaSetDevice(H->device));
    const size_t row = (size_t)width * (frame_type == TVL1_FRAME_F32 ? 4 : 1);
    const size_t plane = (size_t)width * height * 4;
    if (H->stage_w != width || H->stage_h != height || H->stage_pitch < row) {
        void** bufs[6] = {&H->d_f0, &H->d_f1, (void**)&H->d_uo, (void**)&H->d_vo, (void**)&H->d_ui, (void**)&H->d_vi};
        for (void** b : bufs) { if (*b) cudaFree(*b); *b = nullptr; }
        H->stage_w = H->stage_h = 0;
        H->stage_pitch = (size_t)round_up((int)row, 128);
        CK(cudaMalloc(&H->d_f0, H->stage_pitch * height));
        CK(cudaMalloc(&H->d_f1, H->stage_pitch * height));
        CK(cudaMalloc(&H->d_uo, plane));
        CK(cudaMalloc(&H->d_vo, plane));
        H->stage_w = width; H->stage_h = height;
    }
    if (h_u0 && !H->d_ui) {
        CK(cudaMalloc(&H->d_ui, plane));
        CK(cudaMalloc(&H->d_vi, plane));
    }
    cudaStream_t st = H->own_stream;
    CK(cudaMemcpy2DAsync(H->d_f0, H->stage_pitch, h_frame0, pitch0, row, height, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpy2DAsync(H->d_f1, H->stage_pitch, h_frame1, pitch1, row, height, cudaMemcpyHostToDevice, st));
    if (h_u0) {
        CK(cudaMemcpy2DAsync(H->d_ui, (size_t)width * 4, h_u0, pitch_init, (size_t)width * 4, height, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpy2DAsync(H->d_vi, (size_t)width * 4, h_v0, pitch_init, (size_t)width * 4, height, cudaMemcpyHostToDevice, st));
    }
    rc = calc_device(H, frame_type, H->d_f0, H->stage_pitch, H->d_f1, H->stage_pitch, width, height,
                     h_u0 ? H->d_ui : nullptr, h_u0 ? H->d_vi : nullptr, (size_t)width * 4, H->d_uo, H->d_vo,
                     (size_t)width * 4, st, stats);
    if (rc) return rc;
    CK(cudaMemcpy2DAsync(h_u, pitch_out, H->d_uo, (size_t)width * 4, (size_t)width * 4, height, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpy2DAsync(h_v, pitch_out, H->d_vo, (size_t)width * 4, (size_t)width * 4, height, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return TVL1_OK;
}

int tvl1_calc_batch_ex(tvl1_handle* H, int n, int frame_type, const void* const* d_frame0, size_t pitch0,
                       const void* const* d_frame1, size_t pitch1, int width, int height,
                       const float* const* d_u0, const float* const* d_v0, size_t pitch_init,
                       float* const* d_u, float* const* d_v, size_t pitch_out, void* stream, tvl1_stats* stats)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    return calc_batch(H, n, frame_type, d_frame0, pitch0, d_frame1, pitch1, width, height, d_u0, d_v0, pitch_init, d_u, d_v,
                      pitch_out, (cudaStream_t)stream, stats);
}

int tvl1_calc_batch_u8(tvl1_handle* H, int n, const uint8_t* const* d_frame0, size_t pitch0,
                       const uint8_t* const* d_frame1, size_t pitch1, int width, int height,
                       float* const* d_u, float* const* d_v, size_t pitch_out, void* stream, tvl1_stats* stats)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    if (H->prm.semantics == TVL1_SEMANTICS_CUDA)
        return fail(TVL1_ERR_UNSUPPORTED, "tvl1_calc_batch_u8 solves in CPU-class semantics only, not cuda semantics");
    if (H->prm.gamma != 0.0) return fail(TVL1_ERR_UNSUPPORTED, "tvl1_calc_batch_u8 does not support gamma != 0");
    return calc_batch(H, n, TVL1_FRAME_U8, (const void* const*)d_frame0, pitch0, (const void* const*)d_frame1, pitch1, width,
                      height, nullptr, nullptr, 0, d_u, d_v, pitch_out, (cudaStream_t)stream, stats);
}

int tvl1_last_readbacks(const tvl1_handle* H, long long* n)
{
    if (!H || !n) return fail(TVL1_ERR_INVALID, "null handle or output");
    *n = H->readbacks;
    return TVL1_OK;
}

int tvl1_calc_u8_host(tvl1_handle* H, const uint8_t* h_frame0, size_t pitch0, const uint8_t* h_frame1, size_t pitch1,
                      int width, int height, float* h_u, float* h_v, size_t pitch_out, tvl1_stats* stats)
{
    return tvl1_calc_ex_host(H, TVL1_FRAME_U8, h_frame0, pitch0, h_frame1, pitch1, width, height, nullptr, nullptr, 0,
                             h_u, h_v, pitch_out, stats);
}

static int launch_mask_flow(const uint8_t* f1, size_t pitch1, int w, int h, float* u, float* v, size_t pitch_f, int add_grid,
                            cudaStream_t st)
{
    dim3 b(32, 8);
    dim3 g(cdiv(cdiv(w, 4), 32), cdiv(h, 8));
    k_mask_flow<<<g, b, 0, st>>>(f1, pitch1, w, h, u, v, pitch_f, add_grid);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_finish_flow_u8(tvl1_handle* H, const uint8_t* d_frame1, size_t pitch1, int width, int height,
                        float* d_u, float* d_v, size_t pitch_out, int add_grid, void* stream)
{
    if (!H) return fail(TVL1_ERR_INVALID, "handle is null");
    if (!d_u || !d_v || width <= 0 || height <= 0 || pitch_out % 4) return fail(TVL1_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(H->device));
    return launch_mask_flow(d_frame1, pitch1, width, height, d_u, d_v, pitch_out / 4, add_grid > 0 ? 1 : (add_grid < 0 ? -1 : 0),
                            (cudaStream_t)stream);
}

int tvl1_mask_flow_u8(tvl1_handle* H, const uint8_t* d_frame1, size_t pitch1, int width, int height,
                      float* d_u, float* d_v, size_t pitch_out, void* stream)
{
    if (!d_frame1) return fail(TVL1_ERR_INVALID, "frame1 is null");
    return tvl1_finish_flow_u8(H, d_frame1, pitch1, width, height, d_u, d_v, pitch_out, 0, stream);
}

// ---- stack of adjacent slices

static int stack_reserve(tvl1_handle* H, int w, int h)
{
    if (!H->st_in) {
        CK(cudaStreamCreateWithFlags(&H->st_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&H->st_out, cudaStreamNonBlocking));
        for (int i = 0; i < TVL1_STACK_SLOTS; i++) CK(cudaEventCreateWithFlags(&H->st_up[i], cudaEventDisableTiming));
        for (int i = 0; i < 2; i++) {
            CK(cudaEventCreateWithFlags(&H->st_ready[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&H->st_down[i], cudaEventDisableTiming));
        }
    }
    if (H->st_w == w && H->st_h == h) return TVL1_OK;
    for (int i = 0; i < TVL1_STACK_SLOTS; i++) { if (H->st_slice[i]) cudaFree(H->st_slice[i]); H->st_slice[i] = nullptr; }
    for (int i = 0; i < 2; i++)
        for (int j = 0; j < 2; j++) { if (H->st_flow[i][j]) cudaFree(H->st_flow[i][j]); H->st_flow[i][j] = nullptr; }
    H->st_w = H->st_h = 0;
    H->st_pitch8 = (size_t)round_up(w, 128);
    for (int i = 0; i < TVL1_STACK_SLOTS; i++) CK(cudaMalloc(&H->st_slice[i], H->st_pitch8 * h));
    for (int i = 0; i < 2; i++)
        for (int j = 0; j < 2; j++) CK(cudaMalloc(&H->st_flow[i][j], (size_t)w * h * sizeof(float)));
    H->st_w = w; H->st_h = h;
    return TVL1_OK;
}

int tvl1_stack_run(tvl1_handle* H, const tvl1_stack_io* io, float* ms_total)
{
    if (!H || !io) return fail(TVL1_ERR_INVALID, "null handle or io");
    const int n = io->n_slices;
    const int rw = io->width, rh = io->height;          // size of the slices as given
    int w = rw, h = rh;                                 // size the solver works at
    const bool pre = io->prescale > 0.0 && io->prescale != 1.0;
    const bool listed = io->pair_p != nullptr || io->pair_q != nullptr;   // explicit (p, q) pairs instead of (k, k+1)
    if (!io->h_slices || n < 2 || rw <= 0 || rh <= 0 || io->pitch < (size_t)rw)
        return fail(TVL1_ERR_INVALID, "a stack needs >= 2 slices of non-zero size");
    if (listed && (!io->pair_p || !io->pair_q || io->n_pairs < 1)) return fail(TVL1_ERR_INVALID, "pair_p, pair_q and n_pairs go together");
    const int npairs = listed ? io->n_pairs : n - 1;
    if (pre) { int r = tvl1_prescaled_size(rw, rh, io->prescale, &w, &h); if (r) return r; }
    if ((io->h_u == nullptr) != (io->h_v == nullptr)) return fail(TVL1_ERR_INVALID, "h_u and h_v go together");
    if (io->h_u && io->pitch_out < (size_t)w * 4) return fail(TVL1_ERR_INVALID, "pitch_out smaller than a row");
    if (io->npoints >= 0 && (!io->px || !io->py || !io->qx || !io->qy || !io->w || !io->n_out))
        return fail(TVL1_ERR_INVALID, "match output arrays missing");
    for (int k = 0; k < n; k++) if (!io->h_slices[k]) return fail(TVL1_ERR_INVALID, "slice %d is null", k);
    auto pp = [&](int k) { return listed ? io->pair_p[k] : k; };
    auto pq = [&](int k) { return listed ? io->pair_q[k] : k + 1; };
    for (int k = 0; k < npairs; k++)
        if (pp(k) < 0 || pp(k) >= n || pq(k) < 0 || pq(k) >= n) return fail(TVL1_ERR_INVALID, "pair %d names a slice outside the stack", k);
    CK(cudaSetDevice(H->device));
    int rc = stack_reserve(H, w, h);
    if (rc) return rc;
    if (pre && H->st_raw_bytes < (size_t)rw * rh) {
        for (int i = 0; i < 2; i++) {
            if (H->st_raw[i]) cudaFree(H->st_raw[i]);
            H->st_raw[i] = nullptr;
        }
        H->st_raw_bytes = 0;
        for (int i = 0; i < 2; i++) CK(cudaMalloc(&H->st_raw[i], (size_t)rw * rh));
        H->st_raw_bytes = (size_t)rw * rh;
    }
    cudaStream_t cs = H->own_stream;
    const size_t p8 = H->st_pitch8;
    const int cap = io->npoints > 0 ? io->npoints : 1;
    struct EventPair {
        cudaEvent_t a = nullptr, b = nullptr;
        ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    } tev;
    CK(cudaEventCreate(&tev.a));
    CK(cudaEventCreate(&tev.b));
    cudaEvent_t t0 = tev.a, t1 = tev.b;
    CK(cudaEventRecord(t0, cs));
    // Device slots for the (prescaled) slices, kept by slice index: the slice two adjacent pairs share goes
    // up once (src/optflow.cpp:97-103), and the frames of pair k+1 arrive on the copy stream while pair k is
    // being solved.  `held[s]`: last pair that reads slot s -- a slot is only refilled once that pair's solve
    // has completed (the solves are synchronous to the host, so "completed" is known here).
    const int NS = TVL1_STACK_SLOTS;
    int tag[NS], held[NS];
    for (int s = 0; s < NS; s++) { tag[s] = -1; held[s] = -1; }
    int uploads = 0;
    auto find = [&](int slice) { for (int s = 0; s < NS; s++) if (tag[s] == slice) return s; return -1; };
    // slot for `slice` if it is resident or can be brought in without touching a slot that pair `busy` (or a later
    // one) reads
    auto stage = [&](int slice, int for_pair, int busy, int* out) -> int {
        int s = find(slice);
        if (s < 0) {
            for (int c = 0; c < NS; c++)
                if (held[c] < busy && (s < 0 || held[c] < held[s])) s = c;
            if (s < 0) { *out = -1; return TVL1_OK; }   // every slot is still in use: later
            tag[s] = slice;
            if (!pre) {
                CK(cudaMemcpy2DAsync(H->st_slice[s], p8, io->h_slices[slice], io->pitch, w, h, cudaMemcpyHostToDevice, H->st_in));
            } else {
                // raw slice -> device, then the loader's 8-bit resize (src/optflow.cpp:111,124) on the
                // copy stream: the solver never sees the raw size.  Two staging buffers, re-used in stream
                // order (an upload follows the prescale that last read the buffer, on the same stream)
                uint8_t* raw = H->st_raw[uploads & 1];
                CK(cudaMemcpy2DAsync(raw, (size_t)rw, io->h_slices[slice], io->pitch, rw, rh, cudaMemcpyHostToDevice, H->st_in));
                int r = tvl1_prescale_u8(raw, (size_t)rw, rw, rh, io->prescale, H->st_slice[s], p8, H->st_in);
                if (r) return r;
            }
            uploads++;
            CK(cudaEventRecord(H->st_up[s], H->st_in));
        }
        if (held[s] < for_pair) held[s] = for_pair;
        *out = s;
        return TVL1_OK;
    };
    long long rand_skip = 0;
    for (int k = 0; k < npairs; k++) {
        const int fb = k & 1;
        int s0 = -1, s1 = -1, tmp = -1;
        // this pair's frames (pair k-1 has completed: only pair k itself pins slots now)
        if ((rc = stage(pp(k), k, k, &s0)) || (rc = stage(pq(k), k, k, &s1))) return rc;
        if (s0 < 0 || s1 < 0) return fail(TVL1_ERR_CUDA, "no free slice slot (internal)");
        // the next pair's frames go up now, into slots this pair does not read
        if (k + 1 < npairs) {
            if ((rc = stage(pp(k + 1), k + 1, k, &tmp)) || (rc = stage(pq(k + 1), k + 1, k, &tmp))) return rc;
        }
        CK(cudaStreamWaitEvent(cs, H->st_up[s0], 0));
        CK(cudaStreamWaitEvent(cs, H->st_up[s1], 0));
        if (k >= 2 && io->h_u) CK(cudaStreamWaitEvent(cs, H->st_down[fb], 0));   // flow buffer still draining
        float* du = H->st_flow[fb][0];
        float* dv = H->st_flow[fb][1];
        rc = calc_device(H, TVL1_FRAME_U8, H->st_slice[s0], p8, H->st_slice[s1], p8, w, h, nullptr, nullptr, 0, du, dv,
                         (size_t)w * 4, cs, io->stats ? &io->stats[k] : nullptr);
        if (rc) return rc;
        if (io->apply_mask && (rc = launch_mask_flow(H->st_slice[s1], p8, w, h, du, dv, (size_t)w, 0, cs))) return rc;
        if (io->npoints >= 0) {
            long long used = 0;
            const size_t o = (size_t)k * cap;
            rc = tvl1_sample_matches_skip(H, H->st_slice[s0], p8, H->st_slice[s1], p8, du, dv, (size_t)w * 4, w, h,
                                          0, 0, 0, 0, io->scale, io->npoints, io->seed, io->seed < 0 ? rand_skip : 0,
                                          io->px + o, io->py + o, io->qx + o, io->qy + o, io->w + o, nullptr,
                                          &io->n_out[k], &used, cs);
            if (rc) return rc;
            rand_skip += used;
        } else if (io->apply_mask) {
            CK(cudaStreamSynchronize(cs));   // slot s1 is read by the mask kernel: done before it can be refilled
        }
        if (io->h_u) {
            CK(cudaEventRecord(H->st_ready[fb], cs));
            CK(cudaStreamWaitEvent(H->st_out, H->st_ready[fb], 0));
            CK(cudaMemcpy2DAsync(io->h_u[k], io->pitch_out, du, (size_t)w * 4, (size_t)w * 4, h, cudaMemcpyDeviceToHost, H->st_out));
            CK(cudaMemcpy2DAsync(io->h_v[k], io->pitch_out, dv, (size_t)w * 4, (size_t)w * 4, h, cudaMemcpyDeviceToHost, H->st_out));
            CK(cudaEventRecord(H->st_down[fb], H->st_out));
        }
    }
    CK(cudaStreamSynchronize(H->st_out));
    CK(cudaStreamSynchronize(H->st_in));
    CK(cudaEventRecord(t1, cs));
    CK(cudaEventSynchronize(t1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, t0, t1);
    if (ms_total) *ms_total = ms;
    return TVL1_OK;
}

// ---- stage-level entry points

// CUDA-event bracket around the launches of the most recent stage-level call (tvl1_k_last_ms)
static thread_local cudaEvent_t t_ev0 = nullptr, t_ev1 = nullptr;
static void stage_begin(cudaStream_t st)
{
    if (!t_ev0) { cudaEventCreate(&t_ev0); cudaEventCreate(&t_ev1); }
    cudaEventRecord(t_ev0, st);
}
static void stage_end(cudaStream_t st) { cudaEventRecord(t_ev1, st); }

int tvl1_k_last_ms(float* ms)
{
    if (!ms || !t_ev0) return fail(TVL1_ERR_INVALID, "no stage-level call has been timed on this thread");
    CK(cudaEventSynchronize(t_ev1));
    CK(cudaEventElapsedTime(ms, t_ev0, t_ev1));
    return TVL1_OK;
}

int tvl1_k_convert_u8(const uint8_t* d_src, size_t pitch_bytes, int w, int h, float* d_dst, int pitch, void* stream)
{
    if (!d_src || !d_dst || w <= 0 || h <= 0 || pitch % 4 || pitch < w || pitch_bytes < (size_t)w)
        return fail(TVL1_ERR_INVALID, "bad argument");
    return launch_convert(d_src, pitch_bytes, w, h, d_dst, pitch, (cudaStream_t)stream);
}

int tvl1_k_convert_f32(const float* d_src, size_t pitch_bytes, int w, int h, float* d_dst, int pitch, void* stream)
{
    if (!d_src || !d_dst || w <= 0 || h <= 0 || pitch % 4 || pitch < w || pitch_bytes % 4 || pitch_bytes < (size_t)w * 4)
        return fail(TVL1_ERR_INVALID, "bad argument");
    return launch_convert_f32(d_src, pitch_bytes, w, h, d_dst, pitch, (cudaStream_t)stream);
}

int tvl1_k_resize(const float* d_src, int sw, int sh, int spitch, float* d_dst, int dw, int dh, int dpitch,
                  double inv_scale, float mul, void* stream)
{
    if (!d_src || !d_dst || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0) return fail(TVL1_ERR_INVALID, "bad argument");
    return launch_resize(resize_args(d_src, nullptr, sw, sh, spitch, d_dst, nullptr, dw, dh, dpitch), 1, inv_scale, mul,
                         mul != 1.f, (cudaStream_t)stream);
}

int tvl1_k_resize_cuda(const float* d_src, int sw, int sh, int spitch, float* d_dst, int dw, int dh, int dpitch,
                       double inv_scale, float mul, void* stream)
{
    if (!d_src || !d_dst || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || spitch < sw || dpitch < dw)
        return fail(TVL1_ERR_INVALID, "bad argument");
    return launch_resize_cuda(resize_args(d_src, nullptr, sw, sh, spitch, d_dst, nullptr, dw, dh, dpitch), 1, inv_scale, mul,
                              mul != 1.f, (cudaStream_t)stream);
}

int tvl1_k_centered_gradient(const float* d_src, int w, int h, int pitch, float* d_dx, float* d_dy, void* stream)
{
    if (!d_src || !d_dx || !d_dy || w <= 0 || h <= 0) return fail(TVL1_ERR_INVALID, "bad argument");
    return launch_gradient(d_src, w, h, pitch, d_dx, d_dy, (cudaStream_t)stream);
}

int tvl1_k_warp(const float* d_I0, const float* d_I1, const float* d_u1, const float* d_u2, int w, int h,
                int pitch, float* d_I1w, float* d_I1wx, float* d_I1wy, float* d_grad, float* d_rho_c, void* stream)
{
    if (!d_I0 || !d_I1 || !d_u1 || !d_u2 || !d_I1wx || !d_I1wy || !d_rho_c || w <= 0 || h <= 0 || pitch % 4 || pitch < w)
        return fail(TVL1_ERR_INVALID, "bad argument");
    int dev = 0;
    CK(cudaGetDevice(&dev));
    int rc = upload_cubic_table(dev);
    if (rc) return rc;
    WarpArgs a;
    a.I0 = d_I0; a.I1 = d_I1;
    a.u1[0] = a.u1[1] = d_u1; a.u2[0] = a.u2[1] = d_u2;
    a.I1w = d_I1w; a.I1wx = d_I1wx; a.I1wy = d_I1wy; a.grad = d_grad; a.rho_c = d_rho_c;
    a.w = w; a.h = h; a.pitch = pitch; a.level = -1; a.ctrl = nullptr; a.one = 1.0f;
    for (int k = 0; k < 4; k++) a.pz[k] = nullptr;
    for (int k = 0; k < 2; k++)
        if ((rc = make_plane_map(&a.tmI1[k], d_I1, pitch, h, TVL1_WP_RW, k == 0 ? 16 : TVL1_WP_RH))) return rc;
    stage_begin((cudaStream_t)stream);
    rc = launch_warp(a, (cudaStream_t)stream);
    stage_end((cudaStream_t)stream);
    return rc;
}

int tvl1_k_warp_cuda(const float* d_I0, const float* d_I1, const float* d_u1, const float* d_u2, int w, int h,
                     int pitch, float* d_I1w, float* d_I1wx, float* d_I1wy, float* d_grad, float* d_rho_c, void* stream)
{
    if (!d_I0 || !d_I1 || !d_u1 || !d_u2 || !d_I1wx || !d_I1wy || !d_rho_c || w <= 0 || h <= 0 || pitch < w)
        return fail(TVL1_ERR_INVALID, "bad argument");
    WarpArgs a;
    memset(a.tmI1, 0, sizeof(a.tmI1));   // k_warp_cuda stages its windows with plain loads
    a.I0 = d_I0; a.I1 = d_I1;
    a.u1[0] = a.u1[1] = d_u1; a.u2[0] = a.u2[1] = d_u2;
    a.I1w = d_I1w; a.I1wx = d_I1wx; a.I1wy = d_I1wy; a.grad = d_grad; a.rho_c = d_rho_c;
    a.w = w; a.h = h; a.pitch = pitch; a.level = -1; a.ctrl = nullptr; a.one = 1.0f;
    for (int k = 0; k < 4; k++) a.pz[k] = nullptr;
    stage_begin((cudaStream_t)stream);
    const int rc = launch_warp_cuda(a, (cudaStream_t)stream);
    stage_end((cudaStream_t)stream);
    return rc;
}

static int k_iterate_impl(int fused, const float* d_I1wx, const float* d_I1wy, const float* d_grad, const float* d_rho_c,
                   float* d_u1, float* d_u2, float* d_p11, float* d_p12, float* d_p21, float* d_p22,
                   int w, int h, int pitch, float l_t, float theta, float taut, int n, double* errors, void* stream)
{
    if (!d_I1wx || !d_I1wy || !d_grad || !d_rho_c || !d_u1 || !d_u2 || !d_p11 || !d_p12 || !d_p21 || !d_p22 ||
        w <= 0 || h <= 0 || pitch % 4 || pitch < w || n < 0)
        return fail(TVL1_ERR_INVALID, "bad argument");
    if (n > TVL1_MAX_LEVELS * TVL1_MAX_WARPS) return fail(TVL1_ERR_INVALID, "n too large");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t pb = (size_t)pitch * h * sizeof(float);
    const size_t nb = iterate_max_blocks();
    char* tmp = nullptr;
    // the two-iteration pass fills its ring by bulk tensor copies of whole sections (IterMaps): its operands are
    // staged as 15 equally spaced planes {I1wx, I1wy, rho_c | u1, u2 | u1', u2' | p11..p22 | p11'..p22'}; the
    // one-iteration kernel works on the caller's planes with 6 twins
    const int nplanes = fused ? 15 : 6;
    const size_t ctrl_off = nplanes * pb, part_off = ctrl_off + 1024 * ((sizeof(Ctrl) + 1023) / 1024);
    const size_t log_off = part_off + nb * sizeof(double);
    const size_t total = log_off + (size_t)(n + 1) * sizeof(double);
    CK(cudaMalloc(&tmp, total));
    cudaError_t e = cudaMemsetAsync(tmp, 0, total, st);
    if (e != cudaSuccess) { cudaFree(tmp); return fail(TVL1_ERR_CUDA, "memset: %s", cudaGetErrorString(e)); }
    float* tw[15];
    for (int k = 0; k < nplanes; k++) tw[k] = (float*)(tmp + k * pb);
    float* const user[6] = {d_u1, d_u2, d_p11, d_p12, d_p21, d_p22};
    IterArgs a;
    if (fused) {
        const float* cs[3] = {d_I1wx, d_I1wy, d_rho_c};
        for (int k = 0; k < 3; k++) cudaMemcpyAsync(tw[k], cs[k], pb, cudaMemcpyDeviceToDevice, st);
        for (int k = 0; k < 2; k++) cudaMemcpyAsync(tw[3 + k], user[k], pb, cudaMemcpyDeviceToDevice, st);
        for (int k = 0; k < 4; k++) cudaMemcpyAsync(tw[7 + k], user[2 + k], pb, cudaMemcpyDeviceToDevice, st);
        a.I1wx = tw[0]; a.I1wy = tw[1]; a.rho_c = tw[2];
        a.u1[0] = tw[3]; a.u2[0] = tw[4]; a.u1[1] = tw[5]; a.u2[1] = tw[6];
        a.p11[0] = tw[7]; a.p12[0] = tw[8]; a.p21[0] = tw[9]; a.p22[0] = tw[10];
        a.p11[1] = tw[11]; a.p12[1] = tw[12]; a.p21[1] = tw[13]; a.p22[1] = tw[14];
    } else {
        a.I1wx = d_I1wx; a.I1wy = d_I1wy; a.rho_c = d_rho_c;   // grad is recomputed in the kernel
        a.u1[0] = d_u1; a.u1[1] = tw[0]; a.u2[0] = d_u2; a.u2[1] = tw[1];
        a.p11[0] = d_p11; a.p11[1] = tw[2]; a.p12[0] = d_p12; a.p12[1] = tw[3];
        a.p21[0] = d_p21; a.p21[1] = tw[4]; a.p22[0] = d_p22; a.p22[1] = tw[5];
    }
    a.w = w; a.h = h; a.pitch = pitch; a.l_t = l_t; a.theta = theta; a.taut = taut; a.one = 1.0f;
    a.scaled_eps = -1.f;   // never stops
    a.level = 0; a.slot = 0; a.mode = 0; a.inner_max = 1 << 30;
    a.ctrl = (Ctrl*)(tmp + ctrl_off);
    a.partials = (double*)(tmp + part_off);
    a.errlog = (double*)(tmp + log_off);
    int rc = TVL1_OK;
    if (fused && (rc = make_iter_maps(a))) { cudaFree(tmp); return rc; }
    stage_begin(st);
    if (fused == 2) {
        // the shipped schedule: ONE cooperative k_outer launch runs all n iterations (two-iteration
        // passes, plus one single pass when n is odd); scaled_eps < 0 keeps the stop test from firing
        a.mode = 2; a.inner_max = n;
        if (n > 0) rc = launch_outer(a, st);
    } else if (fused) { for (int i = 0; i + 1 < n && !rc; i += 2) rc = launch_iterate2(a, st); }
    else { for (int i = 0; i < n && !rc; i++) rc = launch_iterate(a, st); }
    stage_end(st);
    // passes made = buffer flips: n single passes, n/2 fused ones, n/2 + n%2 inside k_outer.  The copy back
    // covers the kernels' write width (w rounded up to 4), so the caller's padding beyond it stays untouched
    const int flips = fused == 2 ? n / 2 + (n & 1) : (fused ? n / 2 : n);
    if (!rc && (fused || (flips & 1))) {
        const int t = flips & 1;
        float* const src[6] = {a.u1[t], a.u2[t], a.p11[t], a.p12[t], a.p21[t], a.p22[t]};
        const size_t row = (size_t)pitch * sizeof(float), cols = (size_t)((w + 3) & ~3) * sizeof(float);
        for (int k = 0; k < 6 && !rc; k++)
            if (cudaMemcpy2DAsync(user[k], row, src[k], row, cols, h, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
                rc = fail(TVL1_ERR_CUDA, "copy back failed");
    }
    if (!rc && errors && n > 0 &&
        (e = cudaMemcpyAsync(errors, tmp + log_off, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
        rc = fail(TVL1_ERR_CUDA, "error log copy failed: %s", cudaGetErrorString(e));
    e = cudaStreamSynchronize(st);
    if (!rc && e != cudaSuccess) rc = fail(TVL1_ERR_CUDA, "iterate: %s", cudaGetErrorString(e));
    cudaFree(tmp);
    return rc;
}

int tvl1_k_iterate(const float* d_I1wx, const float* d_I1wy, const float* d_grad, const float* d_rho_c,
                   float* d_u1, float* d_u2, float* d_p11, float* d_p12, float* d_p21, float* d_p22,
                   int w, int h, int pitch, float l_t, float theta, float taut, int n, double* errors, void* stream)
{
    return k_iterate_impl(0, d_I1wx, d_I1wy, d_grad, d_rho_c, d_u1, d_u2, d_p11, d_p12, d_p21, d_p22, w, h, pitch,
                          l_t, theta, taut, n, errors, stream);
}

int tvl1_k_iterate_fused2(const float* d_I1wx, const float* d_I1wy, const float* d_grad, const float* d_rho_c,
                          float* d_u1, float* d_u2, float* d_p11, float* d_p12, float* d_p21, float* d_p22,
                          int w, int h, int pitch, float l_t, float theta, float taut, int n, double* errors,
                          void* stream)
{
    if (n & 1) return fail(TVL1_ERR_INVALID, "the fused kernel advances two iterations per launch: n must be even");
    return k_iterate_impl(1, d_I1wx, d_I1wy, d_grad, d_rho_c, d_u1, d_u2, d_p11, d_p12, d_p21, d_p22, w, h, pitch,
                          l_t, theta, taut, n, errors, stream);
}

int tvl1_k_outer(const float* d_I1wx, const float* d_I1wy, const float* d_grad, const float* d_rho_c,
                 float* d_u1, float* d_u2, float* d_p11, float* d_p12, float* d_p21, float* d_p22,
                 int w, int h, int pitch, float l_t, float theta, float taut, int n, double* errors, void* stream)
{
    return k_iterate_impl(2, d_I1wx, d_I1wy, d_grad, d_rho_c, d_u1, d_u2, d_p11, d_p12, d_p21, d_p22, w, h, pitch,
                          l_t, theta, taut, n, errors, stream);
}

int tvl1_k_iterate_gamma(const float* d_I1wx, const float* d_I1wy, const float* d_rho_c,
                         float* d_u1, float* d_u2, float* d_u3, float* d_p11, float* d_p12,
                         float* d_p21, float* d_p22, float* d_p31, float* d_p32, int w, int h,
                         int pitch, float l_t, float theta, float taut, float gamma, int n,
                         double* errors, void* stream)
{
    if (!d_I1wx || !d_I1wy || !d_rho_c || !d_u1 || !d_u2 || !d_u3 || !d_p11 || !d_p12 || !d_p21 || !d_p22 ||
        !d_p31 || !d_p32 || w <= 0 || h <= 0 || pitch % 4 || pitch < w || n < 0)
        return fail(TVL1_ERR_INVALID, "bad argument");
    if (n > TVL1_MAX_LEVELS * TVL1_MAX_WARPS) return fail(TVL1_ERR_INVALID, "n too large");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nb = iterate_max_blocks();
    char* tmp = nullptr;
    const size_t part_off = 1024 * ((sizeof(Ctrl) + 1023) / 1024);
    const size_t log_off = part_off + nb * sizeof(double);
    const size_t total = log_off + (size_t)(n + 1) * sizeof(double);
    CK(cudaMalloc(&tmp, total));
    cudaError_t e = cudaMemsetAsync(tmp, 0, total, st);
    if (e != cudaSuccess) { cudaFree(tmp); return fail(TVL1_ERR_CUDA, "memset: %s", cudaGetErrorString(e)); }
    PlainIterArgs a = {};
    a.I1wx = d_I1wx; a.I1wy = d_I1wy; a.rho_c = d_rho_c;
    a.u1[0] = a.u1[1] = d_u1; a.u2[0] = a.u2[1] = d_u2; a.u3 = d_u3;
    a.p11 = d_p11; a.p12 = d_p12; a.p21 = d_p21; a.p22 = d_p22; a.p31 = d_p31; a.p32 = d_p32;
    a.w = w; a.h = h; a.pitch = pitch; a.l_t = l_t; a.theta = theta; a.taut = taut; a.gamma = gamma;
    a.scaled_eps = -1.f;   // never stops
    a.level = 0; a.slot = 0; a.inner_max = 1 << 30;
    a.ctrl = (Ctrl*)tmp; a.partials = (double*)(tmp + part_off); a.errlog = (double*)(tmp + log_off);
    int rc = TVL1_OK;
    stage_begin(st);
    for (int i = 0; i < n && !rc; i++) rc = launch_gamma_iteration(a, st);
    stage_end(st);
    if (!rc && errors && n > 0 &&
        (e = cudaMemcpyAsync(errors, tmp + log_off, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st)) != cudaSuccess)
        rc = fail(TVL1_ERR_CUDA, "error log copy failed: %s", cudaGetErrorString(e));
    e = cudaStreamSynchronize(st);
    if (!rc && e != cudaSuccess) rc = fail(TVL1_ERR_CUDA, "iterate (gamma): %s", cudaGetErrorString(e));
    cudaFree(tmp);
    return rc;
}

int tvl1_k_median5(const float* d_src, int w, int h, int pitch, float* d_dst, void* stream)
{
    if (!d_src || !d_dst || d_src == d_dst || w <= 0 || h <= 0 || pitch % 4 || pitch < w)
        return fail(TVL1_ERR_INVALID, "bad argument");
    MedianArgs a;
    a.u1[0] = const_cast<float*>(d_src); a.u1[1] = d_dst; a.u2[0] = a.u2[1] = nullptr;
    a.w = w; a.h = h; a.pitch = pitch; a.level = -1; a.slot = 0; a.ctrl = nullptr;
    memset(a.tm, 0, sizeof(a.tm));
    if (int r = make_plane_map(&a.tm[0][0], d_src, pitch, h, TVL1_MED_SW, TVL1_MED_SH)) return r;
    stage_begin((cudaStream_t)stream);
    const int rc = launch_median(a, 1, (cudaStream_t)stream);
    stage_end((cudaStream_t)stream);
    return rc;
}

int tvl1_k_median3(const float* d_src, int w, int h, int pitch, float* d_dst, void* stream)
{
    if (!d_src || !d_dst || d_src == d_dst || w <= 0 || h <= 0 || pitch % 4 || pitch < w)
        return fail(TVL1_ERR_INVALID, "bad argument");
    MedianArgs a;
    a.u1[0] = const_cast<float*>(d_src); a.u1[1] = d_dst; a.u2[0] = a.u2[1] = nullptr;
    a.w = w; a.h = h; a.pitch = pitch; a.level = -1; a.slot = 0; a.ctrl = nullptr;
    memset(a.tm, 0, sizeof(a.tm));
    stage_begin((cudaStream_t)stream);
    const int rc = launch_median3(a, 1, (cudaStream_t)stream);
    stage_end((cudaStream_t)stream);
    return rc;
}

int tvl1_selftest_arith(long long n, unsigned seed, int elo, int ehi, long long* mismatches, long long* unvouched)
{
    if (!mismatches || n <= 0 || elo > ehi || elo < -126 || ehi > 127) return fail(TVL1_ERR_INVALID, "bad argument");
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, 2 * sizeof(*d)));
    cudaMemset(d, 0, 2 * sizeof(*d));
    k_selftest_arith<<<148 * 8, 256>>>(seed, n, elo, ehi, d);
    unsigned long long hres[2] = {0, 0};
    cudaError_t e = cudaMemcpy(hres, d, sizeof(hres), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(TVL1_ERR_CUDA, "selftest: %s", cudaGetErrorString(e));
    *mismatches = (long long)hres[0];
    if (unvouched) *unvouched = (long long)hres[1];
    return TVL1_OK;
}

int tvl1_pyramid_sizes(int w, int h, int nscales, double scale_step, int* ws, int* hs)
{
    if (!ws || !hs || w <= 0 || h <= 0 || nscales <= 0) return fail(TVL1_ERR_INVALID, "bad argument");
    return pyramid_sizes(w, h, nscales, scale_step, ws, hs);
}

// ---- 8-bit prescale of the loader (reference src/optflow.cpp:111,124)

static int scaled_size_i(int n, double f) { return (int)lrint((double)n * f); }   // cvRound

int tvl1_prescaled_size(int w, int h, double scale, int* dw, int* dh)
{
    if (!dw || !dh || w <= 0 || h <= 0 || !(scale > 0.0)) return fail(TVL1_ERR_INVALID, "bad argument");
    *dw = scaled_size_i(w, scale);
    *dh = scaled_size_i(h, scale);
    if (*dw <= 0 || *dh <= 0) return fail(TVL1_ERR_INVALID, "scale %g leaves no pixels of %dx%d", scale, w, h);
    return TVL1_OK;
}

int tvl1_prescale_u8(const uint8_t* d_src, size_t spitch, int w, int h, double scale, uint8_t* d_dst, size_t dpitch,
                     void* stream)
{
    int dw = 0, dh = 0;
    int rc = tvl1_prescaled_size(w, h, scale, &dw, &dh);
    if (rc) return rc;
    if (!d_src || !d_dst || spitch < (size_t)w || dpitch < (size_t)dw) return fail(TVL1_ERR_INVALID, "bad buffer or pitch");
    cudaStream_t st = (cudaStream_t)stream;
    dim3 b(32, 8);
    const double inv = 1.0 / scale;
    if (inv == 2.0) k_prescale_half_u8<<<grid2d(dw, dh, b), b, 0, st>>>(d_src, spitch, w, h, d_dst, dpitch, dw, dh);
    else k_prescale_u8<<<grid2d(dw, dh, b), b, 0, st>>>(d_src, spitch, w, h, inv, d_dst, dpitch, dw, dh);
    CK(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_prescale_u8_host(int device, const uint8_t* src, size_t spitch, int w, int h, double scale, uint8_t* dst,
                          size_t dpitch)
{
    int dw = 0, dh = 0;
    int rc = tvl1_prescaled_size(w, h, scale, &dw, &dh);
    if (rc) return rc;
    if (!src || !dst || spitch < (size_t)w || dpitch < (size_t)dw) return fail(TVL1_ERR_INVALID, "bad buffer or pitch");
    if (device < 0 || device >= 64) return fail(TVL1_ERR_INVALID, "device out of range");
    CK(cudaSetDevice(device));
    // grow-only scratch per device (this entry point has no handle to keep it in): no cudaMalloc per call
    struct Scratch { uint8_t* p = nullptr; size_t cap = 0; };
    static Scratch scratch[64];
    static std::mutex mtx;
    std::lock_guard<std::mutex> lock(mtx);
    Scratch& S = scratch[device];
    const size_t raw = ((size_t)w * h + 255) / 256 * 256, need = raw + (size_t)dw * dh;
    if (S.cap < need) {
        if (S.p) cudaFree(S.p);
        S.p = nullptr; S.cap = 0;
        CK(cudaMalloc(&S.p, need));
        S.cap = need;
    }
    uint8_t *ds = S.p, *dd = S.p + raw;
    if (cudaMemcpy2D(ds, w, src, spitch, w, h, cudaMemcpyHostToDevice) != cudaSuccess) return fail(TVL1_ERR_CUDA, "upload failed");
    if ((rc = tvl1_prescale_u8(ds, w, w, h, scale, dd, dw, nullptr))) return rc;
    if (cudaMemcpy2D(dst, dpitch, dd, dw, dw, dh, cudaMemcpyDeviceToHost) != cudaSuccess)
        return fail(TVL1_ERR_CUDA, "download failed: %s", cudaGetErrorString(cudaGetLastError()));
    return TVL1_OK;
}

// ---- device-memory helpers

int tvl1_dev_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int tvl1_dev_alloc(int device, size_t bytes, void** out)
{
    if (!out) return fail(TVL1_ERR_INVALID, "out is null");
    CK(cudaSetDevice(device));
    CK(cudaMalloc(out, bytes ? bytes : 1));
    return TVL1_OK;
}

int tvl1_dev_free(int device, void* p)
{
    CK(cudaSetDevice(device));
    CK(cudaFree(p));
    return TVL1_OK;
}

int tvl1_dev_memset(void* d, int v, size_t bytes) { CK(cudaMemset(d, v, bytes)); return TVL1_OK; }
int tvl1_dev_h2d(void* d, const void* h, size_t bytes) { CK(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice)); return TVL1_OK; }
int tvl1_dev_d2h(void* h, const void* d, size_t bytes) { CK(cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost)); return TVL1_OK; }
int tvl1_dev_sync(int device) { CK(cudaSetDevice(device)); CK(cudaDeviceSynchronize()); return TVL1_OK; }
int tvl1_set_device(int device) { CK(cudaSetDevice(device)); return TVL1_OK; }
int tvl1_stream_create(int device, void** out)
{
    if (!out) return fail(TVL1_ERR_INVALID, "out is null");
    CK(cudaSetDevice(device));
    cudaStream_t s;
    CK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *out = (void*)s;
    return TVL1_OK;
}
int tvl1_stream_destroy(void* stream) { CK(cudaStreamDestroy((cudaStream_t)stream)); return TVL1_OK; }
int tvl1_stream_sync(void* stream) { CK(cudaStreamSynchronize((cudaStream_t)stream)); return TVL1_OK; }
// everything enqueued on `signaller` so far must finish before work enqueued on `waiter` after this call
int tvl1_stream_wait(void* waiter, void* signaller)
{
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    cudaError_t r = cudaEventRecord(e, (cudaStream_t)signaller);
    if (r == cudaSuccess) r = cudaStreamWaitEvent((cudaStream_t)waiter, e, 0);
    cudaEventDestroy(e);   // released once the recorded work has completed
    if (r != cudaSuccess) return fail(TVL1_ERR_CUDA, "stream wait: %s", cudaGetErrorString(r));
    return TVL1_OK;
}
int tvl1_stream_query(void* stream)
{
    const cudaError_t r = cudaStreamQuery((cudaStream_t)stream);
    if (r == cudaSuccess) return 1;
    if (r == cudaErrorNotReady) { cudaGetLastError(); return 0; }
    return fail(TVL1_ERR_CUDA, "stream query: %s", cudaGetErrorString(r));
}
int tvl1_dev_h2d_async(void* d, const void* h, size_t bytes, void* stream)
{
    CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return TVL1_OK;
}
int tvl1_dev_d2h_async(void* h, const void* d, size_t bytes, void* stream)
{
    CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return TVL1_OK;
}
int tvl1_host_alloc_pinned(size_t bytes, void** out)
{
    if (!out) return fail(TVL1_ERR_INVALID, "out is null");
    CK(cudaMallocHost(out, bytes ? bytes : 1));
    return TVL1_OK;
}
int tvl1_host_free_pinned(void* p) { CK(cudaFreeHost(p)); return TVL1_OK; }

}  // extern "C"
