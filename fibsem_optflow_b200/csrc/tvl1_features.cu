// tvl1_features.cu -- N4: the feature pre-alignment the reference runs in front of the flow stage.
//
// Replaces find_alignment (reference src/features.cpp:46-167) and the two cv::cuda::warpAffine call
// sites (src/optflow.cpp:374, 431-432): keypoints + binary descriptors on both frames, brute-force
// Hamming 2-NN, ratio test, RANSAC homography, sanity check, the top 2x3 of the homography as the
// affine that moves frame1 into frame0's coordinates.
//
// What the reference computes there is not reproducible bit for bit by anybody (cv::cuda::ORB's keypoint
// ties, RANSAC's random draws), so this is the same PIPELINE on sm_100a, not OpenCV's ORB:
//   * pyramid of `nlevels` by 1/scaleFactor (the loader's 8-bit bilinear resize, k_prescale_u8);
//   * FAST-9 corners (threshold `fastThreshold`), 3x3 non-maximum suppression on the FAST score, ranked
//     by Harris response (7x7 block, k = 0.04) and cut to ORB's per-level quota of `nfeatures`;
//   * orientation by the intensity centroid of the radius-15 disc, 256-bit steered BRIEF on the 7x7
//     Gaussian-smoothed level (sigma 2) -- the test pattern is this library's own (fixed seed), OpenCV's
//     learned table being part of its source;
//   * 2-NN by Hamming distance on the device; ratio test, sort and RANSAC (4-point DLT, reprojection
//     threshold `ransac`, adaptive iteration count, refit on the inliers + Gauss-Newton) on the host in
//     fp64 with a fixed-seed generator, so a job is reproducible run to run;
//   * warpAffine as cv::warpAffine computes it (inverse map in fp64, 1/32-px fixed-point source
//     coordinates, bilinear, constant 0 border): 8-bit frames with the 15-bit weight table, fp32 planes
//     (the map of src/optflow.cpp:431-432) with the float table.
// SURF (the reference's default `features` type, 2) is non-free and absent: both types take this path.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "tvl1_internal.h"

namespace tvl1 {

#define CKF(call)                                                                         \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(TVL1_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                              \
    } while (0)

static inline int cdivf(int a, int b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------ device kernels

__constant__ signed char c_brief[256 * 4];   // test i: (ax, ay) vs (bx, by), |coord| <= 13
__constant__ int c_disc_umax[16];            // half-width of row v of the radius-15 disc

// 7x7 Gaussian (sigma 2), separable, reflect-101 border, 8-bit in -> 8-bit out (rounded)
__global__ void __launch_bounds__(256) k_gauss7_u8(const uint8_t* __restrict__ src, size_t sp, int w, int h,
                                                   uint8_t* __restrict__ dst, size_t dp)
{
    // cv::getGaussianKernel(7, 2) rounded to fp32: centre, +-1, +-2, +-3 (they sum to 1)
    const float k[4] = {0.216105938f, 0.190712824f, 0.131074876f, 0.0701593235f};
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    auto refl = [](int p, int n) { p = p < 0 ? -p : p; return p >= n ? 2 * n - 2 - p : p; };
    float acc = 0.f;
#pragma unroll
    for (int dy = -3; dy <= 3; dy++) {
        const uint8_t* r = src + (size_t)min(max(refl(y + dy, h), 0), h - 1) * sp;
        float row = 0.f;
#pragma unroll
        for (int dx = -3; dx <= 3; dx++) row += k[dx < 0 ? -dx : dx] * (float)r[min(max(refl(x + dx, w), 0), w - 1)];
        acc += k[dy < 0 ? -dy : dy] * row;
    }
    dst[(size_t)y * dp + x] = (uint8_t)min(max(__float2int_rn(acc), 0), 255);
}

// FAST-9 score of every pixel at least `border` away from the frame: 0 = no corner, else the sum of
// |ring - centre| - t over the ring pixels on the corner's side (the original FAST ranking function)
__global__ void __launch_bounds__(256) k_fast_score(const uint8_t* __restrict__ img, size_t pitch, int w, int h, int border,
                                                    int t, float* __restrict__ score, int spitch)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    float out = 0.f;
    if (x >= border && y >= border && x < w - border && y < h - border) {
        const int ox[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
        const int oy[16] = {-3, -3, -2, -1, 0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3};
        const int c = img[(size_t)y * pitch + x];
        unsigned br = 0, dk = 0;
        int d[16];
#pragma unroll
        for (int k = 0; k < 16; k++) {
            d[k] = (int)img[(size_t)(y + oy[k]) * pitch + x + ox[k]] - c;
            br |= (d[k] > t ? 1u : 0u) << k;
            dk |= (d[k] < -t ? 1u : 0u) << k;
        }
        auto arc9 = [](unsigned m) {   // 9 contiguous set bits on the 16-ring
            m |= m << 16;
            unsigned r = m;
#pragma unroll
            for (int k = 1; k < 9; k++) r &= m >> k;
            return (r & 0xffffu) != 0;
        };
        const bool cb = arc9(br), cd = arc9(dk);
        if (cb || cd) {
            int sb = 0, sd = 0;
#pragma unroll
            for (int k = 0; k < 16; k++) {
                sb += d[k] > t ? d[k] - t : 0;
                sd += d[k] < -t ? -d[k] - t : 0;
            }
            out = (float)max(cb ? sb : 0, cd ? sd : 0);
        }
    }
    score[(size_t)y * spitch + x] = out;
}

struct Cand { float harris; unsigned short x, y; };

// 3x3 non-maximum suppression of the FAST score, Harris response (7x7 block, Sobel 3x3, k = 0.04) of the
// survivors, append to the candidate list (atomic counter; entries past the capacity are dropped but still
// counted, so that the caller can grow the list and run again) and to a 2048-bin histogram of the response's
// float bits (monotone for positive floats) for the top-N cut
__global__ void __launch_bounds__(256) k_nms_harris(const float* __restrict__ score, int spitch, const uint8_t* __restrict__ img,
                                                    size_t pitch, int w, int h, int border, Cand* __restrict__ cand,
                                                    int cap, int* __restrict__ count, int* __restrict__ hist)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < border || y < border || x >= w - border || y >= h - border) return;
    const float s = score[(size_t)y * spitch + x];
    if (s <= 0.f) return;
#pragma unroll
    for (int dy = -1; dy <= 1; dy++)
#pragma unroll
        for (int dx = -1; dx <= 1; dx++) {
            if (!dx && !dy) continue;
            const float o = score[(size_t)(y + dy) * spitch + x + dx];
            // ties: the earlier pixel in raster order wins
            if (o > s || (o == s && (dy < 0 || (dy == 0 && dx < 0)))) return;
        }
    float a = 0.f, b = 0.f, c = 0.f;
    for (int dy = -3; dy <= 3; dy++) {
        const uint8_t* r0 = img + (size_t)(y + dy - 1) * pitch + x;
        const uint8_t* r1 = r0 + pitch;
        const uint8_t* r2 = r1 + pitch;
        for (int dx = -3; dx <= 3; dx++) {
            const float ix = (float)((int)r0[dx + 1] - r0[dx - 1] + 2 * ((int)r1[dx + 1] - r1[dx - 1]) + (int)r2[dx + 1] - r2[dx - 1]);
            const float iy = (float)((int)r2[dx - 1] - r0[dx - 1] + 2 * ((int)r2[dx] - r0[dx]) + (int)r2[dx + 1] - r0[dx + 1]);
            a += ix * ix; b += iy * iy; c += ix * iy;
        }
    }
    const float sc = 1.f / (4.f * 7.f * 255.f);   // OpenCV's HarrisResponses scale: 1 / ((1 << 2) * blockSize * 255)
    const float sc4 = sc * sc * sc * sc;
    float hr = (a * b - c * c - 0.04f * (a + b) * (a + b)) * sc4;
    if (!(hr > 1e-30f)) hr = 1e-30f;               // keep every corner rankable (flat responses last)
    const int k = atomicAdd(count, 1);
    if (k < cap) { cand[k].harris = hr; cand[k].x = (unsigned short)x; cand[k].y = (unsigned short)y; }
    atomicAdd(hist + (__float_as_uint(hr) >> 20), 1);   // sign 0: 2048 bins over exponent + 3 mantissa bits
}

// candidates whose response bin is >= cut, compacted
__global__ void __launch_bounds__(256) k_select(const Cand* __restrict__ cand, int n, unsigned cut, Cand* __restrict__ out,
                                                int cap, int* __restrict__ count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Cand c = cand[i];
    if ((__float_as_uint(c.harris) >> 20) < cut) return;
    const int k = atomicAdd(count, 1);
    if (k < cap) out[k] = c;
}

struct KeyPt { float x, y, angle; int level; };   // x, y in level-0 pixels

// one warp per keypoint: intensity-centroid angle on the level image, then the 256 steered tests on the
// smoothed level; lane l produces byte l of the descriptor.  `pitch` is the level's, `bpitch` the smoothed copy's.
__global__ void __launch_bounds__(128) k_describe(const uint8_t* __restrict__ img, size_t pitch, const uint8_t* __restrict__ blur,
                                                  size_t bpitch, const Cand* __restrict__ kp, int n, float scale, int level,
                                                  KeyPt* __restrict__ out_kp, uint32_t* __restrict__ out_desc, int out_base)
{
    const int wi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wi >= n) return;
    const int cx = kp[wi].x, cy = kp[wi].y;
    const uint8_t* c = img + (size_t)cy * pitch + cx;
    int m01 = 0, m10 = 0;
    // rows v = -15 .. 15 of the disc, 31 rows over 32 lanes
    if (lane < 31) {
        const int v = lane - 15, um = c_disc_umax[v < 0 ? -v : v];
        const uint8_t* r = c + (ptrdiff_t)v * (ptrdiff_t)pitch;
        int sx = 0, sv = 0;
        for (int u = -um; u <= um; u++) { const int p = r[u]; sx += u * p; sv += p; }
        m10 = sx; m01 = v * sv;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { m01 += __shfl_xor_sync(0xffffffffu, m01, o); m10 += __shfl_xor_sync(0xffffffffu, m10, o); }
    const float ang = atan2f((float)m01, (float)m10);
    float sn, cs;
    sincosf(ang, &sn, &cs);
    const uint8_t* b = blur + (size_t)cy * bpitch + cx;
    unsigned byte = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const signed char* t = c_brief + (lane * 8 + k) * 4;
        const int ax = __float2int_rn(t[0] * cs - t[1] * sn), ay = __float2int_rn(t[0] * sn + t[1] * cs);
        const int bx = __float2int_rn(t[2] * cs - t[3] * sn), by = __float2int_rn(t[2] * sn + t[3] * cs);
        const int va = b[(ptrdiff_t)ay * (ptrdiff_t)bpitch + ax], vb = b[(ptrdiff_t)by * (ptrdiff_t)bpitch + bx];
        byte |= (va < vb ? 1u : 0u) << k;
    }
    // four lanes -> one 32-bit word
    unsigned word = byte << (8 * (lane & 3));
    word |= __shfl_xor_sync(0xffffffffu, word, 1);
    word |= __shfl_xor_sync(0xffffffffu, word, 2);
    if ((lane & 3) == 0) out_desc[(size_t)(out_base + wi) * 8 + (lane >> 2)] = word;
    if (lane == 0) {
        KeyPt o;
        o.x = (float)cx * scale; o.y = (float)cy * scale; o.angle = ang; o.level = level;
        out_kp[out_base + wi] = o;
    }
}

// brute-force Hamming 2-NN: one thread per query descriptor, train descriptors through shared memory
__global__ void __launch_bounds__(128) k_knn2(const uint32_t* __restrict__ q, int nq, const uint32_t* __restrict__ t, int nt,
                                              int* __restrict__ idx1, int* __restrict__ d1, int* __restrict__ d2)
{
    __shared__ uint32_t tile[128 * 8];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t d[8];
#pragma unroll
    for (int k = 0; k < 8; k++) d[k] = i < nq ? q[(size_t)i * 8 + k] : 0u;
    int b1 = 1 << 30, b2 = 1 << 30, bi = -1;
    for (int base = 0; base < nt; base += 128) {
        const int m = min(128, nt - base);
        __syncthreads();
        for (int k = threadIdx.x; k < m * 8; k += 128) tile[k] = t[(size_t)base * 8 + k];
        __syncthreads();
        for (int j = 0; j < m; j++) {
            int dist = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) dist += __popc(d[k] ^ tile[j * 8 + k]);
            if (dist < b1) { b2 = b1; b1 = dist; bi = base + j; }
            else if (dist < b2) b2 = dist;
        }
    }
    if (i < nq) { idx1[i] = bi; d1[i] = b1; d2[i] = b2; }
}

// ---- warpAffine as cv::warpAffine computes it (imgproc, INTER_LINEAR, BORDER_CONSTANT 0).  M = the inverse
// map (destination -> source) in fp64; source coordinates in 1/1024 px, rounded to 1/32 px.
struct AffineFix { double m[6]; };

__device__ __forceinline__ int sat_int(double v) { return __double2int_rn(fmin(fmax(v, -2147483648.0), 2147483647.0)); }

__device__ __forceinline__ void affine_src(const AffineFix& A, int x, int y, int& sx, int& sy, int& fx, int& fy)
{
    const int X0 = sat_int((A.m[1] * y + A.m[2]) * 1024.0) + 16, Y0 = sat_int((A.m[4] * y + A.m[5]) * 1024.0) + 16;
    const int X = (X0 + sat_int(A.m[0] * x * 1024.0)) >> 5, Y = (Y0 + sat_int(A.m[3] * x * 1024.0)) >> 5;
    sx = min(max(X >> 5, -32768), 32767); sy = min(max(Y >> 5, -32768), 32767);
    fx = X & 31; fy = Y & 31;
}

__global__ void __launch_bounds__(256) k_warp_affine_u8(const uint8_t* __restrict__ src, size_t sp, int sw, int sh,
                                                        uint8_t* __restrict__ dst, size_t dp, int dw, int dh, AffineFix A)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int sx, sy, fx, fy;
    affine_src(A, x, y, sx, sy, fx, fy);
    // 15-bit weights of the 32 x 32 bilinear table: rounded products, the rounding residue folded into the
    // largest (resp. smallest) of the four so that they add up to exactly 1 << 15
    const float ax = fx * (1.f / 32), ay = fy * (1.f / 32);
    const float wf[4] = {(1.f - ay) * (1.f - ax), (1.f - ay) * ax, ay * (1.f - ax), ay * ax};
    int wi[4], sum = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) { wi[k] = min(max(__float2int_rn(wf[k] * 32768.f), -32768), 32767); sum += wi[k]; }
    if (sum != 32768) {
        const int diff = sum - 32768;
        int kmax = 0, kmin = 0;
#pragma unroll
        for (int k = 1; k < 4; k++) { if (wi[k] > wi[kmax]) kmax = k; if (wi[k] < wi[kmin]) kmin = k; }
        if (diff < 0) wi[kmax] -= diff; else wi[kmin] -= diff;
    }
    auto px = [&](int xx, int yy) { return ((unsigned)xx < (unsigned)sw && (unsigned)yy < (unsigned)sh) ? (int)src[(size_t)yy * sp + xx] : 0; };
    const int v = px(sx, sy) * wi[0] + px(sx + 1, sy) * wi[1] + px(sx, sy + 1) * wi[2] + px(sx + 1, sy + 1) * wi[3];
    dst[(size_t)y * dp + x] = (uint8_t)min(max((v + (1 << 14)) >> 15, 0), 255);
}

__global__ void __launch_bounds__(256) k_warp_affine_f32(const float* __restrict__ src, size_t sp, int sw, int sh,
                                                         float* __restrict__ dst, size_t dp, int dw, int dh, AffineFix A)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= dw || y >= dh) return;
    int sx, sy, fx, fy;
    affine_src(A, x, y, sx, sy, fx, fy);
    const float ax = fx * (1.f / 32), ay = fy * (1.f / 32);
    const float w0 = (1.f - ay) * (1.f - ax), w1 = (1.f - ay) * ax, w2 = ay * (1.f - ax), w3 = ay * ax;
    auto px = [&](int xx, int yy) { return ((unsigned)xx < (unsigned)sw && (unsigned)yy < (unsigned)sh) ? src[(size_t)yy * sp + xx] : 0.f; };
    dst[(size_t)y * dp + x] = px(sx, sy) * w0 + px(sx + 1, sy) * w1 + px(sx, sy + 1) * w2 + px(sx + 1, sy + 1) * w3;
}

// ------------------------------------------------------------------ host: homography

struct Pt { double x, y; };

// solves the n x n system a x = b in place (partial pivoting); false if singular
static bool solve_linear(std::vector<double>& a, std::vector<double>& b, int n)
{
    for (int c = 0; c < n; c++) {
        int p = c;
        for (int r = c + 1; r < n; r++) if (std::fabs(a[(size_t)r * n + c]) > std::fabs(a[(size_t)p * n + c])) p = r;
        if (std::fabs(a[(size_t)p * n + c]) < 1e-12) return false;
        if (p != c) { for (int k = 0; k < n; k++) std::swap(a[(size_t)p * n + k], a[(size_t)c * n + k]); std::swap(b[p], b[c]); }
        for (int r = c + 1; r < n; r++) {
            const double f = a[(size_t)r * n + c] / a[(size_t)c * n + c];
            if (f == 0.0) continue;
            for (int k = c; k < n; k++) a[(size_t)r * n + k] -= f * a[(size_t)c * n + k];
            b[r] -= f * b[c];
        }
    }
    for (int r = n - 1; r >= 0; r--) {
        double s = b[r];
        for (int k = r + 1; k < n; k++) s -= a[(size_t)r * n + k] * b[k];
        b[r] = s / a[(size_t)r * n + r];
    }
    return true;
}

// least-squares homography (h22 = 1) of the listed correspondences, Hartley-normalised
static bool fit_homography(const std::vector<Pt>& p, const std::vector<Pt>& q, const std::vector<int>& idx, double* H)
{
    const int n = (int)idx.size();
    if (n < 4) return false;
    auto norm = [&](const std::vector<Pt>& v, double& cx, double& cy, double& s) {
        cx = cy = 0;
        for (int i : idx) { cx += v[i].x; cy += v[i].y; }
        cx /= n; cy /= n;
        double d = 0;
        for (int i : idx) d += std::hypot(v[i].x - cx, v[i].y - cy);
        s = d > 1e-12 ? std::sqrt(2.0) * n / d : 1.0;
    };
    double pcx, pcy, ps, qcx, qcy, qs;
    norm(p, pcx, pcy, ps);
    norm(q, qcx, qcy, qs);
    std::vector<double> ata(64, 0.0), atb(8, 0.0);
    for (int i : idx) {
        const double x = (p[i].x - pcx) * ps, y = (p[i].y - pcy) * ps, u = (q[i].x - qcx) * qs, v = (q[i].y - qcy) * qs;
        const double r1[8] = {x, y, 1, 0, 0, 0, -u * x, -u * y}, r2[8] = {0, 0, 0, x, y, 1, -v * x, -v * y};
        for (int a = 0; a < 8; a++) {
            for (int b = 0; b < 8; b++) ata[a * 8 + b] += r1[a] * r1[b] + r2[a] * r2[b];
            atb[a] += r1[a] * u + r2[a] * v;
        }
    }
    if (!solve_linear(ata, atb, 8)) return false;
    // H = Tq^-1 * Hn * Tp
    const double hn[9] = {atb[0], atb[1], atb[2], atb[3], atb[4], atb[5], atb[6], atb[7], 1.0};
    const double tp[9] = {ps, 0, -ps * pcx, 0, ps, -ps * pcy, 0, 0, 1};
    const double tqi[9] = {1 / qs, 0, qcx, 0, 1 / qs, qcy, 0, 0, 1};
    double t[9], r[9];
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) { t[a * 3 + b] = 0; for (int k = 0; k < 3; k++) t[a * 3 + b] += hn[a * 3 + k] * tp[k * 3 + b]; }
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) { r[a * 3 + b] = 0; for (int k = 0; k < 3; k++) r[a * 3 + b] += tqi[a * 3 + k] * t[k * 3 + b]; }
    if (std::fabs(r[8]) < 1e-12) return false;
    for (int k = 0; k < 9; k++) H[k] = r[k] / r[8];
    return true;
}

static inline double reproj2(const double* H, const Pt& a, const Pt& b)
{
    const double w = H[6] * a.x + H[7] * a.y + H[8];
    if (std::fabs(w) < 1e-12) return 1e300;
    const double dx = (H[0] * a.x + H[1] * a.y + H[2]) / w - b.x, dy = (H[3] * a.x + H[4] * a.y + H[5]) / w - b.y;
    return dx * dx + dy * dy;
}

// a few Gauss-Newton steps on the reprojection error of the inliers (8 parameters, h22 = 1)
static void refine_homography(const std::vector<Pt>& p, const std::vector<Pt>& q, const std::vector<int>& in, double* H)
{
    for (int it = 0; it < 10; it++) {
        std::vector<double> jtj(64, 0.0), jtr(8, 0.0);
        for (int i : in) {
            const double x = p[i].x, y = p[i].y, w = H[6] * x + H[7] * y + 1.0;
            if (std::fabs(w) < 1e-12) continue;
            const double u = (H[0] * x + H[1] * y + H[2]) / w, v = (H[3] * x + H[4] * y + H[5]) / w;
            const double ju[8] = {x / w, y / w, 1 / w, 0, 0, 0, -u * x / w, -u * y / w};
            const double jv[8] = {0, 0, 0, x / w, y / w, 1 / w, -v * x / w, -v * y / w};
            const double ru = q[i].x - u, rv = q[i].y - v;
            for (int a = 0; a < 8; a++) {
                for (int b = 0; b < 8; b++) jtj[a * 8 + b] += ju[a] * ju[b] + jv[a] * jv[b];
                jtr[a] += ju[a] * ru + jv[a] * rv;
            }
        }
        if (!solve_linear(jtj, jtr, 8)) return;
        double step = 0;
        for (int k = 0; k < 8; k++) { H[k] += jtr[k]; step += jtr[k] * jtr[k]; }
        if (step < 1e-24) return;
    }
}

// cv::findHomography(points_0, points_1, method, threshold): RANSAC (method 8; 4 and 16 are served by it too)
// or plain least squares (0).  false: no model.
static bool find_homography(const std::vector<Pt>& p, const std::vector<Pt>& q, int method, double thr, double* H)
{
    const int n = (int)p.size();
    std::vector<int> all(n);
    for (int i = 0; i < n; i++) all[i] = i;
    if (method == 0) return fit_homography(p, q, all, H);
    const double thr2 = thr * thr;
    uint64_t rng = 0x9E3779B97F4A7C15ull;   // fixed seed: a job is reproducible
    auto next = [&]() { rng ^= rng << 13; rng ^= rng >> 7; rng ^= rng << 17; return rng; };
    int best = 0, niters = 2000;
    double bestH[9];
    for (int it = 0; it < niters; it++) {
        int s[4];
        for (int k = 0; k < 4;) {
            s[k] = (int)(next() % (uint64_t)n);
            bool dup = false;
            for (int j = 0; j < k; j++) dup = dup || s[j] == s[k];
            if (!dup) k++;
        }
        // degenerate samples: three (nearly) collinear points on either side
        bool bad = false;
        for (int a = 0; a < 4 && !bad; a++)
            for (int b = a + 1; b < 4 && !bad; b++)
                for (int c = b + 1; c < 4 && !bad; c++) {
                    const double ap = (p[s[b]].x - p[s[a]].x) * (p[s[c]].y - p[s[a]].y) - (p[s[b]].y - p[s[a]].y) * (p[s[c]].x - p[s[a]].x);
                    const double aq = (q[s[b]].x - q[s[a]].x) * (q[s[c]].y - q[s[a]].y) - (q[s[b]].y - q[s[a]].y) * (q[s[c]].x - q[s[a]].x);
                    bad = std::fabs(ap) < 1e-3 || std::fabs(aq) < 1e-3;
                }
        if (bad) continue;
        double Hc[9];
        if (!fit_homography(p, q, std::vector<int>(s, s + 4), Hc)) continue;
        int cnt = 0;
        for (int i = 0; i < n; i++) cnt += reproj2(Hc, p[i], q[i]) <= thr2;
        if (cnt > best) {
            best = cnt;
            std::memcpy(bestH, Hc, sizeof(bestH));
            // adaptive count for 99.5 % confidence, as cv::RANSACUpdateNumIters
            const double wi = (double)cnt / n, denom = std::log(std::max(1.0 - wi * wi * wi * wi, 1e-300));
            const double need = denom < 0 ? std::log(1.0 - 0.995) / denom : 0.0;
            if (need < niters) niters = std::max((int)std::ceil(need), it + 1);
        }
    }
    if (best < 4) return false;
    std::vector<int> in;
    for (int i = 0; i < n; i++) if (reproj2(bestH, p[i], q[i]) <= thr2) in.push_back(i);
    if (!fit_homography(p, q, in, H)) std::memcpy(H, bestH, sizeof(bestH));
    refine_homography(p, q, in, H);
    return true;
}

// ------------------------------------------------------------------ host: per-frame feature extraction

struct FeatScratch {
    int device = -1;
    uint8_t *lvl = nullptr, *blur = nullptr;      // one pyramid level and its smoothed copy
    float* score = nullptr;
    size_t img_cap = 0;
    Cand *cand = nullptr, *sel = nullptr;
    int cand_cap = 0, sel_cap = 0;
    int* counters = nullptr;                      // [0] candidates, [1] selected, [2 ..] histogram (2048)
    KeyPt* kp[2] = {nullptr, nullptr};
    uint32_t* desc[2] = {nullptr, nullptr};
    int kp_cap = 0;
    int *idx1 = nullptr, *d1 = nullptr, *d2 = nullptr;
};

void features_release(void* p)
{
    FeatScratch* S = (FeatScratch*)p;
    if (!S) return;
    cudaFree(S->lvl); cudaFree(S->blur); cudaFree(S->score); cudaFree(S->cand); cudaFree(S->sel); cudaFree(S->counters);
    for (int k = 0; k < 2; k++) { cudaFree(S->kp[k]); cudaFree(S->desc[k]); }
    cudaFree(S->idx1); cudaFree(S->d1); cudaFree(S->d2);
    delete S;
}

// the current device's BRIEF pattern and disc table
static int upload_tables(int device)
{
    static bool done[64] = {false};          // __constant__ tables live per device, not per handle
    if (done[device & 63]) return TVL1_OK;
    // 256 test pairs: isotropic Gaussian (sigma = patch / 5) clipped to +-13, fixed seed
    signed char pat[256 * 4];
    uint64_t r = 0x2545F4914F6CDD1Dull;
    auto uni = [&]() { r ^= r << 13; r ^= r >> 7; r ^= r << 17; return (double)((r >> 11) + 1) / 9007199254740993.0; };
    for (int k = 0; k < 256 * 4; k += 2) {
        double gx, gy;
        do {
            const double u1 = uni(), u2 = uni(), m = std::sqrt(-2.0 * std::log(u1)) * 6.2;
            gx = m * std::cos(6.283185307179586 * u2);
            gy = m * std::sin(6.283185307179586 * u2);
        } while (std::fabs(gx) > 13.0 || std::fabs(gy) > 13.0);
        pat[k] = (signed char)std::lrint(gx);
        pat[k + 1] = (signed char)std::lrint(gy);
    }
    CKF(cudaMemcpyToSymbol(c_brief, pat, sizeof(pat)));
    int umax[16];
    for (int v = 0; v <= 15; v++) umax[v] = (int)std::floor(std::sqrt(15.0 * 15.0 - (double)v * v) + 1e-9);
    CKF(cudaMemcpyToSymbol(c_disc_umax, umax, sizeof(umax)));
    done[device & 63] = true;
    return TVL1_OK;
}

template <class T>
static int grow(T** p, size_t have, size_t want)
{
    if (have >= want) return TVL1_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    CKF(cudaMalloc(p, want * sizeof(T)));
    return TVL1_OK;
}

// keypoints + descriptors of one frame into slot `which`; returns their number
static int extract(FeatScratch& S, const uint8_t* d_img, size_t pitch, int w, int h, const tvl1_feature_params& P, int which,
                   cudaStream_t st, int* n_out)
{
    int rc;
    const int border = std::max(P.edge_threshold, 19);   // ring 3 + disc 15 resp. rotated test offsets <= 18.4
    const size_t px = (size_t)w * h;
    if (S.img_cap < px) {
        cudaFree(S.lvl); cudaFree(S.blur); cudaFree(S.score);
        S.lvl = S.blur = nullptr; S.score = nullptr; S.img_cap = 0;
        CKF(cudaMalloc(&S.lvl, px)); CKF(cudaMalloc(&S.blur, px)); CKF(cudaMalloc(&S.score, px * sizeof(float)));
        S.img_cap = px;
    }
    // the candidate list starts at 4M entries and grows when a level has more NMS survivors; the selection
    // is sized per level from the histogram
    const int cand_cap = 1 << 22, kp_cap = P.nfeatures + 64;
    if ((rc = grow(&S.cand, (size_t)S.cand_cap, (size_t)cand_cap))) return rc;
    S.cand_cap = std::max(S.cand_cap, cand_cap);
    if (!S.counters) CKF(cudaMalloc(&S.counters, sizeof(int) * (2 + 2048)));
    if (S.kp_cap < kp_cap) {
        for (int k = 0; k < 2; k++) { cudaFree(S.kp[k]); cudaFree(S.desc[k]); S.kp[k] = nullptr; S.desc[k] = nullptr; }
        cudaFree(S.idx1); cudaFree(S.d1); cudaFree(S.d2);
        S.idx1 = S.d1 = S.d2 = nullptr;
        for (int k = 0; k < 2; k++) { CKF(cudaMalloc(&S.kp[k], sizeof(KeyPt) * kp_cap)); CKF(cudaMalloc(&S.desc[k], 32 * (size_t)kp_cap)); }
        CKF(cudaMalloc(&S.idx1, sizeof(int) * kp_cap)); CKF(cudaMalloc(&S.d1, sizeof(int) * kp_cap)); CKF(cudaMalloc(&S.d2, sizeof(int) * kp_cap));
        S.kp_cap = kp_cap;
    }
    // ORB's quota per level: nfeatures * (1 - f) / (1 - f^nlevels) * f^level, f = 1 / scaleFactor; the last gets the rest
    const double f = 1.0 / P.scale_factor;
    std::vector<int> quota(P.nlevels);
    {
        double per = P.nfeatures * (1.0 - f) / (1.0 - std::pow(f, P.nlevels));
        int sum = 0;
        for (int l = 0; l + 1 < P.nlevels; l++) { quota[l] = (int)std::lrint(per); sum += quota[l]; per *= f; }
        quota[P.nlevels - 1] = std::max(P.nfeatures - sum, 0);
    }
    int total = 0;
    std::vector<int> h_cnt(2 + 2048);
    std::vector<Cand> h_sel;
    dim3 b(32, 8);
    for (int l = 0; l < P.nlevels && total < P.nfeatures; l++) {
        const double sc = std::pow(P.scale_factor, l);
        int lw = w, lh = h;
        const uint8_t* img = d_img;
        size_t lp = pitch;
        if (l > 0) {
            if ((rc = tvl1_prescaled_size(w, h, 1.0 / sc, &lw, &lh))) return rc;
            if ((rc = tvl1_prescale_u8(d_img, pitch, w, h, 1.0 / sc, S.lvl, (size_t)lw, st))) return rc;
            img = S.lvl; lp = (size_t)lw;
        }
        if (lw <= 2 * border + 8 || lh <= 2 * border + 8) break;
        dim3 g(cdivf(lw, 32), cdivf(lh, 8));
        CKF(cudaMemsetAsync(S.counters, 0, sizeof(int) * (2 + 2048), st));
        k_fast_score<<<g, b, 0, st>>>(img, lp, lw, lh, border, P.fast_threshold, S.score, lw);
        k_nms_harris<<<g, b, 0, st>>>(S.score, lw, img, lp, lw, lh, border, S.cand, S.cand_cap, S.counters, S.counters + 2);
        k_gauss7_u8<<<g, b, 0, st>>>(img, lp, lw, lh, S.blur, (size_t)lw);
        CKF(cudaGetLastError());
        CKF(cudaMemcpyAsync(h_cnt.data(), S.counters, sizeof(int) * (2 + 2048), cudaMemcpyDeviceToHost, st));
        CKF(cudaStreamSynchronize(st));
        if (h_cnt[0] > S.cand_cap) {
            // more survivors than the list holds (the atomics decided which were dropped): grow it, list them again
            if ((rc = grow(&S.cand, (size_t)S.cand_cap, (size_t)h_cnt[0]))) return rc;
            S.cand_cap = h_cnt[0];
            CKF(cudaMemsetAsync(S.counters, 0, sizeof(int) * (2 + 2048), st));
            k_nms_harris<<<g, b, 0, st>>>(S.score, lw, img, lp, lw, lh, border, S.cand, S.cand_cap, S.counters, S.counters + 2);
            CKF(cudaGetLastError());
            CKF(cudaMemcpyAsync(h_cnt.data(), S.counters, sizeof(int) * (2 + 2048), cudaMemcpyDeviceToHost, st));
            CKF(cudaStreamSynchronize(st));
        }
        const int ncand = h_cnt[0], want = std::min(quota[l], P.nfeatures - total);
        if (ncand == 0 || want == 0) continue;
        // highest histogram bin such that the bins from it upwards hold at least `want` candidates; those bins
        // hold exactly `nsel`, and the selection has room for all of them
        unsigned cut = 0;
        int nsel = ncand;
        for (int bin = 2047, acc = 0; bin >= 0; bin--) {
            acc += h_cnt[2 + bin];
            if (acc >= want) { cut = (unsigned)bin; nsel = acc; break; }
        }
        if ((rc = grow(&S.sel, (size_t)S.sel_cap, (size_t)nsel))) return rc;
        S.sel_cap = std::max(S.sel_cap, nsel);
        k_select<<<cdivf(ncand, 256), 256, 0, st>>>(S.cand, ncand, cut, S.sel, S.sel_cap, S.counters + 1);
        CKF(cudaGetLastError());
        h_sel.resize((size_t)nsel);
        CKF(cudaMemcpyAsync(h_sel.data(), S.sel, sizeof(Cand) * (size_t)nsel, cudaMemcpyDeviceToHost, st));
        CKF(cudaStreamSynchronize(st));
        // strongest first; position breaks ties, so that neither the set kept nor its order depends on the atomics
        std::sort(h_sel.begin(), h_sel.end(), [](const Cand& a, const Cand& c) {
            if (a.harris != c.harris) return a.harris > c.harris;
            if (a.y != c.y) return a.y < c.y;
            return a.x < c.x;
        });
        const int keep = std::min(nsel, want);
        CKF(cudaMemcpyAsync(S.sel, h_sel.data(), sizeof(Cand) * (size_t)keep, cudaMemcpyHostToDevice, st));
        k_describe<<<cdivf(keep * 32, 128), 128, 0, st>>>(img, lp, S.blur, (size_t)lw, S.sel, keep, (float)sc, l, S.kp[which],
                                                          S.desc[which], total);
        CKF(cudaGetLastError());
        CKF(cudaStreamSynchronize(st));   // h_sel is re-used by the next level
        total += keep;
    }
    *n_out = total;
    return TVL1_OK;
}

static int check_feature_params(const tvl1_feature_params& P)
{
    if (P.nfeatures < 16 || P.nfeatures > (1 << 20) || P.nlevels < 1 || P.nlevels > 16 || !(P.scale_factor > 1.f) ||
        P.fast_threshold < 1 || P.fast_threshold > 254 || !(P.ratio > 0.f) || !(P.ransac > 0.0))
        return fail(TVL1_ERR_INVALID, "feature parameters out of range");
    if (P.first_level != 0) return fail(TVL1_ERR_UNSUPPORTED, "firstLevel != 0 is not supported");
    return TVL1_OK;
}

// the handle's feature scratch on its device, with the device's tables uploaded
static int feature_scratch(tvl1_handle* H, FeatScratch** out)
{
    const int dev = handle_device(H);
    CKF(cudaSetDevice(dev));
    void** slot = handle_feature_slot(H);
    if (!*slot) *slot = new FeatScratch();
    FeatScratch* S = (FeatScratch*)*slot;
    S->device = dev;
    *out = S;
    return upload_tables(dev);
}

}  // namespace tvl1

using namespace tvl1;

extern "C" {

void tvl1_default_feature_params(tvl1_feature_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    // orb_defaults (src/features.cpp:19-32), ratio / ransac / homo (src/features.cpp:107, 133)
    p->nfeatures = 5000; p->scale_factor = 1.2f; p->nlevels = 8; p->edge_threshold = 31; p->first_level = 0;
    p->patch_size = 31; p->fast_threshold = 20; p->ratio = 0.8f; p->ransac = 5.0; p->homo = 8;
}

int tvl1_find_alignment(tvl1_handle* H, const uint8_t* d_moving, size_t pitch_m, int wm, int hm, const uint8_t* d_fixed,
                        size_t pitch_f, int wf, int hf, const tvl1_feature_params* prm, float* affine, int* n_matches,
                        int* n_good, void* stream)
{
    if (!H || !d_moving || !d_fixed || !prm || !affine) return fail(TVL1_ERR_INVALID, "null argument");
    if (wm <= 0 || hm <= 0 || wf <= 0 || hf <= 0 || pitch_m < (size_t)wm || pitch_f < (size_t)wf) return fail(TVL1_ERR_INVALID, "bad geometry");
    if (wm > 65535 || hm > 65535 || wf > 65535 || hf > 65535) return fail(TVL1_ERR_INVALID, "frame side > 65535");
    tvl1_feature_params P = *prm;
    int rc = check_feature_params(P);
    if (rc) return rc;
    FeatScratch* Sp = nullptr;
    if ((rc = feature_scratch(H, &Sp))) return rc;
    FeatScratch& S = *Sp;
    cudaStream_t st = (cudaStream_t)stream;
    // identity unless a trustworthy transform is found (src/features.cpp:141-164)
    const float ident[6] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f};
    memcpy(affine, ident, sizeof(ident));
    if (n_matches) *n_matches = 0;
    if (n_good) *n_good = 0;
    int n0 = 0, n1 = 0;   // 0: the moving frame (the reference's descriptors_0 = query), 1: the fixed one (train)
    if ((rc = extract(S, d_moving, pitch_m, wm, hm, P, 0, st, &n0))) return rc;
    if ((rc = extract(S, d_fixed, pitch_f, wf, hf, P, 1, st, &n1))) return rc;
    if (n0 == 0 || n1 < 2) {
        if (P.debug) printf("Number of features: %d\nNumber of good features: 0\n", n0);
        printf("Not enough matches. Using no transformation\n");
        return TVL1_OK;
    }
    k_knn2<<<cdivf(n0, 128), 128, 0, st>>>(S.desc[0], n0, S.desc[1], n1, S.idx1, S.d1, S.d2);
    CKF(cudaGetLastError());
    std::vector<int> idx((size_t)n0), d1((size_t)n0), d2((size_t)n0);
    std::vector<KeyPt> k0((size_t)n0), k1((size_t)n1);
    CKF(cudaMemcpyAsync(idx.data(), S.idx1, sizeof(int) * (size_t)n0, cudaMemcpyDeviceToHost, st));
    CKF(cudaMemcpyAsync(d1.data(), S.d1, sizeof(int) * (size_t)n0, cudaMemcpyDeviceToHost, st));
    CKF(cudaMemcpyAsync(d2.data(), S.d2, sizeof(int) * (size_t)n0, cudaMemcpyDeviceToHost, st));
    CKF(cudaMemcpyAsync(k0.data(), S.kp[0], sizeof(KeyPt) * (size_t)n0, cudaMemcpyDeviceToHost, st));
    CKF(cudaMemcpyAsync(k1.data(), S.kp[1], sizeof(KeyPt) * (size_t)n1, cudaMemcpyDeviceToHost, st));
    CKF(cudaStreamSynchronize(st));
    // ratio test over the first min(n_train - 1, n_query) queries (the reference's loop bound, src/features.cpp:105),
    // then std::sort(good) = ascending distance
    struct Good { int dist, q, t; };
    std::vector<Good> good;
    for (int i = 0; i < std::min(n1 - 1, n0); i++)
        if ((float)d1[(size_t)i] < P.ratio * (float)d2[(size_t)i]) good.push_back(Good{d1[(size_t)i], i, idx[(size_t)i]});
    std::stable_sort(good.begin(), good.end(), [](const Good& a, const Good& b) { return a.dist < b.dist; });
    if (n_matches) *n_matches = n0;
    if (n_good) *n_good = (int)good.size();
    if (P.debug) printf("Number of features: %d\nNumber of good features: %zu\n", n0, good.size());
    if (good.size() <= 10) {
        printf("Not enough matches. Using no transformation\n");
        return TVL1_OK;
    }
    std::vector<Pt> p(good.size()), q(good.size());
    for (size_t i = 0; i < good.size(); i++) {
        p[i] = Pt{k0[(size_t)good[i].q].x, k0[(size_t)good[i].q].y};
        q[i] = Pt{k1[(size_t)good[i].t].x, k1[(size_t)good[i].t].y};
    }
    double Hm[9];
    const bool found = find_homography(p, q, P.homo, P.ransac, Hm);
    if (!found || std::fabs(1 - Hm[0]) > 0.20 || std::fabs(1 - Hm[4]) > 0.20) {
        printf("More than twenty percent variance in zoom or no homography found, this is probably an error, ignoring the transformation.\n");
        return TVL1_OK;
    }
    if (P.debug) printf("%g %g %g\n%g %g %g\n%g %g %g\n", Hm[0], Hm[1], Hm[2], Hm[3], Hm[4], Hm[5], Hm[6], Hm[7], Hm[8]);
    for (int k = 0; k < 6; k++) affine[k] = (float)Hm[k];   // homo(Range(0,2), Range(0,3)).copyTo(affine)
    return TVL1_OK;
}

static int invert_affine(const float* a, AffineFix* out)
{
    // cv::warpAffine without WARP_INVERSE_MAP: M is inverted in fp64 first
    double M[6];
    for (int k = 0; k < 6; k++) M[k] = (double)a[k];
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    const double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11; M[1] *= -D; M[3] *= -D; M[4] = A22;
    const double b1 = -M[0] * M[2] - M[1] * M[5], b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1; M[5] = b2;
    for (int k = 0; k < 6; k++) out->m[k] = M[k];
    return TVL1_OK;
}

int tvl1_warp_affine_u8(const uint8_t* d_src, size_t spitch, int sw, int sh, const float* affine, uint8_t* d_dst, size_t dpitch,
                        int dw, int dh, void* stream)
{
    if (!d_src || !d_dst || !affine || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || spitch < (size_t)sw || dpitch < (size_t)dw)
        return fail(TVL1_ERR_INVALID, "bad argument");
    AffineFix A;
    invert_affine(affine, &A);
    dim3 b(32, 8), g(cdivf(dw, 32), cdivf(dh, 8));
    k_warp_affine_u8<<<g, b, 0, (cudaStream_t)stream>>>(d_src, spitch, sw, sh, d_dst, dpitch, dw, dh, A);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_warp_affine_f32(const float* d_src, size_t spitch, int sw, int sh, const float* affine, float* d_dst, size_t dpitch,
                         int dw, int dh, void* stream)
{
    if (!d_src || !d_dst || !affine || sw <= 0 || sh <= 0 || dw <= 0 || dh <= 0 || spitch % 4 || dpitch % 4 ||
        spitch < (size_t)sw * 4 || dpitch < (size_t)dw * 4)
        return fail(TVL1_ERR_INVALID, "bad argument");
    AffineFix A;
    invert_affine(affine, &A);
    dim3 b(32, 8), g(cdivf(dw, 32), cdivf(dh, 8));
    k_warp_affine_f32<<<g, b, 0, (cudaStream_t)stream>>>(d_src, spitch / 4, sw, sh, d_dst, dpitch / 4, dw, dh, A);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

// ---- stage-level entry points of the feature kernels (launches only; extract() is the production sequence)

int tvl1_k_gauss7_u8(const uint8_t* d_src, size_t spitch, int w, int h, uint8_t* d_dst, size_t dpitch, void* stream)
{
    if (!d_src || !d_dst || w <= 0 || h <= 0 || spitch < (size_t)w || dpitch < (size_t)w) return fail(TVL1_ERR_INVALID, "bad argument");
    dim3 b(32, 8), g(cdivf(w, 32), cdivf(h, 8));
    k_gauss7_u8<<<g, b, 0, (cudaStream_t)stream>>>(d_src, spitch, w, h, d_dst, dpitch);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_k_fast_corners(const uint8_t* d_img, size_t pitch, int w, int h, int border, int t, float* d_score, int spitch,
                        void* d_cand, int cap, int* d_count, int* d_hist, void* stream)
{
    if (!d_img || !d_score || !d_cand || !d_count || !d_hist || w <= 0 || h <= 0 || w > 65535 || h > 65535 ||
        pitch < (size_t)w || spitch < w || border < 4 || cap < 0)
        return fail(TVL1_ERR_INVALID, "bad argument");
    dim3 b(32, 8), g(cdivf(w, 32), cdivf(h, 8));
    k_fast_score<<<g, b, 0, (cudaStream_t)stream>>>(d_img, pitch, w, h, border, t, d_score, spitch);
    k_nms_harris<<<g, b, 0, (cudaStream_t)stream>>>(d_score, spitch, d_img, pitch, w, h, border, (Cand*)d_cand, cap, d_count, d_hist);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_k_describe(const uint8_t* d_img, size_t pitch, const uint8_t* d_blur, size_t bpitch, const void* d_cand, int n,
                    float scale, int level, void* d_kp, uint32_t* d_desc, void* stream)
{
    if (!d_img || !d_blur || !d_cand || !d_kp || !d_desc || n < 0) return fail(TVL1_ERR_INVALID, "bad argument");
    int dev = 0;
    CKF(cudaGetDevice(&dev));
    if (int rc = upload_tables(dev)) return rc;
    if (n == 0) return TVL1_OK;
    k_describe<<<cdivf(n * 32, 128), 128, 0, (cudaStream_t)stream>>>(d_img, pitch, d_blur, bpitch, (const Cand*)d_cand, n, scale,
                                                                     level, (KeyPt*)d_kp, d_desc, 0);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_k_knn2(const uint32_t* d_q, int nq, const uint32_t* d_t, int nt, int* d_idx1, int* d_d1, int* d_d2, void* stream)
{
    if (!d_q || !d_t || !d_idx1 || !d_d1 || !d_d2 || nq < 0 || nt < 1) return fail(TVL1_ERR_INVALID, "bad argument");
    if (nq == 0) return TVL1_OK;
    k_knn2<<<cdivf(nq, 128), 128, 0, (cudaStream_t)stream>>>(d_q, nq, d_t, nt, d_idx1, d_d1, d_d2);
    CKF(cudaGetLastError());
    return TVL1_OK;
}

int tvl1_features_extract(tvl1_handle* H, const uint8_t* d_img, size_t pitch, int w, int h, const tvl1_feature_params* prm,
                          void* d_kp, uint32_t* d_desc, int cap, int* n_out, void* stream)
{
    if (!H || !d_img || !prm || !d_kp || !d_desc || !n_out) return fail(TVL1_ERR_INVALID, "null argument");
    if (w <= 0 || h <= 0 || pitch < (size_t)w || w > 65535 || h > 65535) return fail(TVL1_ERR_INVALID, "bad geometry");
    const tvl1_feature_params P = *prm;
    int rc = check_feature_params(P);
    if (rc) return rc;
    if (cap < P.nfeatures) return fail(TVL1_ERR_INVALID, "cap %d < nfeatures %d", cap, P.nfeatures);
    FeatScratch* S = nullptr;
    if ((rc = feature_scratch(H, &S))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    int n = 0;
    if ((rc = extract(*S, d_img, pitch, w, h, P, 0, st, &n))) return rc;
    if (n > 0) {
        CKF(cudaMemcpyAsync(d_kp, S->kp[0], sizeof(KeyPt) * (size_t)n, cudaMemcpyDeviceToDevice, st));
        CKF(cudaMemcpyAsync(d_desc, S->desc[0], 32 * (size_t)n, cudaMemcpyDeviceToDevice, st));
    }
    CKF(cudaStreamSynchronize(st));
    *n_out = n;
    return TVL1_OK;
}

}  // extern "C"
