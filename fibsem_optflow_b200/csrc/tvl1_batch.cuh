// tvl1_batch.cuh -- the kernels of tvl1_calc_batch_u8: n pairs of one size per launch.
//
// The batch arena holds n copies of a pair's state at one fixed distance, `stride` bytes (a multiple of 256): pair b's
// copy of a plane -- and its Ctrl -- is the pair-0 pointer plus b * stride.  blockIdx.z is the pair everywhere.  These
// kernels serve the small-frame regime, where a pair alone leaves most of the GPU idle and the launch latency
// dominates: no TMA staging, plain global loads, and the iteration is the in-place two-launch form of k_gamma_u /
// k_gamma_p with the IEEE operators and the canonical hypot.  Every value is computed with the operations, and in the
// order, of the single-pair kernels (tvl1_kernels.cuh), so each pair's flow and iteration counts are those of
// tvl1_calc_u8.  Each pair keeps its own stop state in its own Ctrl; every kernel but the warp returns at once for a
// pair whose `done` is set.
#pragma once
#include "tvl1_kernels.cuh"

namespace tvl1 {

template <class T>
__device__ __forceinline__ T* at_pair(T* p, size_t stride, int b)
{
    return reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + stride * (size_t)b);
}

// A.2: 8-bit -> fp32, as k_convert_u8.  src: the 2n frame pointers, frame0 of every pair then frame1 of every pair;
// blockIdx.z = 2 * pair + frame
__global__ void __launch_bounds__(256) k_bconvert_u8(const uint8_t* const* __restrict__ src, size_t pitch0, size_t pitch1,
                                                     int w, int h, float* I0, float* I1, int dpitch, size_t stride)
{
    const int b = blockIdx.z >> 1, f = blockIdx.z & 1;
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (y >= h || x >= w) return;
    const uint8_t* s = src[f * (gridDim.z >> 1) + b] + (size_t)y * (f ? pitch1 : pitch0) + x;
    float4 o;
    if (x + 3 < w && ((reinterpret_cast<uintptr_t>(s) & 3) == 0)) {
        const uchar4 v = *reinterpret_cast<const uchar4*>(s);
        o = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
    } else {
        o.x = (float)s[0];
        o.y = x + 1 < w ? (float)s[1] : 0.f;
        o.z = x + 2 < w ? (float)s[2] : 0.f;
        o.w = x + 3 < w ? (float)s[3] : 0.f;
    }
    *reinterpret_cast<float4*>(at_pair(f ? I1 : I0, stride, b) + (size_t)y * dpitch + x) = o;
}

// two planes of every pair resized alike (A.2): the pyramid step of I0 | I1 or the flow upsample of u1 | u2.
// blockIdx.z = 2 * pair + plane.  With ctrl, the source is the twin ctrl->ucur[level] holds the live flow in.
struct BResizeArgs {
    const float* src[2][2];   // [plane][twin], pair 0
    float* dst[2];
    const Ctrl* ctrl;         // null: twin 0
    int level;
    int sw, sh, sp, dw, dh, dp;
    double scale_x, scale_y, mul;   // k_resize's arguments
    int apply_mul;
    size_t stride;
};

__device__ __forceinline__ void bresize_planes(const BResizeArgs& a, const float*& src, float*& dst)
{
    const int b = blockIdx.z >> 1, pl = blockIdx.z & 1;
    const int t = a.ctrl ? at_pair(a.ctrl, a.stride, b)->ucur[a.level] : 0;
    src = at_pair(a.src[pl][t], a.stride, b);
    dst = at_pair(a.dst[pl], a.stride, b);
}

// bilinear, as k_resize
__global__ void __launch_bounds__(256) k_bresize(const __grid_constant__ BResizeArgs a)
{
    const int dx = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int dy = blockIdx.y * blockDim.y + threadIdx.y;
    if (dx >= a.dw || dy >= a.dh) return;
    const float* src;
    float* dst;
    bresize_planes(a, src, dst);
    float fy = (float)__dsub_rn(__dmul_rn((double)dy + 0.5, a.scale_y), 0.5);
    const int sy = __float2int_rd(fy);
    fy -= (float)sy;
    const float b0 = 1.f - fy, b1 = fy;
    const float* S0 = src + (size_t)min(max(sy, 0), a.sh - 1) * a.sp;
    const float* S1 = src + (size_t)min(max(sy + 1, 0), a.sh - 1) * a.sp;
    float* out = dst + (size_t)dy * a.dp + dx;
    for (int k = 0; k < 4 && dx + k < a.dw; k++) out[k] = resize_px(S0, S1, a.sw, dx + k, a.scale_x, b0, b1, a.mul, a.apply_mul);
}

// scaleStep 0.5: OpenCV's INTER_AREA path, as k_resize_half
__global__ void __launch_bounds__(256) k_bresize_half(const __grid_constant__ BResizeArgs a)
{
    const int dx = blockIdx.x * blockDim.x + threadIdx.x;
    const int dy = blockIdx.y * blockDim.y + threadIdx.y;
    if (dx >= a.dw || dy >= a.dh) return;
    const float* src;
    float* dst;
    bresize_planes(a, src, dst);
    const int sw = a.sw, sh = a.sh, spitch = a.sp;
    const int sx = 2 * dx, sy = 2 * dy;
    const float* S0 = src + (size_t)sy * spitch + sx;
    float d;
    if (sx + 1 < sw && sy + 1 < sh) {
        const float* S1 = S0 + spitch;
        const float s0 = S0[0], s1 = S0[1], s2 = S1[0], s3 = S1[1];
        d = dx < (sw / 2) / 4 * 4 ? ((s0 + s1) + (s2 + s3)) * 0.25f : (s0 + s1 + s2 + s3) * 0.25f;
    } else if (sx >= sw || sy >= sh) {
        d = 0.f;
    } else {
        float sum = 0.f;
        int count = 0;
        for (int r = 0; r < 2 && sy + r < sh; r++)
            for (int c = 0; c < 2 && sx + c < sw; c++) { sum += S0[(size_t)r * spitch + c]; count++; }
        d = sum / (float)count;
    }
    dst[(size_t)dy * a.dp + dx] = scale_px(d, a.mul, a.apply_mul);
}

struct BWarpArgs {
    const float *I0, *I1;
    const float* u1[2];
    const float* u2[2];
    float *I1wx, *I1wy, *rho_c;
    float* pz[4];   // first warp of a level: p11 .. p22, which start the level at zero; null otherwise
    Ctrl* ctrl;
    int w, h, pitch, level;
    size_t stride;
};

// A.3 + A.4, one pixel per thread: k_warp's pixel-by-pixel path (its source position, its 6x6 ring gathered with
// replicate addressing, warp_combine), writing I1wx, I1wy and rho_c.  Like k_warp it re-arms the pair's stop test.
__global__ void __launch_bounds__(256) k_bwarp(const __grid_constant__ BWarpArgs a)
{
    __shared__ __align__(16) float tab[128];
    const int tid = threadIdx.y * 32 + threadIdx.x, b = blockIdx.z;
    if (tid < 128) tab[tid] = c_cubic_tab[tid];
    Ctrl* c = at_pair(a.ctrl, a.stride, b);
    if (blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) {   // error = FLT_MAX
        c->done = 0; c->replay = 0; c->single = 0; c->inner = 0; c->error = 3.0e38f;
    }
    __syncthreads();
    const int w = a.w, h = a.h, pitch = a.pitch;
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= w || y >= h) return;
    const int uc = c->ucur[a.level];
    const size_t i = (size_t)y * pitch + x;
    const float u1 = at_pair(a.u1[uc], a.stride, b)[i], u2 = at_pair(a.u2[uc], a.stride, b)[i];
    const float i0 = at_pair(a.I0, a.stride, b)[i];
    const float* I1 = at_pair(a.I1, a.stride, b);
    // source position, as k_warp's
    const float mx = (float)x + u1, my = (float)y + u2;
    const int qx = __float2int_rn(mx * 32.f), qy = __float2int_rn(my * 32.f);
    const int sx = min(max(qx >> 5, -32768), 32767) - 1;
    const int sy = min(max(qy >> 5, -32768), 32767) - 1;
    float iw = 0.f, iwx = 0.f, iwy = 0.f;
    if (!(sx >= w || sx + 4 <= 0 || sy >= h || sy + 4 <= 0)) {   // outside: all three samples are 0
        const bool inside = (unsigned)sx < (unsigned)max(w - 3, 0) && (unsigned)sy < (unsigned)max(h - 3, 0);
        float wt[16];
        warp_weights(tab, ((qy & 31) << 5) | (qx & 31), wt);
        float nb[6][6];
        nb[0][0] = nb[0][5] = nb[5][0] = nb[5][5] = 0.f;   // corners are never used
#pragma unroll
        for (int r = 0; r < 6; r++) {
            const float* g = I1 + (size_t)min(max(sy - 1 + r, 0), h - 1) * pitch;
#pragma unroll
            for (int cc = 0; cc < 6; cc++)
                if (!((r == 0 || r == 5) && (cc == 0 || cc == 5))) nb[r][cc] = g[min(max(sx - 1 + cc, 0), w - 1)];
        }
        warp_combine<0, 6>(nb, wt, inside, sx, sy, w, h, iw, iwx, iwy);
    }
    at_pair(a.I1wx, a.stride, b)[i] = iwx;
    at_pair(a.I1wy, a.stride, b)[i] = iwy;
    at_pair(a.rho_c, a.stride, b)[i] = (iw - iwx * u1 - iwy * u2 - i0);
    if (a.pz[0])
        for (int k = 0; k < 4; k++) at_pair(a.pz[k], a.stride, b)[i] = 0.f;
}

struct BMedianArgs {
    float* u1[2];
    float* u2[2];
    Ctrl* ctrl;
    int w, h, pitch, level, slot;
    size_t stride;
};

// end of a median launch for pair b: its last block flips the pair's ucur and counts the outer iteration
__device__ __forceinline__ void bmedian_done(const BMedianArgs& a, Ctrl* c, int uc)
{
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        __threadfence();
        s_last = atomicAdd(&c->ticket, 1u) == gridDim.x - 1;
        if (s_last) {
            c->ucur[a.level] = uc ^ 1;
            c->outer[a.slot] += 1;
            c->ticket = 0;
        }
    }
}

// A.7: medianBlur(u, 5) of u1 and u2, replicate border, [cur] -> [cur^1]: 8 outputs of a row per thread, selected
// by k_median5's network from clamped global loads
__global__ void __launch_bounds__(256) k_bmedian5(const __grid_constant__ BMedianArgs a)
{
    const int b = blockIdx.z;
    Ctrl* c = at_pair(a.ctrl, a.stride, b);
    if (*reinterpret_cast<volatile int*>(&c->done)) return;
    const int uc = c->ucur[a.level];
    const int w = a.w, h = a.h, pitch = a.pitch;
    const int qx = (w + 7) / 8;
    const long long n = (long long)qx * h * 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int z = (int)(i / ((long long)qx * h));
        const long long r = i - (long long)z * qx * h;
        const int y = (int)(r / qx), x = (int)(r - (long long)y * qx) * 8;
        const float* src = at_pair(z == 0 ? a.u1[uc] : a.u2[uc], a.stride, b);
        float* dst = at_pair(z == 0 ? a.u1[uc ^ 1] : a.u2[uc ^ 1], a.stride, b);
        float col[12][5];
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const float* row = src + (size_t)min(max(y - 2 + k, 0), h - 1) * pitch;
#pragma unroll
            for (int j = 0; j < 12; j++) col[j][k] = row[min(max(x - 2 + j, 0), w - 1)];
        }
        float o[8];
        median5_select8(col, o);
        float* out = dst + (size_t)y * pitch + x;
        *reinterpret_cast<float4*>(out) = make_float4(o[0], o[1], o[2], o[3]);
        if (x + 4 < w) *reinterpret_cast<float4*>(out + 4) = make_float4(o[4], o[5], o[6], o[7]);
    }
    bmedian_done(a, c, uc);
}

// medianBlur(u, 3), as k_median3
__global__ void __launch_bounds__(256) k_bmedian3(const __grid_constant__ BMedianArgs a)
{
    const int b = blockIdx.z;
    Ctrl* c = at_pair(a.ctrl, a.stride, b);
    if (*reinterpret_cast<volatile int*>(&c->done)) return;
    const int uc = c->ucur[a.level];
    const int w = a.w, h = a.h, pitch = a.pitch;
    const int qx = (w + 3) / 4;
    const long long n = (long long)qx * h * 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int z = (int)(i / ((long long)qx * h));
        const long long r = i - (long long)z * qx * h;
        const int y = (int)(r / qx), x = (int)(r - (long long)y * qx) * 4;
        median3_px4(at_pair(z == 0 ? a.u1[uc] : a.u2[uc], a.stride, b), at_pair(z == 0 ? a.u1[uc ^ 1] : a.u2[uc ^ 1], a.stride, b),
                    w, h, pitch, x, y);
    }
    bmedian_done(a, c, uc);
}

// ---- the primal-dual iteration (A.5), in place on u[ucur] and p: two launches per inner iteration
//   k_biter_u  estimateV + divergence + estimateU (u' of a pixel needs its own u and p at x-1 / y-1, which this
//              kernel does not write), the error sum over the pair's per-block partials and the pair's stop test
//   k_biter_p  forward gradient of u' + dual update (p' of a pixel needs its own p and u' at x+1 / y+1)
struct BIterArgs {
    const float *I1wx, *I1wy, *rho_c;
    float* u1[2];
    float* u2[2];
    float *p11, *p12, *p21, *p22;
    int w, h, pitch;
    float l_t, theta, taut, scaled_eps;
    int level, slot, inner_max;
    Ctrl* ctrl;
    double* partials;   // per pair: one per block (gridDim.x)
    size_t stride;
};

#define TVL1_BITER_NW 4            // warps per block of the batched iteration kernels
#define TVL1_BATCH_MAX_BLOCKS 256  // blocks per pair of a batched launch (per-pair partial sums of the error)

__global__ void __launch_bounds__(32 * TVL1_BITER_NW) k_biter_u(const __grid_constant__ BIterArgs a)
{
    const int b = blockIdx.z;
    Ctrl* c = at_pair(a.ctrl, a.stride, b);
    if (*reinterpret_cast<volatile int*>(&c->done)) return;
    if (*reinterpret_cast<volatile int*>(&c->inner) >= a.inner_max) return;
    const int uc = c->ucur[a.level];
    const size_t st = a.stride;
    float* __restrict__ u1 = at_pair(a.u1[uc], st, b);
    float* __restrict__ u2 = at_pair(a.u2[uc], st, b);
    const float* __restrict__ p11 = at_pair(a.p11, st, b);
    const float* __restrict__ p12 = at_pair(a.p12, st, b);
    const float* __restrict__ p21 = at_pair(a.p21, st, b);
    const float* __restrict__ p22 = at_pair(a.p22, st, b);
    const float* __restrict__ I1wx = at_pair(a.I1wx, st, b);
    const float* __restrict__ I1wy = at_pair(a.I1wy, st, b);
    const float* __restrict__ rho_c = at_pair(a.rho_c, st, b);
    const int w = a.w, h = a.h, pitch = a.pitch, lane = threadIdx.x;
    const float l_t = a.l_t, theta = a.theta;
    const int nsx = (w + 127) / 128, ntiles = nsx * h;
    double acc[1] = {0.0};
    for (int tile = blockIdx.x * TVL1_BITER_NW + threadIdx.y; tile < ntiles; tile += gridDim.x * TVL1_BITER_NW) {
        const int y = tile / nsx, x = (tile - y * nsx) * 128 + lane * 4;
        if (x >= w) continue;
        const size_t i = (size_t)y * pitch + x;
        float wx[4], wy[4], rc[4], o1[4], o2[4], a1[4], b1[4], a2[4], b2[4], t1[4], t2[4];
        unpack4(ld4(I1wx + i), wx); unpack4(ld4(I1wy + i), wy); unpack4(ld4(rho_c + i), rc);
        unpack4(ld4(u1 + i), o1); unpack4(ld4(u2 + i), o2);
        unpack4(ld4(p11 + i), a1); unpack4(ld4(p12 + i), b1);
        unpack4(ld4(p21 + i), a2); unpack4(ld4(p22 + i), b2);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        unpack4(y > 0 ? ld4(p12 + i - pitch) : z, t1);   // b(y-1); zeros above the image: b - 0 == b
        unpack4(y > 0 ? ld4(p22 + i - pitch) : z, t2);
        float l1 = 0.f, l2 = 0.f;                        // a(x-1)
        if (x > 0) { l1 = p11[i - 1]; l2 = p21[i - 1]; }
        float n1[4], n2[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            n1[k] = o1[k]; n2[k] = o2[k];
            if (x + k >= w) continue;
            const float g = wx[k] * wx[k] + wy[k] * wy[k];
            const float rho = rc[k] + (wx[k] * o1[k] + wy[k] * o2[k]);
            float d1 = 0.f, d2 = 0.f;
            if (rho < -l_t * g) { d1 = l_t * wx[k]; d2 = l_t * wy[k]; }
            else if (rho > l_t * g) { d1 = -l_t * wx[k]; d2 = -l_t * wy[k]; }
            else if (g > FLT_EPSILON) { const float fi = -rho / g; d1 = fi * wx[k]; d2 = fi * wy[k]; }
            const float v1 = o1[k] + d1, v2 = o2[k] + d2;
            const float pl1 = k == 0 ? l1 : a1[k - 1], pl2 = k == 0 ? l2 : a2[k - 1];
            float div1, div2;
            if (x + k == 0) {   // first column: a + b - b(y-1)
                div1 = a1[k] + b1[k] - t1[k]; div2 = a2[k] + b2[k] - t2[k];
            } else {
                div1 = (a1[k] - pl1) + (b1[k] - t1[k]); div2 = (a2[k] - pl2) + (b2[k] - t2[k]);
            }
            n1[k] = v1 + theta * div1; n2[k] = v2 + theta * div2;
            const float e1 = n1[k] - o1[k], e2 = n2[k] - o2[k];
            const float term = e1 * e1 + e2 * e2;
            acc[0] += (double)term;
        }
        *reinterpret_cast<float4*>(u1 + i) = pack4(n1);
        *reinterpret_cast<float4*>(u2 + i) = pack4(n2);
    }
    double tot[1];
    if (!reduce_errors<TVL1_BITER_NW, 1>(acc, at_pair(a.partials, st, b), c, tot)) return;
    const float e = (float)tot[0];
    c->iters[a.slot] += 1;
    c->inner += 1;
    c->error = e;
    c->ticket = 0;
    c->pad[0] = 1;   // the dual update of this iteration is due (it also runs for the iteration that stops)
    if (!(e > a.scaled_eps)) c->done = 1;
}

__global__ void __launch_bounds__(32 * TVL1_BITER_NW) k_biter_p(const __grid_constant__ BIterArgs a)
{
    const int b = blockIdx.z;
    Ctrl* c = at_pair(a.ctrl, a.stride, b);
    if (!*reinterpret_cast<volatile int*>(&c->pad[0])) return;   // no estimateU ran for this pair in front of this launch
    const int uc = c->ucur[a.level];
    const size_t st = a.stride;
    const float* __restrict__ u[2] = {at_pair(a.u1[uc], st, b), at_pair(a.u2[uc], st, b)};
    float* __restrict__ pa[2] = {at_pair(a.p11, st, b), at_pair(a.p21, st, b)};
    float* __restrict__ pb[2] = {at_pair(a.p12, st, b), at_pair(a.p22, st, b)};
    const int w = a.w, h = a.h, pitch = a.pitch, lane = threadIdx.x;
    const float taut = a.taut;
    const int nsx = (w + 127) / 128, ntiles = nsx * h;
    for (int tile = blockIdx.x * TVL1_BITER_NW + threadIdx.y; tile < ntiles; tile += gridDim.x * TVL1_BITER_NW) {
        const int y = tile / nsx, x = (tile - y * nsx) * 128 + lane * 4;
        if (x >= w) continue;
        const size_t i = (size_t)y * pitch + x;
#pragma unroll
        for (int ch = 0; ch < 2; ch++) {
            float cu[4], dn[4], qa[4], qb[4];
            unpack4(ld4(u[ch] + i), cu);
            unpack4(y < h - 1 ? ld4(u[ch] + i + pitch) : ld4(u[ch] + i), dn);
            const float right = x + 4 < w ? u[ch][i + 4] : 0.f;
            unpack4(ld4(pa[ch] + i), qa); unpack4(ld4(pb[ch] + i), qb);
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (x + k >= w) continue;
                const float ux = x + k == w - 1 ? 0.f : (k == 3 ? right : cu[k + 1]) - cu[k];
                const float uy = y == h - 1 ? 0.f : dn[k] - cu[k];
                const float g = hypot_canon(ux, uy);
                const float ng = 1.0f + taut * g;
                qa[k] = (qa[k] + taut * ux) / ng;
                qb[k] = (qb[k] + taut * uy) / ng;
            }
            *reinterpret_cast<float4*>(pa[ch] + i) = pack4(qa);
            *reinterpret_cast<float4*>(pb[ch] + i) = pack4(qb);
        }
    }
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        __threadfence();
        s_last = atomicAdd(&c->ticket, 1u) == gridDim.x - 1;
        if (s_last) { c->ticket = 0; c->pad[0] = 0; }
    }
}

// the first `words` 32-bit words of every pair's Ctrl -> dst[pair * sizeof(Ctrl) / 4 + word] in pinned host memory
// (the stop-test read-back of the whole batch in one launch; see copy_words)
__global__ void __launch_bounds__(256) k_bctrl_read(const Ctrl* ctrl, size_t stride, int words, int n, int* dst)
{
    const int per = (int)(sizeof(Ctrl) / 4);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n * words; i += gridDim.x * blockDim.x) {
        const int b = i / words, k = i - b * words;
        dst[(size_t)b * per + k] = reinterpret_cast<const int*>(at_pair(ctrl, stride, b))[k];
    }
    __threadfence_system();
}

}  // namespace tvl1
