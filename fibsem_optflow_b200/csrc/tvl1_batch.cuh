// tvl1_batch.cuh -- the kernels only batches (tvl1_calc_batch_ex, tvl1_calc_batch_u8) launch: n pairs of one size
// per launch.
//
// The batch arena holds n copies of a pair's state at one fixed distance, `stride` bytes (a multiple of 256): pair b's
// copy of a plane -- and its Ctrl -- is the pair-0 pointer plus b * stride (at_pair).  blockIdx.z is the pair
// everywhere.  These kernels serve the small-frame regime, where a pair alone leaves most of the GPU idle and the
// launch latency dominates: no TMA staging, plain global loads.  A batch also launches the kernels of tvl1_kernels.cuh
// that take a pair: k_resize / k_resize_half / k_resize_cuda, k_median3, k_warp_cuda and the plain iteration
// k_plain_u / k_plain_p.  Every value is computed with the operations, and in the order, of the single-pair kernels,
// so each pair's flow and iteration counts are those of tvl1_calc_ex.  Each pair keeps its own stop state in its own Ctrl; every kernel but
// the warp returns at once for a pair whose `done` is set.
#pragma once
#include "tvl1_kernels.cuh"

namespace tvl1 {

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

// A.2 for fp32 frames, as k_convert_f32 (convert_f32_px); pitch0 / pitch1 in elements; src and blockIdx.z as
// k_bconvert_u8's
__global__ void __launch_bounds__(256) k_bconvert_f32(const float* const* __restrict__ src, size_t pitch0, size_t pitch1,
                                                      int w, int h, float* I0, float* I1, int dpitch, size_t stride)
{
    const int b = blockIdx.z >> 1, f = blockIdx.z & 1;
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (y >= h || x >= w) return;
    const float* s = src[f * (gridDim.z >> 1) + b] + (size_t)y * (f ? pitch1 : pitch0) + x;
    *reinterpret_cast<float4*>(at_pair(f ? I1 : I0, stride, b) + (size_t)y * dpitch + x) = convert_f32_px(s, x, w);
}

// useInitialFlow: every pair's (u0, v0) -> its level-0 twin 0 (u1, u2), columns 0 .. w - 1 as the single pair's
// row copy.  src: the 2n plane pointers, u0 of every pair then v0 of every pair; spitch in elements;
// blockIdx.z = 2 * pair + plane
__global__ void __launch_bounds__(256) k_bload_flow(const float* const* __restrict__ src, size_t spitch, int w, int h,
                                                    float* u1, float* u2, int dpitch, size_t stride)
{
    const int b = blockIdx.z >> 1, f = blockIdx.z & 1;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (y >= h || x >= w) return;
    at_pair(f ? u2 : u1, stride, b)[(size_t)y * dpitch + x] = __ldg(src[f * (gridDim.z >> 1) + b] + (size_t)y * spitch + x);
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

// A.7: medianBlur(u, 5) of u1 and u2, replicate border, [cur] -> [cur^1]: 8 outputs of a row per thread, selected
// by k_median5's network from clamped global loads (MedianArgs::tm is not used); the bookkeeping of k_median3
__global__ void __launch_bounds__(256) k_bmedian5(const __grid_constant__ MedianArgs a, size_t stride)
{
    const int b = blockIdx.z;
    Ctrl* c = at_pair(a.ctrl, stride, b);
    if (*reinterpret_cast<volatile int*>(&c->done)) return;
    const int uc = c->ucur[a.level];
    const int w = a.w, h = a.h, pitch = a.pitch;
    const int qx = (w + 7) / 8;
    const long long n = (long long)qx * h * 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int z = (int)(i / ((long long)qx * h));
        const long long r = i - (long long)z * qx * h;
        const int y = (int)(r / qx), x = (int)(r - (long long)y * qx) * 8;
        const float* src = at_pair(z == 0 ? a.u1[uc] : a.u2[uc], stride, b);
        float* dst = at_pair(z == 0 ? a.u1[uc ^ 1] : a.u2[uc ^ 1], stride, b);
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
    median_done(a, c, uc);
}

#define TVL1_BATCH_MAX_BLOCKS 256  // blocks per pair of a batched launch (per-pair partial sums of the error)

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
