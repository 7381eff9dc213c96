// clahe16.cu — CLAHE in OpenCV semantics for uint16 images: 65 536 bins, uint16 LUTs
// (cv::CLAHE::apply on CV_16UC1; SURVEY.md §8(a) A1', §8(f) F2, Appendix A).  This is the only CLAHE
// variant with an executable third-party oracle in the image (cv2 4.13), and the natural mode for
// 12/16-bit CT / MR / X-ray data: no quantisation to 256 levels anywhere.
//
// A 65 536-bin histogram does not fit next to a block's other state as 32-bit counters (256 KB), and
// 16-bit counters overflow for tiles of >= 65 536 pixels, so one block (1024 threads) owns one tile and
// sweeps the grey range in two halves of 32 768 bins (128 KB of 32-bit shared-memory counters, padded
// by one word per 32 so that "thread t owns bins 32t .. 32t+31" is bank-conflict free):
//   phase A (only when clipping):  clipped = sum max(h - clip, 0)          -> redistribution batch / residual
//   phase B:  h' = min(h, clip) + batch + residual term;  running prefix sum;  lut = sat(rint(cum * scale))
// Each half re-reads the tile (8 KB .. 128 KB, L1/L2 resident); the 128 KB LUT per tile is written once
// with 16-byte stores and stays in L2 for the interpolation pass, which gathers four uint16 entries
// per pixel.  The caller's workspace bounds how many images' LUTs exist at a time (mie_clahe loops over
// groups of images), so a batch never needs more LUT memory than fits in L2.
#include <cooperative_groups.h>


#include "clahe.cuh"

namespace mie {

constexpr int kBins16 = 65536;
constexpr int kHalf16 = 32768;
constexpr int kThreads16 = 1024;
constexpr int kOwn16 = kHalf16 / kThreads16;  // 32 consecutive bins per thread and half

__device__ __forceinline__ int pad16(int i) { return i + (i >> 5); }

struct Lut16Params {
    int clip;         // per-bin ceiling (0 = clipping disabled)
    float lut_scale;  // float(65535) / float(area)
};

// Histogram of one half of the grey range of the block's tile (reflect-101 padded beyond the image).
__device__ __forceinline__ void tile_hist_half(const uint16_t* __restrict__ plane, int64_t ssh, const ClaheGeom& g,
                                               int ty, int tx, int half, int* s_h) {
    for (int i = threadIdx.x; i < kHalf16 + kHalf16 / 32; i += kThreads16) s_h[i] = 0;
    __syncthreads();
    const int area = g.th * g.tw;
    for (int i = threadIdx.x; i < area; i += kThreads16) {
        const int yy = i / g.tw, xx = i - yy * g.tw;
        const int sy = border_index(ty * g.th + yy, g.h, MIE_BORDER_REFLECT);
        const int sx = border_index(tx * g.tw + xx, g.w, MIE_BORDER_REFLECT);
        const int v = plane[(int64_t)sy * ssh + sx];
        if ((v >> 15) == half) atomicAdd(&s_h[pad16(v & (kHalf16 - 1))], 1);
    }
    __syncthreads();
}

__device__ __forceinline__ int block_sum_1024(int v, int* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    int t = s_red[lane];
    t = warp_sum(t);
    return t;
}

// Exclusive prefix over the 1024 threads; *total receives the block sum.
__device__ __forceinline__ int block_excl_scan_1024(int v, int* s_red, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_red[warp] = incl;
    __syncthreads();
    int wv = s_red[lane], winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += t;
    }
    const int warp_off = __shfl_sync(0xffffffffu, winc - wv, warp);
    *total = __shfl_sync(0xffffffffu, winc, 31);
    return warp_off + incl - v;
}

__global__ void __launch_bounds__(kThreads16)
clahe16_lut_kernel(const uint16_t* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, Lut16Params lp,
                   uint16_t* __restrict__ luts) {
    extern __shared__ __align__(16) int s_h[];  // kHalf16 + kHalf16/32 counters
    __shared__ int s_red[32];
    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % g.gw), ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const uint16_t* plane = src + n * ssn;
    const int tid = threadIdx.x;

    int rb = 0, res = 0, step = 1;
    if (lp.clip > 0) {
        int local = 0;
        for (int half = 0; half < 2; ++half) {
            tile_hist_half(plane, ssh, g, ty, tx, half, s_h);
#pragma unroll 8
            for (int k = 0; k < kOwn16; ++k) local += max(s_h[tid * (kOwn16 + 1) + k] - lp.clip, 0);
            __syncthreads();
        }
        const int clipped = block_sum_1024(local, s_red);
        rb = clipped / kBins16;
        res = clipped - rb * kBins16;
        step = res ? max(kBins16 / res, 1) : 1;
    }
    int running = 0;
    uint16_t* lut = luts + tile * (int64_t)kBins16;
    for (int half = 0; half < 2; ++half) {
        tile_hist_half(plane, ssh, g, ty, tx, half, s_h);
        int hv[kOwn16];
        const int u0 = half * kHalf16 + tid * kOwn16;
        int sum = 0;
#pragma unroll
        for (int k = 0; k < kOwn16; ++k) {
            int c = s_h[tid * (kOwn16 + 1) + k];
            if (lp.clip > 0) {
                const int u = u0 + k;
                const int q = u / step;
                c = min(c, lp.clip) + rb + ((res && q * step == u && q < res) ? 1 : 0);
            }
            sum += c;
            hv[k] = sum;  // inclusive within the thread
        }
        int total;
        const int base = running + block_excl_scan_1024(sum, s_red, &total);
        running += total;
        uint32_t packed[kOwn16 / 2];
#pragma unroll
        for (int k = 0; k < kOwn16; k += 2) {
            float f0 = rintf(__fmul_rn((float)(base + hv[k]), lp.lut_scale));
            float f1 = rintf(__fmul_rn((float)(base + hv[k + 1]), lp.lut_scale));
            f0 = fminf(fmaxf(f0, 0.0f), 65535.0f);
            f1 = fminf(fmaxf(f1, 0.0f), 65535.0f);
            packed[k / 2] = (uint32_t)(int)f0 | ((uint32_t)(int)f1 << 16);
        }
        uint4* dst = reinterpret_cast<uint4*>(lut + u0);
#pragma unroll
        for (int k = 0; k < kOwn16 / 8; ++k)
            dst[k] = make_uint4(packed[4 * k], packed[4 * k + 1], packed[4 * k + 2], packed[4 * k + 3]);
        __syncthreads();
    }
}

// ---------------------------------------------------------------- tiles of fewer than 65 536 pixels
// The common case (64x64 .. 255x255-pixel tiles): every count fits 16 bits, so the WHOLE grey range fits the
// 128 KB of shared memory as 16-bit counters packed two per word — one zeroing and one pass over the tile
// instead of four of each — and the rest is trimmed to what the 65 536 LUT entries per tile really need:
//   * the residual rule (+1 at bins 0, step, 2 step, ... for the first `res` positions) walks a running
//     "next multiple of step" instead of dividing per bin;
//   * lut = sat(rint(float(cum) * scale)) without I2F / FRND / F2I (conversion pipe, 16 lanes per clock):
//     float(cum) by OR-ing the integer into the mantissa of 2^23, rint by adding 1.5 * 2^23, the result read
//     back from the mantissa — the same values as the generic kernel, bit for bit.
// Thread t owns bins 64t .. 64t+63 = words 32t .. 32t+31 (one padding word per 32: conflict-free).
__device__ __forceinline__ int padw(int w) { return w + (w >> 5); }

__global__ void __launch_bounds__(kThreads16)
clahe16_lut_small_kernel(const uint16_t* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, Lut16Params lp,
                         uint16_t* __restrict__ luts) {
    extern __shared__ __align__(16) int s_h[];   // 32768 + 1024 words
    __shared__ int s_red[32];
    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % g.gw), ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const uint16_t* plane = src + n * ssn;
    const int tid = threadIdx.x;
    uint32_t* s_w = reinterpret_cast<uint32_t*>(s_h);
    for (int i = tid; i < kHalf16 + kHalf16 / 32; i += kThreads16) s_w[i] = 0u;
    __syncthreads();
    const int area = g.th * g.tw;
    const bool inside = (ty + 1) * g.th <= g.h && (tx + 1) * g.tw <= g.w;   // block-uniform: no reflect padding
    for (int i = tid; i < area; i += kThreads16) {
        const int yy = i / g.tw, xx = i - yy * g.tw;
        int sy = ty * g.th + yy, sx = tx * g.tw + xx;
        if (!inside) {
            sy = border_index(sy, g.h, MIE_BORDER_REFLECT);
            sx = border_index(sx, g.w, MIE_BORDER_REFLECT);
        }
        const uint32_t v = plane[(int64_t)sy * ssh + sx];
        atomicAdd(&s_w[padw((int)(v >> 1))], (v & 1u) ? 0x10000u : 1u);
    }
    __syncthreads();

    const uint32_t* mine = s_w + tid * 33;       // padw(32 tid + k) = 33 tid + k for k < 32
    const uint32_t clip = (uint32_t)lp.clip;
    int rb = 0, res = 0, step = 1;
    if (lp.clip > 0) {
        int local = 0;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            const uint32_t wv = mine[k];
            const uint32_t c0 = wv & 0xFFFFu, c1 = wv >> 16;
            local += (int)(c0 > clip ? c0 - clip : 0u) + (int)(c1 > clip ? c1 - clip : 0u);
        }
        const int clipped = block_sum_1024(local, s_red);
        rb = clipped / kBins16;
        res = clipped - rb * kBins16;
        step = res ? max(kBins16 / res, 1) : 1;
    }
    // value of bin u after clipping / redistribution; the residual walk state is (next multiple, its index)
    const int u0 = tid * 64;
    int q = (u0 + step - 1) / step, next = q * step;
    auto bin_value = [&](uint32_t c, int u) {
        if (lp.clip > 0) {
            c = min(c, clip) + (uint32_t)rb;
            if (u == next) {
                c += (res && q < res) ? 1u : 0u;
                next += step; ++q;
            }
        }
        return (int)c;
    };
    int sum = 0;
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
        const uint32_t wv = mine[k];
        sum += bin_value(wv & 0xFFFFu, u0 + 2 * k);
        sum += bin_value(wv >> 16, u0 + 2 * k + 1);
    }
    int total;
    int cum = block_excl_scan_1024(sum, s_red, &total);
    q = (u0 + step - 1) / step; next = q * step;                 // restart the walk for the second pass
    const float scale = lp.lut_scale;
    auto lut_entry = [&](int c) {                                  // sat(rint(float(c) * scale)), c < 2^23
        const float f = __fsub_rn(__uint_as_float(0x4B000000u | (uint32_t)c), 8388608.0f);
        const uint32_t r = __float_as_uint(__fadd_rn(__fmul_rn(f, scale), 12582912.0f)) - 0x4B400000u;
        return min(r, 65535u);
    };
    uint4* dst = reinterpret_cast<uint4*>(luts + tile * (int64_t)kBins16 + u0);
#pragma unroll 2
    for (int k4 = 0; k4 < 8; ++k4) {
        uint32_t packed[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = 4 * k4 + j;
            const uint32_t wv = mine[k];
            cum += bin_value(wv & 0xFFFFu, u0 + 2 * k);
            const uint32_t e0 = lut_entry(cum);
            cum += bin_value(wv >> 16, u0 + 2 * k + 1);
            packed[j] = e0 | (lut_entry(cum) << 16);
        }
        dst[k4] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    }
}

// ---------------------------------------------------------------- the same, one tile per CLUSTER of two CTAs
// With one 1 024-thread block per SM (135 KB of counters) nothing hides the latency of the per-tile passes
// (zero, count, two sweeps, two block-wide reductions).  A thread-block cluster of two 512-thread CTAs splits the
// grey range: CTA r owns bins r * 32 768 .. + 32 767 (66 KB of 16-bit counters), counts only its own pixels, and
// the two numbers the halves need from each other — the clipped excess and the prefix total of the lower half —
// travel through distributed shared memory between two cluster barriers.  Three CTAs fit an SM: 48 warps from
// three different tiles interleave.
constexpr int kClThreads = 512;

template <int NW>
__device__ __forceinline__ int block_sum_nw(int v, int* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) s_red[warp] = v;
    __syncthreads();
    int t = lane < NW ? s_red[lane] : 0;
    return warp_sum(t);
}
template <int NW>
__device__ __forceinline__ int block_excl_scan_nw(int v, int* s_red, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_red[warp] = incl;
    __syncthreads();
    int wv = lane < NW ? s_red[lane] : 0, winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += t;
    }
    const int warp_off = __shfl_sync(0xffffffffu, winc - wv, warp);
    *total = __shfl_sync(0xffffffffu, winc, 31);
    return warp_off + incl - v;
}

// `vmax` (optional): device word holding an upper bound of every pixel value of the batch (clahe16_max_kernel).  LUT
// entries above it are never looked up: only the live bins are zeroed, swept and written (spread over all threads of the
// block), and a bound below 32 768 retires the upper-half CTA at once.  12-bit data in a 16-bit container — the usual
// CT / MR case — costs 1/16 of the sweeps and of the LUT traffic, and the interpolation pass then gathers from 8 KB per
// tile instead of 128 KB.  The entries that ARE written are the same as without the bound (prefix sums only look down).
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kClThreads)
clahe16_lut_cluster_kernel(const uint16_t* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, Lut16Params lp,
                           uint16_t* __restrict__ luts, const uint32_t* __restrict__ vmax) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) int s_h[];   // 16384 + 512 words: this CTA's half of the grey range
    __shared__ int s_red[32];
    __shared__ int s_xchg[2];                    // [0] clipped excess of this half, [1] prefix total of this half
    const unsigned rank = cluster.block_rank();  // 0: bins 0 .. 32767, 1: bins 32768 .. 65535
    const int64_t tile = blockIdx.x >> 1;
    const int tx = (int)(tile % g.gw), ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const uint16_t* plane = src + n * ssn;
    const int tid = threadIdx.x;
    uint32_t* s_w = reinterpret_cast<uint32_t*>(s_h);
    // highest live bin of this half (local index; negative: the whole half lies above the bound)
    const uint32_t bound = vmax ? min(__ldg(vmax), 65535u) : 65535u;
    const bool both = bound >= (uint32_t)kHalf16;                    // cluster-uniform: does the upper half take part?
    if (!both && rank == 1) return;                                  // (the lower half then skips the cluster barriers)
    const int lmax = min((int)bound - (int)rank * kHalf16, kHalf16 - 1);
    // the live bins are spread over ALL threads: thread t owns words t * wpt .. + wpt - 1 (two bins per word), wpt the
    // smallest of 4 / 8 / 16 / 32 that covers them — 12-bit data: 8 bins per thread instead of 64 bins on 64 threads
    const int live_bins = lmax + 1;
    const int wpt = live_bins <= 4096 ? 4 : live_bins <= 8192 ? 8 : live_bins <= 16384 ? 16 : 32;
    const int w0 = tid * wpt;
    const bool live = 2 * w0 <= lmax;
    {
        const int live_words = ((lmax >> 1) / wpt + 1) * wpt;        // up to the end of the last live thread's words
        for (int i = tid; i < padw(live_words - 1) + 1; i += kClThreads) s_w[i] = 0u;
    }
    __syncthreads();
    const int area = g.th * g.tw;
    const bool inside = (ty + 1) * g.th <= g.h && (tx + 1) * g.tw <= g.w;   // block-uniform: no reflect padding
    auto count = [&](uint32_t v) {
        if ((v >> 15) == rank) atomicAdd(&s_w[padw((int)((v & 0x7FFFu) >> 1))], (v & 1u) ? 0x10000u : 1u);
    };
    // tiles inside the image with 16-byte aligned rows of a multiple of 8 pixels: ONE 128-bit load per thread and step
    // (a 64 x 64 tile is one step of the block) instead of eight dependent 2-byte loads — the count phase was the top
    // stall of the kernel (long_scoreboard 4.7 warps per issue, profiles/r2_ncu_full_clahe16_bounded_lut.txt)
    const bool vec = inside && (g.tw & 7) == 0 && (ssh & 7) == 0 && (ssn & 7) == 0 && ((uintptr_t)src & 15) == 0;
    if (vec) {
        const int gpr = g.tw >> 3, groups = g.th * gpr;
        const uint16_t* t0 = plane + (int64_t)ty * g.th * ssh + tx * g.tw;
        for (int i = tid; i < groups; i += kClThreads) {
            const int yy = i / gpr, c8 = i - yy * gpr;
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(t0 + (int64_t)yy * ssh + 8 * c8));
            count(q.x & 0xFFFFu); count(q.x >> 16); count(q.y & 0xFFFFu); count(q.y >> 16);
            count(q.z & 0xFFFFu); count(q.z >> 16); count(q.w & 0xFFFFu); count(q.w >> 16);
        }
    } else {
        for (int i = tid; i < area; i += kClThreads) {
            const int yy = i / g.tw, xx = i - yy * g.tw;
            int sy = ty * g.th + yy, sx = tx * g.tw + xx;
            if (!inside) {
                sy = border_index(sy, g.h, MIE_BORDER_REFLECT);
                sx = border_index(sx, g.w, MIE_BORDER_REFLECT);
            }
            count(plane[(int64_t)sy * ssh + sx]);
        }
    }
    __syncthreads();

    const uint32_t* mine = s_w + padw(w0);       // wpt divides 32: the thread's words are contiguous behind the padding
    const uint32_t clip = (uint32_t)lp.clip;
    int rb = 0, res = 0, step = 1;
    if (lp.clip > 0) {
        int local = 0;
        if (live) {
#pragma unroll 4
            for (int k = 0; k < wpt; ++k) {
                const uint32_t wv = mine[k];
                const uint32_t c0 = wv & 0xFFFFu, c1 = wv >> 16;
                local += (int)(c0 > clip ? c0 - clip : 0u) + (int)(c1 > clip ? c1 - clip : 0u);
            }
        }
        const int mine_clipped = block_sum_nw<kClThreads / 32>(local, s_red);
        int clipped = mine_clipped;
        if (both) {
            if (tid == 0) s_xchg[0] = mine_clipped;
            cluster.sync();
            clipped += *cluster.map_shared_rank(&s_xchg[0], rank ^ 1u);
        }
        rb = clipped / kBins16;
        res = clipped - rb * kBins16;
        step = res ? max(kBins16 / res, 1) : 1;
    }
    const int u0 = (int)rank * kHalf16 + 2 * w0;
    int q = (u0 + step - 1) / step, next = q * step;
    auto bin_value = [&](uint32_t c, int u) {
        if (lp.clip > 0) {
            c = min(c, clip) + (uint32_t)rb;
            if (u == next) {
                c += (res && q < res) ? 1u : 0u;
                next += step; ++q;
            }
        }
        return (int)c;
    };
    int sum = 0;
    if (live) {
#pragma unroll 4
        for (int k = 0; k < wpt; ++k) {
            const uint32_t wv = mine[k];
            sum += bin_value(wv & 0xFFFFu, u0 + 2 * k);
            sum += bin_value(wv >> 16, u0 + 2 * k + 1);
        }
    }
    int total;
    int cum = block_excl_scan_nw<kClThreads / 32>(sum, s_red, &total);   // dead threads add 0: prefixes only look down
    if (both) {
        if (tid == 0) s_xchg[1] = total;
        cluster.sync();
        if (rank == 1) cum += *cluster.map_shared_rank(&s_xchg[1], 0u);   // the upper half continues the lower half's prefix
    }
    q = (u0 + step - 1) / step; next = q * step;
    const float scale = lp.lut_scale;
    auto lut_entry = [&](int c) {
        const float f = __fsub_rn(__uint_as_float(0x4B000000u | (uint32_t)c), 8388608.0f);
        const uint32_t r = __float_as_uint(__fadd_rn(__fmul_rn(f, scale), 12582912.0f)) - 0x4B400000u;
        return min(r, 65535u);
    };
    uint4* dst = reinterpret_cast<uint4*>(luts + tile * (int64_t)kBins16 + u0);
    if (live) {
        for (int k4 = 0; k4 < wpt / 4; ++k4) {
            uint32_t packed[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = 4 * k4 + j;
                const uint32_t wv = mine[k];
                cum += bin_value(wv & 0xFFFFu, u0 + 2 * k);
                const uint32_t e0 = lut_entry(cum);
                cum += bin_value(wv >> 16, u0 + 2 * k + 1);
                packed[j] = e0 | (lut_entry(cum) << 16);
            }
            dst[k4] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
        }
    }
    if (both) cluster.sync();   // the peer may still be reading this CTA's s_xchg
}

// Upper bound of the pixel values of a batch: one atomicMax per block into *vmax (zeroed by the caller).
__global__ void __launch_bounds__(256)
clahe16_max_kernel(const uint16_t* __restrict__ src, int64_t ssn, int64_t ssh, int64_t n, int h, int w, uint32_t* __restrict__ vmax) {
    const int64_t rows = n * h;
    uint32_t m = 0u;
    for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < rows; r += (int64_t)gridDim.x * 8) {
        const uint16_t* row = src + (r / h) * ssn + (r % h) * ssh;
        for (int x = threadIdx.x & 31; x < w; x += 32) m = max(m, (uint32_t)row[x]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ uint32_t s_m[8];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; ++i) m = max(m, s_m[i]);
        if (m) atomicMax(vmax, m);
    }
}

// Interpolation pass (cv::CLAHE_Interpolation_Body, fp32 in OpenCV's operation order): 4 pixels per thread.
__global__ void __launch_bounds__(256)
clahe16_apply_kernel(const uint16_t* __restrict__ src, uint16_t* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                     int64_t dsh, ClaheGeom g, const uint16_t* __restrict__ luts) {
    const int x0 = (blockIdx.x * 64 + (threadIdx.x & 63)) * 4;
    const int y = blockIdx.y * 4 + (threadIdx.x >> 6);
    const int64_t n = blockIdx.z;
    if (y >= g.h || x0 >= g.w) return;
    const uint16_t* srow = src + n * ssn + (int64_t)y * ssh;
    uint16_t* drow = dst + n * dsn + (int64_t)y * dsh;
    const uint16_t* nl = luts + n * (int64_t)g.gh * g.gw * kBins16;
    int j0, j1;
    float ya, ya1;
    opencv_axis(y, __fdiv_rn(1.0f, (float)g.th), g.gh, j0, j1, ya, ya1);
    const uint16_t* r0 = nl + (int64_t)j0 * g.gw * kBins16;
    const uint16_t* r1 = nl + (int64_t)j1 * g.gw * kBins16;
    const float inv_tw = __fdiv_rn(1.0f, (float)g.tw);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int x = x0 + k;
        if (x >= g.w) break;
        int i0, i1;
        float xa, xa1;
        opencv_axis(x, inv_tw, g.gw, i0, i1, xa, xa1);
        const int v = srow[x];
        const float l11 = (float)__ldg(r0 + (int64_t)i0 * kBins16 + v), l12 = (float)__ldg(r0 + (int64_t)i1 * kBins16 + v);
        const float l21 = (float)__ldg(r1 + (int64_t)i0 * kBins16 + v), l22 = (float)__ldg(r1 + (int64_t)i1 * kBins16 + v);
        float res = rintf(opencv_blend(l11, l12, l21, l22, xa, xa1, ya, ya1));
        res = fminf(fmaxf(res, 0.0f), 65535.0f);
        drow[x] = (uint16_t)(int)res;
    }
}

static Lut16Params make_lut16_params(const ClaheGeom& g, double clip_limit) {
    Lut16Params p;
    const int area = g.th * g.tw;
    p.clip = 0;
    if (clip_limit > 0.0) {
        const double q = clip_limit * (double)area / (double)kBins16;
        const int c = q > 2147483647.0 ? 2147483647 : (int)q;
        p.clip = c < 1 ? 1 : c;
    }
    p.lut_scale = (float)(kBins16 - 1) / (float)area;
    return p;
}

int clahe16_luts_impl(const void* src, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int gh, int gw,
                      double clip_limit, uint16_t* luts, cudaStream_t st, uint32_t* vmax = nullptr) {
    if (n < 0 || h <= 0 || w <= 0) return MIE_E_SHAPE;
    if (n > 0 && (!src || !luts)) return MIE_E_NULL;
    if (!plane_strides_ok({src, MIE_U16, ssn, ssh}, n, h, w)) return MIE_E_STRIDE;
    ClaheGeom g;
    int rc = make_clahe_geom(h, w, gh, gw, MIE_CLAHE_OPENCV, &g);
    if (rc) return rc;
    if ((int64_t)g.th * g.tw > 2147483647LL / 2) return MIE_E_SHAPE;
    const int64_t tiles = n * gh * gw;
    if (tiles == 0) return MIE_OK;
    if (tiles > 2147483647LL) return MIE_E_SHAPE;
    const size_t smem = (size_t)(kHalf16 + kHalf16 / 32) * sizeof(int);
    const bool no_small = kernel_policy(MIE_POLICY_CLAHE16_TWO_SWEEP);
    const bool no_cluster = kernel_policy(MIE_POLICY_CLAHE16_NO_CLUSTER);
    if ((int64_t)g.th * g.tw < 65536 && !no_small && !no_cluster && tiles <= 1073741823LL) {
        // counts fit 16 bits: single pass, one tile per cluster of two CTAs
        const size_t csmem = (size_t)(kHalf16 / 2 + kHalf16 / 64) * sizeof(int);
        MIE_ENSURE_SMEM(clahe16_lut_cluster_kernel, csmem);
        if (vmax) {   // bound the LUTs by the largest pixel value of the batch (mie_clahe; the stage API returns full LUTs)
            cudaError_t e = cudaMemsetAsync(vmax, 0, sizeof(uint32_t), st);
            if (e != cudaSuccess) return (int)e;
            const int64_t rows = n * h;
            clahe16_max_kernel<<<(unsigned)(rows / 8 < 1 ? 1 : (rows / 8 > 4 * 148 ? 4 * 148 : rows / 8)), 256, 0, st>>>(
                (const uint16_t*)src, ssn, ssh, n, h, w, vmax);
            int rcm = check_launch();
            if (rcm) return rcm;
        }
        clahe16_lut_cluster_kernel<<<(unsigned)(2 * tiles), kClThreads, csmem, st>>>((const uint16_t*)src, ssn, ssh, g,
                                                                                  make_lut16_params(g, clip_limit), luts, vmax);
        return check_launch();
    }
    if ((int64_t)g.th * g.tw < 65536 && !no_small) {   // counts fit 16 bits: single-pass kernel
        MIE_ENSURE_SMEM(clahe16_lut_small_kernel, smem);
        clahe16_lut_small_kernel<<<(unsigned)tiles, kThreads16, smem, st>>>((const uint16_t*)src, ssn, ssh, g,
                                                                         make_lut16_params(g, clip_limit), luts);
        return check_launch();
    }
    MIE_ENSURE_SMEM(clahe16_lut_kernel, smem);
    clahe16_lut_kernel<<<(unsigned)tiles, kThreads16, smem, st>>>((const uint16_t*)src, ssn, ssh, g,
                                                               make_lut16_params(g, clip_limit), luts);
    return check_launch();
}

int clahe16_apply_impl(const void* src, void* dst, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int64_t dsn,
                       int64_t dsh, int gh, int gw, const uint16_t* luts, cudaStream_t st) {
    ClaheGeom g;
    int rc = make_clahe_geom(h, w, gh, gw, MIE_CLAHE_OPENCV, &g);
    if (rc) return rc;
    if (n == 0) return MIE_OK;
    if (n > 65535) return MIE_E_SHAPE;
    dim3 grid(ceil_div(w, 256), ceil_div(h, 4), (unsigned)n);
    clahe16_apply_kernel<<<grid, 256, 0, st>>>((const uint16_t*)src, (uint16_t*)dst, ssn, ssh, dsn, dsh, g, luts);
    return check_launch();
}

// luts + apply for a batch, LUTs of at most `group` images alive at a time.
int clahe16_impl(const void* src, void* dst, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                 int gh, int gw, double clip_limit, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    if (h <= 0 || w <= 0 || n < 0) return MIE_E_SHAPE;   // validated BEFORE the grid enters a division below
    if (gh <= 0 || gw <= 0) return MIE_E_GRID;
    const size_t per_image = (size_t)gh * gw * kBins16 * sizeof(uint16_t);
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if (workspace_bytes < per_image) return MIE_E_WORKSPACE;
    int64_t group = (int64_t)(workspace_bytes / per_image);
    if (group > 65535) group = 65535;
    // 256 spare bytes behind the LUTs hold the batch's largest pixel value (see clahe16_lut_cluster_kernel)
    uint32_t* vmax = nullptr;
    // (a single slice is launch-latency bound: the two extra launches of the bound would cost what it saves)
    if (!kernel_policy(MIE_POLICY_CLAHE16_FULL_LUTS) && n * gh * gw >= 2 * 148) {
        if (workspace_bytes >= (size_t)group * per_image + 256) vmax = (uint32_t*)((char*)workspace + (size_t)group * per_image);
        else if (group > 1) { --group; vmax = (uint32_t*)((char*)workspace + (size_t)group * per_image); }
    }
    for (int64_t i0 = 0; i0 < n; i0 += group) {
        const int64_t m = (n - i0) < group ? (n - i0) : group;
        const uint16_t* s = (const uint16_t*)src + i0 * ssn;
        uint16_t* d = (uint16_t*)dst + i0 * dsn;
        int rc = clahe16_luts_impl(s, m, h, w, ssn, ssh, gh, gw, clip_limit, (uint16_t*)workspace, st, vmax);
        if (rc) return rc;
        rc = clahe16_apply_impl(s, d, m, h, w, ssn, ssh, dsn, dsh, gh, gw, (const uint16_t*)workspace, st);
        if (rc) return rc;
    }
    return MIE_OK;
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_clahe16_lut_bytes(int gh, int gw) {
    if (gh <= 0 || gw <= 0) return 0;
    return (size_t)gh * gw * kBins16 * sizeof(uint16_t);
}

int mie_clahe16_luts(const void* src, int64_t n, int h, int w, int64_t src_stride_n, int64_t src_stride_h, int gh,
                     int gw, double clip_limit, uint16_t* luts, void* stream) {
    return clahe16_luts_impl(src, n, h, w, src_stride_n, src_stride_h, gh, gw, clip_limit, luts, (cudaStream_t)stream);
}

}  // extern "C"
