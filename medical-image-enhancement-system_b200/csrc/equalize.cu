// equalize.cu — global histogram equalisation, one histogram per plane.
// Replaces kornia.enhance.equalize -> _scale_channel, the rule torchvision's
// equalize uses as well (reference pyproject.toml:8,16; SURVEY.md §8(a) A2,
// site-packages/torchvision/transforms/_functional_tensor.py:863-881):
//   v = x01 * 255; hist = histc(v, bins=256, min=0, max=255);
//   step = (sum(nonzero) - last_nonzero) // 255;
//   lut = [0, ((cumsum(hist) + step//2) // step)[:-1]] clamped to [0,255];
//   out = lut[trunc(v)] / 255, or v / 255 when step == 0.
// Default-range integer planes that fit the shared memory of one thread-block cluster run in ONE launch
// (equalize_fused_cluster_kernel: every pixel crosses HBM once in each direction); everything else takes three
// launches: per-plane histogram (shared-memory sub-histograms, one global atomic per non-empty bin per block),
// LUT (one block per plane), apply.

#include <cooperative_groups.h>
#include <type_traits>

#include "march.cuh"
#include "window.cuh"

namespace mie {

struct EqPlaneState {  // per plane, in the caller's workspace
    unsigned int hist[kBins];
    float lut[kBins];
    int step_nonzero;
    int pad[3];
};

__device__ __forceinline__ int eq_bin(float v) {  // torch.histc(v, 256, 0, 255); -1 = ignored
    if (!(v >= 0.0f && v <= 255.0f)) return -1;
    const int b = (int)__fmul_rn(div255(v), 256.0f);
    return b > 255 ? 255 : b;
}

template <typename SrcT>
__global__ void __launch_bounds__(256)
equalize_hist_kernel(const SrcT* __restrict__ src, int64_t ssn, int64_t ssh, int h, int w, int rows_per_block,
                     float lo, float rg, EqPlaneState* __restrict__ state) {
    __shared__ int s_hist[8 * kBins];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int i = 0; i < 8; ++i) s_hist[i * kBins + tid] = 0;
    __syncthreads();
    const int64_t n = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    const SrcT* plane = src + n * ssn;
    for (int y = y0 + warp; y < y1; y += 8) {
        const SrcT* row = plane + (int64_t)y * ssh;
        for (int x0 = 0; x0 < w; x0 += 32) {
            const int x = x0 + lane;
            int bin = -1;
            if (x < w) bin = eq_bin(__fmul_rn(Px<SrcT>::to01(row[x], lo, rg), 255.0f));
            hist_add(s_hist + warp * kBins, bin);
        }
    }
    __syncthreads();
    int hv = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) hv += s_hist[i * kBins + tid];
    if (hv) atomicAdd(&state[n].hist[tid], (unsigned int)hv);
}

__global__ void __launch_bounds__(256) equalize_lut_kernel(EqPlaneState* __restrict__ state) {
    __shared__ int s_red[8];
    __shared__ int s_last;
    EqPlaneState& st = state[blockIdx.x];
    const int b = threadIdx.x;
    const int hv = (int)st.hist[b];
    const int total = block_sum_256(hv, s_red);
    // index of the last non-empty bin
    int cand = hv ? b : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand = max(cand, __shfl_xor_sync(0xffffffffu, cand, o));
    __syncthreads();
    if ((b & 31) == 0) s_red[b >> 5] = cand;
    __syncthreads();
    if (b == 0) {
        int m = -1;
        for (int i = 0; i < 8; ++i) m = max(m, s_red[i]);
        s_last = m;
    }
    __syncthreads();
    const int last = s_last >= 0 ? (int)st.hist[s_last] : 0;
    const int step = (total - last) / 255;
    const int cum = block_scan_256(hv, s_red);  // inclusive
    if (step > 0) {
        // lut[b+1] = (cum[b] + step/2) / step, lut[0] = 0
        const long long q = ((long long)cum + step / 2) / step;
        if (b < 255) st.lut[b + 1] = (float)(q > 255 ? 255 : q);
        if (b == 0) st.lut[0] = 0.0f;
    }
    if (b == 0) st.step_nonzero = step > 0 ? 1 : 0;
}

template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256)
equalize_apply_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                      int64_t dsh, int h, int w, float lo, float rg, const EqPlaneState* __restrict__ state) {
    __shared__ float s_lut[kBins];
    const int64_t n = blockIdx.z;
    const EqPlaneState& st = state[n];
    s_lut[threadIdx.x] = st.lut[threadIdx.x];
    const int active = st.step_nonzero;
    __syncthreads();
    const int x = blockIdx.x * 64 + (threadIdx.x & 63);
    const int y = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (x >= w || y >= h) return;
    const float v = __fmul_rn(Px<SrcT>::to01(src[n * ssn + (int64_t)y * ssh + x], lo, rg), 255.0f);
    float r = v;
    if (active) {
        const float c = fminf(fmaxf(v, 0.0f), 255.0f);
        r = s_lut[__float2int_rz(c)];
    }
    dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(div255(r), lo, rg);
}


// ---------------------------------------------------------------- tuned path: integer pixels, default range
// Same integers (histogram, LUT) and the same fp32 mapping as the kernels above, but 128-bit loads /
// stores, the divide-free pixel conversion of chain_fast.cuh, one ATOMS.POPC.INC per pixel into a single
// block histogram, and — because lut[trunc(v)] takes only 256 values — a per-block table of the 256
// possible OUTPUT codes, so a pixel costs one conversion, one shared-memory lookup and a pack.
template <typename SrcT, bool WIN, bool IDX>
__global__ void __launch_bounds__(256)
equalize_hist_fast_kernel(const SrcT* __restrict__ src, int64_t ssn, int64_t ssh, int h, int w, int rows_per_block,
                          EqPlaneState* __restrict__ state, WinCvt cv) {
    __shared__ __align__(16) int s_hist[kBins + 8];
    const int tid = threadIdx.x;
    for (int i = tid; i < kBins + 8; i += 256) s_hist[i] = 0;
    __syncthreads();
    const int64_t n = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    const SrcT* base = src + n * ssn + (int64_t)y0 * ssh;
    const uint32_t h32 = hist_base32(s_hist);
    const int chunks = w >> 3, total = chunks * (y1 - y0);
    for (int i = tid; i < total; i += 256) {
        const int r = i / chunks, c = i - r * chunks;
        if constexpr (IDX) {   // default-range integers: eq_bin is an integer function of the code (window.cuh)
            uint32_t u[8];
            Codes<SrcT>::load8(base + (int64_t)r * ssh + 8 * c, u);
#pragma unroll
            for (int k = 0; k < 8; ++k) hist_add_nobranch(s_hist, (int)Codes<SrcT>::bin(u[k]));
        } else {
            float x[8];
            PixIO<SrcT, WIN>::load8(base + (int64_t)r * ssh + 8 * c, x, cv);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (WIN) hist_add(s_hist, eq_bin(__fmul_rn(x[k], 255.0f)));               // pixels outside the window: ignored
                else hist_add_le1(h32, div255(__fmul_rn(x[k], 255.0f)));                  // eq_bin, x in [0,1]
            }
        }
    }
    __syncthreads();
    int hv = s_hist[tid];
    if (tid == kBins - 1) hv += s_hist[kBins];   // slot 256 = pixels equal to 1.0 (see hist_add_le1)
    if (hv) atomicAdd(&state[n].hist[tid], (unsigned int)hv);
}

__device__ __forceinline__ void eq_store8(uint16_t* p, const uint16_t* s_out, const uint32_t* i) {
    uint4 o;
    o.x = (uint32_t)s_out[i[0]] | ((uint32_t)s_out[i[1]] << 16);
    o.y = (uint32_t)s_out[i[2]] | ((uint32_t)s_out[i[3]] << 16);
    o.z = (uint32_t)s_out[i[4]] | ((uint32_t)s_out[i[5]] << 16);
    o.w = (uint32_t)s_out[i[6]] | ((uint32_t)s_out[i[7]] << 16);
    __stcs(reinterpret_cast<uint4*>(p), o);   // streaming store: the output should not push the input out of L2
}
__device__ __forceinline__ void eq_store8(int16_t* p, const int16_t* s_out, const uint32_t* i) {
    eq_store8(reinterpret_cast<uint16_t*>(p), reinterpret_cast<const uint16_t*>(s_out), i);
}
__device__ __forceinline__ void eq_store8(uint8_t* p, const uint8_t* s_out, const uint32_t* i) {
    uint2 o;
    o.x = (uint32_t)s_out[i[0]] | ((uint32_t)s_out[i[1]] << 8) | ((uint32_t)s_out[i[2]] << 16) | ((uint32_t)s_out[i[3]] << 24);
    o.y = (uint32_t)s_out[i[4]] | ((uint32_t)s_out[i[5]] << 8) | ((uint32_t)s_out[i[6]] << 16) | ((uint32_t)s_out[i[7]] << 24);
    *reinterpret_cast<uint2*>(p) = o;
}
__device__ __forceinline__ void eq_store8(float* p, const float* s_out, const uint32_t* i) {
    *reinterpret_cast<float4*>(p) = make_float4(s_out[i[0]], s_out[i[1]], s_out[i[2]], s_out[i[3]]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(s_out[i[4]], s_out[i[5]], s_out[i[6]], s_out[i[7]]);
}

template <typename SrcT, typename DstT, bool WIN, bool IDX>
__global__ void __launch_bounds__(256)
equalize_apply_fast_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh,
                           int64_t dsn, int64_t dsh, int h, int w, int rows_per_block, float lo, float rg,
                           const EqPlaneState* __restrict__ state, WinCvt cv) {
    __shared__ __align__(16) DstT s_out[kBins];
    const int tid = threadIdx.x;
    const int64_t n = blockIdx.y;
    const EqPlaneState& st = state[n];
    const int active = st.step_nonzero;
    s_out[tid] = Px<DstT>::from01(div255(st.lut[tid]), lo, rg);
    __syncthreads();
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    const SrcT* sp = src + n * ssn + (int64_t)y0 * ssh;
    DstT* dp = dst + n * dsn + (int64_t)y0 * dsh;
    const int chunks = w >> 3, total = chunks * (y1 - y0);
    if (active) {
#pragma unroll 2
        for (int i = tid; i < total; i += 256) {
            const int r = i / chunks, c = i - r * chunks;
            uint32_t idx[8];
            if constexpr (IDX) {
                Codes<SrcT>::load8(sp + (int64_t)r * ssh + 8 * c, idx);
#pragma unroll
                for (int k = 0; k < 8; ++k) idx[k] = Codes<SrcT>::index(idx[k]);
            } else {
                float x[8];
                PixIO<SrcT, WIN>::load8(sp + (int64_t)r * ssh + 8 * c, x, cv);
#pragma unroll
                for (int k = 0; k < 8; ++k)   // trunc(clamp(x*255, 0, 255))
                    idx[k] = (WIN ? fast_idx_bits<false>(x[k]) : fast_idx_bits_le1(x[k])) & 0xFFu;
            }
            eq_store8(dp + (int64_t)r * dsh + 8 * c, s_out, idx);
        }
    } else {   // step == 0 (e.g. a constant plane): v/255 goes back unchanged
        for (int i = tid; i < total; i += 256) {
            const int r = i / chunks, c = i - r * chunks;
            float x[8];
            PixIO<SrcT, WIN>::load8(sp + (int64_t)r * ssh + 8 * c, x, cv);
            DstT* o = dp + (int64_t)r * dsh + 8 * c;
#pragma unroll
            for (int k = 0; k < 8; ++k) o[k] = Px<DstT>::from01(div255(__fmul_rn(x[k], 255.0f)), lo, rg);
        }
    }
}

// ---------------------------------------------------------------- fused path: one thread-block cluster per plane
// The three-launch path reads every pixel twice (histogram pass, apply pass): 6 B/pixel of HBM traffic for 4
// algorithmic bytes.  Here a cluster of 1 / 2 / 4 / 8 CTAs owns one plane: CTA r pulls its slab of rows into shared
// memory with bulk copies (TMA, four mbarrier stages so that counting starts when the first quarter has landed),
// counts it, adds its 256 counts to every CTA's total through distributed shared memory (remote shared atomics, one
// cluster barrier), every CTA derives the plane's LUT (256 threads = 256 bins, the arithmetic of equalize_lut_kernel) and maps its
// slab out of shared memory — so a pixel is read from HBM once and written once.  Slabs of at most 72 KB keep three
// CTAs on an SM: one loads while another counts or stores.  SLAB = false (small planes, contiguous rows): no slab and
// no bulk copies — both passes read global memory, the second one out of L2 (see launch_equalize_fused).
template <typename T> struct SlabCodes;   // 8 pixel codes (v - dtype_min) from shared memory
template <> struct SlabCodes<uint16_t> {
    static __device__ __forceinline__ void load8(const uint16_t* p, uint32_t* u) {
        const uint4 b = *reinterpret_cast<const uint4*>(p);
        u[0] = b.x & 0xFFFFu; u[1] = b.x >> 16; u[2] = b.y & 0xFFFFu; u[3] = b.y >> 16;
        u[4] = b.z & 0xFFFFu; u[5] = b.z >> 16; u[6] = b.w & 0xFFFFu; u[7] = b.w >> 16;
    }
};
template <> struct SlabCodes<int16_t> {
    static __device__ __forceinline__ void load8(const int16_t* p, uint32_t* u) {
        uint4 b = *reinterpret_cast<const uint4*>(p);
        b.x ^= 0x80008000u; b.y ^= 0x80008000u; b.z ^= 0x80008000u; b.w ^= 0x80008000u;
        u[0] = b.x & 0xFFFFu; u[1] = b.x >> 16; u[2] = b.y & 0xFFFFu; u[3] = b.y >> 16;
        u[4] = b.z & 0xFFFFu; u[5] = b.z >> 16; u[6] = b.w & 0xFFFFu; u[7] = b.w >> 16;
    }
};
template <> struct SlabCodes<uint8_t> {
    static __device__ __forceinline__ void load8(const uint8_t* p, uint32_t* u) {
        const uint2 b = *reinterpret_cast<const uint2*>(p);
        u[0] = b.x & 0xFFu; u[1] = (b.x >> 8) & 0xFFu; u[2] = (b.x >> 16) & 0xFFu; u[3] = b.x >> 24;
        u[4] = b.y & 0xFFu; u[5] = (b.y >> 8) & 0xFFu; u[6] = (b.y >> 16) & 0xFFu; u[7] = b.y >> 24;
    }
};
template <> struct SlabCodes<float> {   // never launched; keeps the dispatch macros compiling
    static __device__ __forceinline__ void load8(const float*, uint32_t* u) { for (int k = 0; k < 8; ++k) u[k] = 0; }
};

constexpr int kEqStages = 4;

template <typename SrcT, typename DstT, bool SLAB = true>
__global__ void __launch_bounds__(256)
equalize_fused_cluster_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh,
                              int64_t dsn, int64_t dsh, int h, int w, int rows_per_cta, float lo, float rg) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(128) unsigned char s_slab_raw[];
    __shared__ __align__(16) int s_hist[kBins];
    __shared__ __align__(16) int s_total[kBins];
    __shared__ __align__(16) DstT s_out[kBins];
    __shared__ float s_lut[kBins];
    __shared__ int s_red[8];
    __shared__ int s_last;
    __shared__ __align__(8) unsigned long long s_bar[kEqStages];
    SrcT* slab = reinterpret_cast<SrcT*>(s_slab_raw);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned cs = cluster.num_blocks(), rank = cluster.block_rank();
    const int64_t n = blockIdx.x / cs;
    const int y0 = min((int)rank * rows_per_cta, h), rows = min(y0 + rows_per_cta, h) - y0;
    const int rows_per_stage = (rows + kEqStages - 1) / kEqStages;
    const uint32_t row_bytes = (uint32_t)w * (uint32_t)sizeof(SrcT);
    const uint32_t bar32 = (uint32_t)__cvta_generic_to_shared(s_bar);

    s_hist[tid] = 0;
    s_total[tid] = 0;
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kEqStages; ++s) mbar_init(bar32 + 8 * s, 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    cluster.barrier_arrive();   // "my s_total is zero": the matching wait stands in front of the remote adds below
    const SrcT* gsrc = src + n * ssn + (int64_t)y0 * ssh;   // !SLAB: contiguous rows (ssh == w), second read through L2
    auto ld8 = [&](size_t g, uint32_t* u) {
        if constexpr (SLAB) SlabCodes<SrcT>::load8(slab + 8 * g, u);
        else Codes<SrcT>::load8(gsrc + 8 * g, u);
    };
    // second read of the no-slab variant: last use of the line (ld.global.cs = evict-first), 16-bit pixels; together with
    // the streaming stores 0.0617 -> 0.0599 ms (ncu before: 221 MB read from DRAM for 134 MB of pixels)
    auto ld8_last = [&](size_t g, uint32_t* u) {
        if constexpr (!SLAB && sizeof(SrcT) == 2) {
            uint4 b = __ldcs(reinterpret_cast<const uint4*>(gsrc + 8 * g));
            if (std::is_signed<SrcT>::value) { b.x ^= 0x80008000u; b.y ^= 0x80008000u; b.z ^= 0x80008000u; b.w ^= 0x80008000u; }
            u[0] = b.x & 0xFFFFu; u[1] = b.x >> 16; u[2] = b.y & 0xFFFFu; u[3] = b.y >> 16;
            u[4] = b.z & 0xFFFFu; u[5] = b.z >> 16; u[6] = b.w & 0xFFFFu; u[7] = b.w >> 16;
            return;
        }
        ld8(g, u);
    };
    if (SLAB && warp == 0) {   // producer warp: one arrival (with the stage's byte count) per stage, then one copy per row
        if (lane < kEqStages) {
            const int r0 = min(lane * rows_per_stage, rows), r1 = min(r0 + rows_per_stage, rows);
            mbar_expect_tx(bar32 + 8 * lane, (uint32_t)(r1 - r0) * row_bytes);
        }
        __syncwarp();
        const char* plane = reinterpret_cast<const char*>(src + n * ssn + (int64_t)y0 * ssh);
        const uint32_t slab32 = (uint32_t)__cvta_generic_to_shared(slab);
        for (int r = lane; r < rows; r += 32)
            bulk_g2s(slab32 + (uint32_t)r * row_bytes, plane + (int64_t)r * ssh * (int64_t)sizeof(SrcT), row_bytes,
                     bar32 + 8 * (r / rows_per_stage));
    }

    // ---- count: the slab is one contiguous run of 8-pixel groups; four groups per thread and step
    const int groups = w >> 3;
    for (int s = 0; s < kEqStages; ++s) {
        const int r0 = min(s * rows_per_stage, rows), r1 = min(r0 + rows_per_stage, rows);
        if (SLAB && r0 < r1) mbar_wait(bar32 + 8 * s, 0u);
        const int g1 = r1 * groups;
        int g = r0 * groups + tid;
        for (; g + 3 * 256 < g1; g += 4 * 256) {
            uint32_t u[4][8];
#pragma unroll
            for (int j = 0; j < 4; ++j) ld8((size_t)(g + j * 256), u[j]);
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 8; ++k) hist_add_nobranch(s_hist, (int)Codes<SrcT>::bin(u[j][k]));
        }
        for (; g < g1; g += 256) {
            uint32_t u[8];
            ld8((size_t)g, u);
#pragma unroll
            for (int k = 0; k < 8; ++k) hist_add_nobranch(s_hist, (int)Codes<SrcT>::bin(u[k]));
        }
    }
    // ---- the plane's histogram: every CTA adds its 256 counts to every CTA's s_total through distributed shared
    //      memory; one cluster barrier later all of them hold the plane's histogram and nobody touches a peer again
    __syncthreads();
    cluster.barrier_wait();
    {
        const int mine = s_hist[tid];
        if (mine)
            for (unsigned r = 0; r < cs; ++r) atomicAdd(cluster.map_shared_rank(&s_total[tid], r), mine);
    }
    cluster.sync();
    const int hv = s_total[tid];

    // ---- LUT (equalize_lut_kernel, every CTA for itself)
    const int total = block_sum_256(hv, s_red);
    int cand = hv ? tid : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand = max(cand, __shfl_xor_sync(0xffffffffu, cand, o));
    __syncthreads();
    if (lane == 0) s_red[warp] = cand;
    __syncthreads();
    if (tid == 0) {
        int m = -1;
        for (int i = 0; i < 8; ++i) m = max(m, s_red[i]);
        s_last = m;
    }
    __syncthreads();
    const int last = s_last >= 0 ? s_total[s_last] : 0;
    const int step = (total - last) / 255;
    const int cum = block_scan_256(hv, s_red);
    if (step > 0) {
        const unsigned q = ((unsigned)cum + (unsigned)(step / 2)) / (unsigned)step;   // cum < 2^31 (h * w < 2^31)
        if (tid < 255) s_lut[tid + 1] = (float)(q > 255u ? 255u : q);
        if (tid == 0) s_lut[0] = 0.0f;
    }
    __syncthreads();
    if (step > 0) s_out[tid] = Px<DstT>::from01(div255(s_lut[tid]), lo, rg);
    __syncthreads();

    // ---- map the slab
    DstT* dp = dst + n * dsn + (int64_t)y0 * dsh;
    if (step > 0 && dsh == w) {   // contiguous output rows: the slab maps group by group
        const int g1 = rows * groups;
#pragma unroll 4
        for (int g = tid; g < g1; g += 256) {
            uint32_t idx[8];
            ld8_last((size_t)g, idx);
#pragma unroll
            for (int k = 0; k < 8; ++k) idx[k] = Codes<SrcT>::index(idx[k]);
            eq_store8(dp + 8 * (size_t)g, s_out, idx);
        }
    } else if (step > 0) {
        for (int r = warp; r < rows; r += 8) {
            const SrcT* row = SLAB ? slab + (size_t)r * w : gsrc + (size_t)r * ssh;
            DstT* orow = dp + (int64_t)r * dsh;
#pragma unroll 2
            for (int c = lane; c < groups; c += 32) {
                uint32_t idx[8];
                SlabCodes<SrcT>::load8(row + 8 * c, idx);
#pragma unroll
                for (int k = 0; k < 8; ++k) idx[k] = Codes<SrcT>::index(idx[k]);
                eq_store8(orow + 8 * c, s_out, idx);
            }
        }
    } else {   // step == 0 (e.g. a constant plane): v/255 goes back unchanged
        for (int r = warp; r < rows; r += 8)
            for (int x = lane; x < w; x += 32)
                dp[(int64_t)r * dsh + x] =
                    Px<DstT>::from01(div255(__fmul_rn(Px<SrcT>::to01(SLAB ? slab[(size_t)r * w + x] : gsrc[(size_t)r * ssh + x], lo, rg), 255.0f)), lo, rg);
    }
}

// Cluster size and rows per CTA of the fused kernel, or 0 when the plane does not fit: the smallest cluster whose
// slabs stay under 72 KB (three CTAs per SM), else eight CTAs with slabs of up to 200 KB (one CTA per SM).
static int equalize_fused_plan(int h, int w, int esz, int* rows_per_cta) {
    // (clusters of 16 CTAs with 32 KB slabs were measured slower on the config-2 batch: 0.076 ms against 0.068 ms)
    for (int cs = 1; cs <= 8; cs *= 2) {
        const int rows = ceil_div(h, cs);
        if ((size_t)rows * w * esz <= 72 * 1024) { *rows_per_cta = rows; return cs; }
    }
    const int rows = ceil_div(h, 8);
    if ((size_t)rows * w * esz <= 200 * 1024) { *rows_per_cta = rows; return 8; }
    return 0;
}

template <typename SrcT, typename DstT>
static int launch_equalize_fused(const Image& s, const Image& d, int64_t n, int h, int w, float lo, float rg, int cs,
                                 int rows, cudaStream_t st) {
    const size_t smem = (size_t)rows * w * sizeof(SrcT);
    // Small planes (148 of them, one per resident cluster, stay L2-resident): no slab at all — the mapping pass reads the
    // pixels a second time through L2, nothing limits the occupancy (8 CTAs per SM instead of 3), and CTAs in different
    // phases hide each other's latencies: 0.0617 ms against 0.0688 ms with slabs on the config-2 batch.
    const size_t plane_bytes = (size_t)h * w * sizeof(SrcT);
    if (s.sh == w && 148 * plane_bytes <= ((size_t)96 << 20) && !kernel_policy(MIE_POLICY_EQUALIZE_SLAB)) {
        int c8 = 8;
        while (c8 > 1 && ceil_div(h, c8) < 8) c8 >>= 1;
        cudaLaunchConfig_t c2 = {};
        c2.gridDim = dim3((unsigned)(n * c8));
        c2.blockDim = dim3(256);
        c2.dynamicSmemBytes = 0;
        c2.stream = st;
        cudaLaunchAttribute a2[1];
        a2[0].id = cudaLaunchAttributeClusterDimension;
        a2[0].val.clusterDim.x = (unsigned)c8; a2[0].val.clusterDim.y = 1; a2[0].val.clusterDim.z = 1;
        c2.attrs = a2; c2.numAttrs = 1;
        cudaError_t e2 = cudaLaunchKernelEx(&c2, equalize_fused_cluster_kernel<SrcT, DstT, false>, (const SrcT*)s.p, (DstT*)d.out(),
                                            s.sn, s.sh, d.sn, d.sh, h, w, ceil_div(h, c8), lo, rg);
        return e2 == cudaSuccess ? check_launch() : (int)e2;
    }
    MIE_ENSURE_SMEM((equalize_fused_cluster_kernel<SrcT, DstT>), 200 * 1024);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n * cs));
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cs;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, equalize_fused_cluster_kernel<SrcT, DstT>, (const SrcT*)s.p, (DstT*)d.out(),
                                       s.sn, s.sh, d.sn, d.sh, h, w, rows, lo, rg);
    return e == cudaSuccess ? check_launch() : (int)e;
}

// The range mode of window.cuh (0, or 1 with *cv filled in) when the tuned kernels cover the request, else -1.
static int equalize_fast_mode(const Image& s, const Image& d, int w, float lo, float hi, WinCvt* cv) {
    if (kernel_policy(MIE_POLICY_GENERIC_EQUALIZE) || (w & 7)) return -1;
    if (!s.aligned(8 * s.bytes()) || !d.aligned(d.dtype == MIE_F32 ? 16 : 8 * d.bytes())) return -1;
    return range_mode(s.dtype, lo, hi, cv);
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_equalize_workspace_bytes(int64_t n) { return n > 0 ? (size_t)n * sizeof(EqPlaneState) : 0; }

int mie_equalize(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                 int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h, float lo,
                 float hi, void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const Image s{src, src_dtype, src_stride_n, src_stride_h}, d{dst, dst_dtype, dst_stride_n, dst_stride_h};
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    rc = check_dtypes(src_dtype, dst_dtype, lo, hi);
    if (rc) return rc;
    if ((int64_t)h * w >= (1LL << 31)) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (n > 65535) return MIE_E_SHAPE;
    if (!workspace) return MIE_E_NULL;
    if (workspace_bytes < mie_equalize_workspace_bytes(n)) return MIE_E_WORKSPACE;
    EqPlaneState* state = (EqPlaneState*)workspace;
    const float rg = hi - lo;
    WinCvt cv = {};
    const int mode = equalize_fast_mode(s, d, w, lo, hi, &cv);
    if (mode >= 0) {
        // ~8 blocks per SM in flight; at least 8 rows per block so the 256 global atomics per block stay rare
        int bpp = (int)((8 * 148 + n - 1) / n);
        int rows = ceil_div(h, bpp < 1 ? 1 : bpp);
        if (rows < 8) rows = 8;
        if (rows > 64) rows = 64;
        dim3 grid((unsigned)ceil_div(h, rows), (unsigned)n);
        // float planes (kornia's native input) may hold values outside [0, 1] or NaN: they take the range-checked
        // code path of the windowed kernels (PixIO<float, true> is a plain load)
        const bool win = mode == 1 || src_dtype == MIE_F32;
        const bool no_int = kernel_policy(MIE_POLICY_EQUALIZE_FLOAT_RULES);
        const bool idx = !win && !no_int && int_rules_ok(src_dtype);
        // one launch, one HBM round trip, when the integer rules apply and a cluster's shared memory holds the plane
        // (bulk copies move whole rows: 16-byte granularity)
        int frows = 0;
        const int fcs = idx && !kernel_policy(MIE_POLICY_EQUALIZE_THREE_PASS) && ((int64_t)w * s.bytes()) % 16 == 0 &&
                                s.aligned(16)
                            ? equalize_fused_plan(h, w, s.bytes(), &frows)
                            : 0;
        if (fcs) {
            MIE_DISPATCH_SRC_DST(src_dtype, dst_dtype,
                                 return (launch_equalize_fused<SrcT, DstT>(s, d, n, h, w, lo, rg, fcs, frows, st)));
        }
        cudaError_t me = cudaMemsetAsync(state, 0, (size_t)n * sizeof(EqPlaneState), st);
        if (me != cudaSuccess) return (int)me;
#define MIE_EQ_HIST(T_)                                                                                            \
    if (win) equalize_hist_fast_kernel<T_, true, false><<<grid, 256, 0, st>>>((const T_*)src, src_stride_n, src_stride_h, h, w, rows, state, cv); \
    else if (idx) equalize_hist_fast_kernel<T_, false, true><<<grid, 256, 0, st>>>((const T_*)src, src_stride_n, src_stride_h, h, w, rows, state, cv); \
    else equalize_hist_fast_kernel<T_, false, false><<<grid, 256, 0, st>>>((const T_*)src, src_stride_n, src_stride_h, h, w, rows, state, cv)
        switch (src_dtype) {
            case MIE_U8: MIE_EQ_HIST(uint8_t); break;
            case MIE_U16: MIE_EQ_HIST(uint16_t); break;
            case MIE_I16: MIE_EQ_HIST(int16_t); break;
            default: MIE_EQ_HIST(float); break;
        }
#undef MIE_EQ_HIST
        rc = check_launch();
        if (rc) return rc;
        equalize_lut_kernel<<<(unsigned)n, 256, 0, st>>>(state);
        rc = check_launch();
        if (rc) return rc;
#define MIE_EQ_APPLY(WIN_, IDX_)                                                                            \
    equalize_apply_fast_kernel<SrcT, DstT, WIN_, IDX_><<<grid, 256, 0, st>>>((const SrcT*)src, (DstT*)dst, src_stride_n, \
                                                                            src_stride_h, dst_stride_n, dst_stride_h, \
                                                                            h, w, rows, lo, rg, state, cv)
        if (win) { MIE_DISPATCH_SRC_DST(src_dtype, dst_dtype, MIE_EQ_APPLY(true, false)); }
        else if (idx) { MIE_DISPATCH_SRC_DST(src_dtype, dst_dtype, MIE_EQ_APPLY(false, true)); }
        else { MIE_DISPATCH_SRC_DST(src_dtype, dst_dtype, MIE_EQ_APPLY(false, false)); }
#undef MIE_EQ_APPLY
        return check_launch();
    }
    cudaError_t me = cudaMemsetAsync(state, 0, (size_t)n * sizeof(EqPlaneState), st);
    if (me != cudaSuccess) return (int)me;
    // enough blocks per plane to fill the machine when n is small, few enough to keep global atomics rare
    int blocks_per_plane = (int)((4 * 148 + n - 1) / n);
    if (blocks_per_plane < 1) blocks_per_plane = 1;
    int rows_per_block = ceil_div(h, blocks_per_plane);
    if (rows_per_block < 8) rows_per_block = 8;
    dim3 hgrid((unsigned)ceil_div(h, rows_per_block), (unsigned)n);
    MIE_DISPATCH_SRC(src_dtype, (equalize_hist_kernel<SrcT><<<hgrid, 256, 0, st>>>(
                                    (const SrcT*)src, src_stride_n, src_stride_h, h, w, rows_per_block, lo, rg, state)));
    rc = check_launch();
    if (rc) return rc;
    equalize_lut_kernel<<<(unsigned)n, 256, 0, st>>>(state);
    rc = check_launch();
    if (rc) return rc;
    dim3 agrid((unsigned)ceil_div(w, 64), (unsigned)ceil_div(h, 4), (unsigned)n);
    MIE_DISPATCH_SRC_DST(src_dtype, dst_dtype, (equalize_apply_kernel<SrcT, DstT><<<agrid, 256, 0, st>>>(
                                                   (const SrcT*)src, (DstT*)dst, src_stride_n, src_stride_h,
                                                   dst_stride_n, dst_stride_h, h, w, lo, rg, state)));
    return check_launch();
}

}  // extern "C"
