// clahe_fast.cu — tuned standalone CLAHE (kornia semantics, 256 bins) for unpadded geometries: tile
// width a multiple of 8, 16-byte aligned rows, the dtype's default value range.  Same integer artefacts
// (histograms, LUTs) and the same fp32 blend, bit for bit, as clahe.cu; what changes:
//   * LUT kernel: one warp per tile, 128-bit loads, divide-free pixel mapping, one ATOMS.POPC.INC per
//     pixel into the warp's histogram (hardware aggregates colliding lanes), LUT built by the same warp;
//   * interpolation: the four neighbouring LUT entries of every interpolation cell are packed into one
//     8-byte table entry per grey level (chain_fast.cu: chain_pack_cells_kernel), a block stages the
//     (gw + 1) tables of one cell row in shared memory, and a pixel costs ONE shared-memory lookup;
//     threads own 4 consecutive columns (64-bit loads / stores), no divides, no F2I.

#include "window.cuh"

#include <type_traits>

namespace mie {

// ---------------------------------------------------------------- histogram -> LUT, one WARP per tile
// A 64x64-pixel tile is only 16 pixels per thread of a 256-thread block: the block prologue, two barriers
// and the single-warp LUT tail then cost more instructions than the histogram itself (ncu: 21 lane-
// instructions per pixel, 7.6 of them in the pixel loop).  So a warp owns a whole tile — 128 pixels per
// lane for 64x64 tiles — with its own 257-slot histogram, no block-level synchronisation at all, and
// builds the LUT as soon as its own tile is done while the other warps of the block keep counting.
template <typename SrcT, bool WIN, bool IDX>
__global__ void __launch_bounds__(256)
clahe_lut_fast_kernel(const SrcT* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, LutParams lp,
                      uint32_t* __restrict__ hist_out, uint8_t* __restrict__ lut_out, int64_t tiles, WinCvt cv) {
    constexpr bool INT = sizeof(SrcT) != 4 && !WIN;  // default-range integer pixels map into [0, 1]: no range tests
    __shared__ __align__(16) int s_all[8][kBins + 8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t tile = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
    if (tile >= tiles) return;               // warp-uniform; no block barriers below
    int* s_hist = s_all[warp];
    for (int i = lane; i < kBins + 8; i += 32) s_hist[i] = 0;
    __syncwarp();
    const int tx = (int)(tile % g.gw), ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const SrcT* base = src + n * ssn + (int64_t)ty * g.th * ssh + (int64_t)tx * g.tw;
    const uint32_t h32 = hist_base32(s_hist);
    const int chunks = g.tw >> 3;              // 8-pixel chunks per tile row
    auto count8 = [&](int r, int c) {
        if constexpr (IDX) {   // default-range integers: the bin is an integer function of the code (window.cuh)
            uint32_t u[8];
            Codes<SrcT>::load8(base + (int64_t)r * ssh + 8 * c, u);
#pragma unroll
            for (int k = 0; k < 8; ++k) hist_add_nobranch(s_hist, (int)Codes<SrcT>::bin(u[k]));
        } else {
            float x[8];
            PixIO<SrcT, WIN>::load8(base + (int64_t)r * ssh + 8 * c, x, cv);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (INT) hist_add_le1(h32, x[k]);
                else hist_add_nobranch(s_hist, fast_bin<false>(x[k]));
            }
        }
    };
    if (chunks <= 32 && (32 % chunks) == 0) {  // a warp covers 32 / chunks whole rows per step
        const int rstep = 32 / chunks, c = lane % chunks;
#pragma unroll 4
        for (int r = lane / chunks; r < g.th; r += rstep) count8(r, c);
    } else {
        const int total = chunks * g.th;
        for (int i = lane; i < total; i += 32) count8(i / chunks, i % chunks);
    }
    __syncwarp();
    if (hist_out) {
        for (int b = lane; b < kBins; b += 32) {
            int v = s_hist[b];
            if (INT && b == kBins - 1) v += s_hist[kBins];   // slot 256 = pixels equal to 1.0 (see hist_add_le1)
            hist_out[tile * kBins + b] = (uint32_t)v;
        }
    }
    if (lut_out) {
        if (INT) warp_build_lut<true>(s_hist, lp, lut_out + tile * kBins, lane);
        else warp_build_lut<false>(s_hist, lp, lut_out + tile * kBins, lane);
    }
}

// ---------------------------------------------------------------- histogram -> LUT, one BLOCK per tile
// Latency variant for small jobs (a single 512x512 slice has 64 tiles: one warp per tile would leave
// most of the machine idle): 256 threads share one tile histogram, warp 0 builds the LUT.
template <typename SrcT, bool WIN, bool IDX>
__global__ void __launch_bounds__(256)
clahe_lut_block_kernel(const SrcT* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, LutParams lp,
                       uint32_t* __restrict__ hist_out, uint8_t* __restrict__ lut_out, WinCvt cv) {
    constexpr bool INT = sizeof(SrcT) != 4 && !WIN;
    __shared__ __align__(16) int s_hist[kBins + 8];
    const int tid = threadIdx.x;
    for (int i = tid; i < kBins + 8; i += 256) s_hist[i] = 0;
    __syncthreads();
    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % g.gw), ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const SrcT* base = src + n * ssn + (int64_t)ty * g.th * ssh + (int64_t)tx * g.tw;
    const uint32_t h32 = hist_base32(s_hist);
    const int chunks = g.tw >> 3;
    const int total = chunks * g.th;
    for (int i = tid; i < total; i += 256) {
        const int r = i / chunks, c = i - r * chunks;
        if constexpr (IDX) {
            uint32_t u[8];
            Codes<SrcT>::load8(base + (int64_t)r * ssh + 8 * c, u);
#pragma unroll
            for (int k = 0; k < 8; ++k) hist_add_nobranch(s_hist, (int)Codes<SrcT>::bin(u[k]));
        } else {
            float x[8];
            PixIO<SrcT, WIN>::load8(base + (int64_t)r * ssh + 8 * c, x, cv);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                if (INT) hist_add_le1(h32, x[k]);
                else hist_add_nobranch(s_hist, fast_bin<false>(x[k]));
            }
        }
    }
    __syncthreads();
    if (hist_out && tid < kBins) {
        int v = s_hist[tid];
        if (INT && tid == kBins - 1) v += s_hist[kBins];
        hist_out[tile * kBins + tid] = (uint32_t)v;
    }
    if (lut_out && tid < 32) {
        if (INT) warp_build_lut<true>(s_hist, lp, lut_out + tile * kBins, tid);
        else warp_build_lut<false>(s_hist, lp, lut_out + tile * kBins, tid);
    }
}

// ---------------------------------------------------------------- interpolation pass
struct ApplyFastArgs {
    const void* src;
    void* dst;
    int64_t ssn, ssh, dsn, dsh;
    ClaheGeom g;
    int rows_per_block;   // divides th / 2
    int blocks_per_image;
    const uint8_t* luts;  // non-null: the block packs its row of cell tables itself (small jobs: one launch less)
};

__device__ __forceinline__ uint2 lds64_(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}

// weight of the upper / left tile at coordinate y of an axis with tile size T (kornia_axis); in the
// outer half-tiles both neighbours are the same tile and the value is irrelevant (t == b there)
__device__ __forceinline__ float axis_weight(int y, int T) {
    const int hh = T >> 1;
    int r = y - hh;
    r = r < 0 ? 0 : r % T;
    return __fdiv_rn((float)(T - 1 - r), (float)(T - 1));
}

// The four pixels of PixIO<DstT, false>::store4 (default range), stored one by one: same quantisation, no alignment.
template <typename DstT>
__device__ __forceinline__ void store4_scalar(DstT* p, const float* y) {
    if constexpr (sizeof(DstT) == 4) {
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = y[k];
    } else if constexpr (sizeof(DstT) == 2) {
        const uint32_t m = std::is_same<DstT, int16_t>::value ? 0x80008000u : 0u;   // as Fast<int16_t>::store4
        const uint32_t a = Fast<uint16_t>::quant2_u16x2(y[0], y[1]) ^ m, b = Fast<uint16_t>::quant2_u16x2(y[2], y[3]) ^ m;
        p[0] = (DstT)(a & 0xFFFFu); p[1] = (DstT)(a >> 16); p[2] = (DstT)(b & 0xFFFFu); p[3] = (DstT)(b >> 16);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = (uint8_t)Fast<uint8_t>::quant(y[k]);
    }
}

// VEC_ST: one 4-pixel vector store per row and thread (destination rows 4-pixel aligned); otherwise the same four
// pixels are stored one by one (a caller's destination crop at any element offset / row stride).
template <typename SrcT, typename DstT, bool WIN, bool IDX, bool VEC_ST = true>
__global__ void __launch_bounds__(1024)
clahe_apply_fast_kernel(ApplyFastArgs a, const uint2* __restrict__ cells, WinCvt cv) {
    constexpr bool INT = sizeof(SrcT) != 4 && !WIN;
    extern __shared__ __align__(16) uint2 s_tab[];   // (gw + 1) x 256 entries: one row of cells
    const ClaheGeom g = a.g;
    const int tid = threadIdx.x, T = blockDim.x;
    const int64_t n = blockIdx.x / a.blocks_per_image;
    const int y0 = (int)(blockIdx.x % a.blocks_per_image) * a.rows_per_block;
    const int cy = (y0 + (g.th >> 1)) / g.th;        // cell row of all rows of this block
    if (a.luts) {   // latency path: cell tables straight from the LUTs (same packing as chain_pack_cells_kernel)
        const int jt = max(cy - 1, 0), jb = min(cy, g.gh - 1);
        for (int gl = tid; gl < kBins; gl += T) {
            const uint8_t* top = a.luts + (n * g.gh + jt) * (int64_t)g.gw * kBins + gl;
            const uint8_t* bot = a.luts + (n * g.gh + jb) * (int64_t)g.gw * kBins + gl;
            int tl = __ldg(top), bl = __ldg(bot);
            for (int cx = 0; cx <= g.gw; ++cx) {
                const int ir = min(cx, g.gw - 1);
                const int tr = __ldg(top + ir * kBins), br = __ldg(bot + ir * kBins);
                s_tab[cx * kBins + gl] = make_uint2(cell_word(tl - tr, tr), cell_word(bl - br, br));
                tl = tr; bl = br;
            }
        }
    } else {
        const uint4* s = reinterpret_cast<const uint4*>(cells + (n * (g.gh + 1) + cy) * (int64_t)(g.gw + 1) * kBins);
        uint4* d = reinterpret_cast<uint4*>(s_tab);
        for (int i = tid; i < (g.gw + 1) * kBins / 2; i += T) d[i] = __ldg(s + i);
    }
    __shared__ float s_wy[32];                      // rows_per_block <= 32: one division per row and block
    for (int i = tid; i < a.rows_per_block; i += T) s_wy[i] = axis_weight(y0 + i, g.th);
    const int x0 = 4 * tid;
    const int cx = (x0 + (g.tw >> 1)) / g.tw;
    const uint32_t tb = (uint32_t)__cvta_generic_to_shared(s_tab + cx * kBins);
    float wxv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) wxv[k] = axis_weight(x0 + k, g.tw);
    const SrcT* sp = (const SrcT*)a.src + n * a.ssn + (int64_t)y0 * a.ssh + x0;
    DstT* dp = (DstT*)a.dst + n * a.dsn + (int64_t)y0 * a.dsh + x0;
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < a.rows_per_block; ++r, sp += a.ssh, dp += a.dsh) {   // running row pointers: no 64-bit multiplies
        float y[4];
        const float wyv = s_wy[r];
        if constexpr (IDX) {   // default-range integers: the lookup index is an integer function of the code
            uint32_t u[4];
            Codes<SrcT>::load4(sp, u);
            // two neighbouring pixels per packed instruction (same per-lane operations as clahe_px)
            const f32x2 wy2 = f2_pack(wyv, wyv);
            const f32x2 ya = clahe_px2(lds64_(tb + Codes<SrcT>::entry_offset(u[0])), lds64_(tb + Codes<SrcT>::entry_offset(u[1])),
                                       f2_pack(wxv[0], wxv[1]), wy2);
            const f32x2 yb = clahe_px2(lds64_(tb + Codes<SrcT>::entry_offset(u[2])), lds64_(tb + Codes<SrcT>::entry_offset(u[3])),
                                       f2_pack(wxv[2], wxv[3]), wy2);
            f2_unpack(ya, y[0], y[1]);
            f2_unpack(yb, y[2], y[3]);
        } else {
            float x[4];
            PixIO<SrcT, WIN>::load4(sp, x, cv);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t bits = INT ? fast_idx_bits_le1(x[k]) : fast_idx_bits<false>(x[k]);
                y[k] = clahe_px(lds64_(tb + (__byte_perm(bits, 0u, 0x4440) << 3)), wxv[k], wyv);
            }
        }
        if constexpr (VEC_ST) PixIO<DstT, WIN>::store4(dp, y, cv);
        else store4_scalar(dp, y);
    }
}

// ---------------------------------------------------------------- host side
static bool int_rules_disabled() {   // keep the float conversion of the input (cross-check of the integer bin rules)
    return kernel_policy(MIE_POLICY_CLAHE_FLOAT_RULES);
}
static bool fast_disabled() { return kernel_policy(MIE_POLICY_GENERIC_CLAHE); }

// The range mode of window.cuh (0, or 1 with *cv filled in) when the tuned LUT kernels cover the request, else -1.
int clahe_lut_fast_mode(const ClaheGeom& g, const Image& s, float lo, float hi, WinCvt* cv) {
    if (fast_disabled()) return -1;
    if (g.hp != g.h || g.wp != g.w || (g.tw & 7)) return -1;
    if (!s.aligned(16)) return -1;
    if (((int64_t)g.tw * s.bytes()) % 16) return -1;   // tile origins 16-byte aligned for load8
    return range_mode(s.dtype, lo, hi, cv);
}

int launch_clahe_lut_fast(const Image& s, int64_t n, const ClaheGeom& g, const LutParams& lp, uint32_t* hist,
                          uint8_t* luts, int mode, const WinCvt& cv, cudaStream_t st) {
    const int64_t tiles = n * g.gh * g.gw;
    if (tiles == 0) return MIE_OK;
    if (tiles > 2147483647LL) return MIE_E_SHAPE;
    const int sd = s.dtype;
    const int wpb = 8;
    const int64_t blocks = (tiles + wpb - 1) / wpb;
#define MIE_LUT_FAST(WIN_, IDX_)                                                                                  \
    if (tiles < 4 * 148) /* small job: spread every tile over a whole block */                                   \
        clahe_lut_block_kernel<SrcT, WIN_, IDX_><<<(unsigned)tiles, 256, 0, st>>>((const SrcT*)s.p, s.sn, s.sh, g, lp, \
                                                                               hist, luts, cv);                   \
    else                                                                                                          \
        clahe_lut_fast_kernel<SrcT, WIN_, IDX_><<<(unsigned)blocks, 32 * wpb, 0, st>>>((const SrcT*)s.p, s.sn, s.sh, g, \
                                                                                    lp, hist, luts, tiles, cv)
    if (mode == 1) { MIE_DISPATCH_SRC(sd, MIE_LUT_FAST(true, false)); }
    else if (sd != MIE_F32 && int_rules_ok(sd) && !int_rules_disabled()) { MIE_DISPATCH_SRC(sd, MIE_LUT_FAST(false, true)); }
    else { MIE_DISPATCH_SRC(sd, MIE_LUT_FAST(false, false)); }
#undef MIE_LUT_FAST
    return check_launch();
}

size_t clahe_cells_bytes(int64_t n, int gh, int gw) { return chain_cells_bytes(n, gh, gw); }

// As clahe_lut_fast_mode, for the tuned interpolation kernel.
int clahe_apply_fast_mode(const ClaheGeom& g, const Image& s, const Image& d, float lo, float hi, WinCvt* cv) {
    if (fast_disabled()) return -1;
    if (g.hp != g.h || g.wp != g.w || (g.tw & 7) || (g.w & 3) || g.w > 4096 || g.gw > 32) return -1;
    if (d.dtype != s.dtype && d.dtype != MIE_F32) return -1;
    if (!s.aligned(16) || !d.aligned(16)) return -1;
    return range_mode(s.dtype, lo, hi, cv);
}

// luts -> cell tables (in `cells`, clahe_cells_bytes) -> interpolation
int launch_clahe_apply_fast(const Image& s, const Image& d, int64_t n, const ClaheGeom& g, const uint8_t* luts,
                            void* cells, int mode, const WinCvt& cv, cudaStream_t st) {
    if (n == 0) return MIE_OK;
    const int sd = s.dtype, dd = d.dtype;
    // small jobs are launch-latency bound (a single 512x512 slice: ~4 us per launch): skip the packing launch
    const bool in_kernel_cells = n * (int64_t)g.gh * g.gw < 4 * 148;
    if (!in_kernel_cells) {
        int rc = launch_pack_cells(luts, cells, n, g.gh, g.gw, st);
        if (rc) return rc;
    }
    ApplyFastArgs a;
    a.luts = in_kernel_cells ? luts : nullptr;
    a.src = s.p; a.dst = d.out(); a.ssn = s.sn; a.ssh = s.sh; a.dsn = d.sn; a.dsh = d.sh; a.g = g;
    int rows = g.th / 2;                        // rows of a block stay inside one cell row
    for (int d = 32; d >= 1; --d)
        if ((g.th / 2) % d == 0) { rows = d; break; }
    if (in_kernel_cells) {
        // latency path (a single slice): 32 rows per block would leave 16 blocks walking 32 rows each on a 148-SM
        // machine; take the largest divisor that still gives ~120 blocks (below 4 rows the in-kernel table packing,
        // 18 entries per thread, outweighs the pixels)
        for (int d = rows; d >= 4; --d)
            if ((g.th / 2) % d == 0) { rows = d; if (n * (int64_t)(g.h / d) >= 120) break; }
    }
    a.rows_per_block = rows;
    a.blocks_per_image = g.h / rows;
    const int64_t blocks = n * a.blocks_per_image;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    const size_t smem = (size_t)(g.gw + 1) * kBins * 8;
#define MIE_APPLY_FAST(WIN_, IDX_)                                                                         \
    MIE_ENSURE_SMEM((clahe_apply_fast_kernel<SrcT, DstT, WIN_, IDX_>), 80 * 1024);                         \
    clahe_apply_fast_kernel<SrcT, DstT, WIN_, IDX_><<<(unsigned)blocks, g.w / 4, smem, st>>>(a, (const uint2*)cells, cv)
    if (mode == 1) { MIE_DISPATCH_SRC_DST(sd, dd, MIE_APPLY_FAST(true, false)); }
    else if (sd != MIE_F32 && int_rules_ok(sd) && !int_rules_disabled()) { MIE_DISPATCH_SRC_DST(sd, dd, MIE_APPLY_FAST(false, true)); }
    else { MIE_DISPATCH_SRC_DST(sd, dd, MIE_APPLY_FAST(false, false)); }
#undef MIE_APPLY_FAST
    return check_launch();
}

// Interpolation pass of the fused bilateral -> CLAHE chain: the source is the 1-byte lookup-index plane (the index IS
// the byte: Codes<uint8_t>), the destination any pixel dtype in its default range.
int launch_clahe_apply_index(const uint8_t* idx, const Image& d, int64_t n, const ClaheGeom& g, const uint8_t* luts,
                             void* cells, cudaStream_t st) {
    if (n == 0) return MIE_OK;
    int rc = launch_pack_cells(luts, cells, n, g.gh, g.gw, st);
    if (rc) return rc;
    ApplyFastArgs a;
    a.luts = nullptr;
    a.src = idx; a.dst = d.out(); a.ssn = (int64_t)g.h * g.w; a.ssh = g.w; a.dsn = d.sn; a.dsh = d.sh; a.g = g;
    int rows = g.th / 2;
    for (int d = 32; d >= 1; --d)
        if ((g.th / 2) % d == 0) { rows = d; break; }
    a.rows_per_block = rows;
    a.blocks_per_image = g.h / rows;
    const int64_t blocks = n * a.blocks_per_image;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    const size_t smem = (size_t)(g.gw + 1) * kBins * 8;
    const WinCvt cv = {};
    // the vector store needs 4-pixel aligned destination rows; any other legal layout takes scalar stores
    const bool vec = d.aligned(4 * d.bytes());
#define MIE_APPLY_IDX_V(D_, V_)                                                                            \
    MIE_ENSURE_SMEM((clahe_apply_fast_kernel<uint8_t, D_, false, true, V_>), 80 * 1024);                   \
    clahe_apply_fast_kernel<uint8_t, D_, false, true, V_><<<(unsigned)blocks, g.w / 4, smem, st>>>(a, (const uint2*)cells, cv)
#define MIE_APPLY_IDX(D_)                                                                                  \
    if (vec) { MIE_APPLY_IDX_V(D_, true); } else { MIE_APPLY_IDX_V(D_, false); }
    switch (d.dtype) {
        case MIE_U8: MIE_APPLY_IDX(uint8_t); break;
        case MIE_U16: MIE_APPLY_IDX(uint16_t); break;
        case MIE_I16: MIE_APPLY_IDX(int16_t); break;
        default: MIE_APPLY_IDX(float); break;
    }
#undef MIE_APPLY_IDX
#undef MIE_APPLY_IDX_V
    return check_launch();
}

}  // namespace mie
