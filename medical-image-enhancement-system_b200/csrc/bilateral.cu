// bilateral.cu — bilateral filter on single-channel planes.
// Replaces kornia.filters.bilateral_blur (reference pyproject.toml:8; SURVEY.md
// §8(a) A7, Appendix B2):  w = space[dy,dx] * exp(-0.5/sigma_color^2 * (v-c)^2),
// out = sum(w*v) / sum(w), full ky x kx window, padding by border_type.
//
// The colour weight is 2^t with t = c2 * d^2, c2 = fp32(-0.5 log2(e) / sigma_color^2), evaluated by
// mie_exp2n(): clamp, n = rint(t) by the 1.5 * 2^23 trick (no FRND / F2I), f = t - n, a degree-5
// polynomial for 2^f (max rel err 1.7e-7) and an exponent-field add — the same sequence as
// oracle/mie_oracle.c:mie_exp2n, so the result is reproducible bit for bit.  This op is FMA-pipe bound
// (81 taps x 14 FMA-pipe operations), not HBM bound (SURVEY.md §7 H5).

#include <cmath>

#include "chain_fast.cuh"
#include "window.cuh"

#define MIE_HAVE_BILATERAL 1

namespace mie {

constexpr int kBilMaxK = 15;

struct SpaceW {
    float w[kBilMaxK * kBilMaxK];
};

__device__ __forceinline__ float mie_exp2n(float t) {
    t = fmaxf(t, -125.0f);
    const float u = __fadd_rn(t, 12582912.0f);
    const float n = __fsub_rn(u, 12582912.0f);
    const float f = __fsub_rn(t, n);
    float p = 0.0013264685403555632f;
    p = __fmaf_rn(p, f, 0.009671504609286785f);
    p = __fmaf_rn(p, f, 0.05550733953714371f);
    p = __fmaf_rn(p, f, 0.24022242426872253f);
    p = __fmaf_rn(p, f, 0.6931470036506653f);
    p = __fmaf_rn(p, f, 1.0f);
    return __uint_as_float(__float_as_uint(p) + (__float_as_uint(u) << 23));
}

// 32x32 output tile per block, 4 pixels per thread (rows ly, ly+8, ly+16, ly+24).
template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256)
bilateral_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                 int64_t dsh, int h, int w, int tiles_x, int tiles_y, int ky, int kx, float coef, int border, float lo,
                 float rg, SpaceW sw) {
    extern __shared__ __align__(16) float smem[];
    constexpr int T = 32;
    const int ry = ky / 2, rx = kx / 2;
    const int ew = T + 2 * rx, eh = T + 2 * ry, pitch = ew | 1;
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * T, ty0 = (int)((tile / tiles_x) % tiles_y) * T;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    const SrcT* plane = src + n * ssn;
    for (int i = threadIdx.x; i < eh * ew; i += 256) {
        const int r = i / ew, c = i - r * ew;
        const int sy = border_index(ty0 - ry + r, h, border), sx = border_index(tx0 - rx + c, w, border);
        smem[r * pitch + c] = (sy < 0 || sx < 0) ? 0.0f : Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], lo, rg);
    }
    __syncthreads();
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    const int x = tx0 + lx;
    float ctr[4], num[4], den[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        ctr[k] = smem[(ly0 + 8 * k + ry) * pitch + lx + rx];
        num[k] = 0.0f; den[k] = 0.0f;
    }
    for (int dy = 0; dy < ky; ++dy) {
        for (int dx = 0; dx < kx; ++dx) {
            const float ws = sw.w[dy * kx + dx];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float v = smem[(ly0 + 8 * k + dy) * pitch + lx + dx];
                const float dv = __fsub_rn(v, ctr[k]);
                const float wgt = __fmul_rn(ws, mie_exp2n(__fmul_rn(coef, __fmul_rn(dv, dv))));
                num[k] = __fmaf_rn(wgt, v, num[k]);
                den[k] = __fadd_rn(den[k], wgt);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = ty0 + ly0 + 8 * k;
        if (y < h && x < w)
            dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(__fdiv_rn(num[k], den[k]), lo, rg);
    }
}

// ---------------------------------------------------------------- packed variant, compile-time window
// The generic kernel above is ISSUE bound (95 % of the issue slots busy, FMA pipe 70 %: ncu,
// profiles/r1_ncu_full_bilateral_generic.txt): 27 instructions per pixel-tap.  This variant processes the
// four pixels of a thread as two f32x2 pairs: every arithmetic step of the weight (difference, square,
// scale, the exp range reduction and polynomial, the spatial weight, both accumulations) is ONE packed
// instruction per pair — same per-lane IEEE rounding, so the result is bit-identical — and the window
// loops are unrolled at compile time.  Per pixel-tap: 6.5 packed + 1 scalar FMA-pipe instructions, 1 LDS,
// 1 FMNMX, 1 exponent-field add: ~10.5 issue slots instead of 27; the FMA pipe becomes the limiter.

struct ExpConsts {
    f32x2 magic, c5, c4, c3, c2, c1, one;
};
__device__ __forceinline__ ExpConsts exp_consts() {
    ExpConsts k;
    k.magic = f2_dup(12582912.0f);
    k.c5 = f2_dup(0.0013264685403555632f); k.c4 = f2_dup(0.009671504609286785f);
    k.c3 = f2_dup(0.05550733953714371f); k.c2 = f2_dup(0.24022242426872253f);
    k.c1 = f2_dup(0.6931470036506653f); k.one = f2_dup(1.0f);
    return k;
}
// ptxas (CUDA 12.9) contracts mul.rn.f32x2 + add.rn.f32x2 — also __fadd2_rn(__fmul2_rn(..)), also with
// -fmad=false, also when the product is written fma(a, b, -0) — into one FFMA2, i.e. one rounding instead
// of two, which the scalar __fmul_rn / __fadd_rn sequence of the oracle never does.  Here the packed product
// c2 * d^2 passes through the scalar clamp before the magic add, and the product that feeds den + w
// (ws * 2^t) is a SCALAR multiply on the halves, which are unpacked there anyway (exponent-field add).
//
// ws * mie_exp2n(t) on both halves of t = c2 * d^2.
__device__ __forceinline__ f32x2 weight_x2(f32x2 t, float ws, const ExpConsts& k) {
    float t0, t1;
    f2_unpack(t, t0, t1);
    t0 = fmaxf(t0, -125.0f);
    t1 = fmaxf(t1, -125.0f);
    t = f2_pack(t0, t1);
    const f32x2 u = f2_add(t, k.magic);
    const f32x2 n = f2_sub(u, k.magic);
    const f32x2 f = f2_sub(t, n);
    f32x2 p = f2_fma(k.c5, f, k.c4);
    p = f2_fma(p, f, k.c3);
    p = f2_fma(p, f, k.c2);
    p = f2_fma(p, f, k.c1);
    p = f2_fma(p, f, k.one);
    float p0, p1, u0, u1;
    f2_unpack(p, p0, p1);
    f2_unpack(u, u0, u1);
    const float e0 = __uint_as_float(__float_as_uint(p0) + (__float_as_uint(u0) << 23));
    const float e1 = __uint_as_float(__float_as_uint(p1) + (__float_as_uint(u1) << 23));
    return f2_pack(__fmul_rn(ws, e0), __fmul_rn(ws, e1));
}

struct SpaceW2 {   // spatial weights, row-major K x K
    float w[81];
};

// Stages the haloed tile and evaluates the window for the thread's four pixels (rows ly0 + 8 k, column lx):
// num[k] / den[k] is the filter output.  Shared by the pixel-output kernel and the index-plane kernel of the fused
// bilateral -> CLAHE chain.
template <typename SrcT, int K>
__device__ __forceinline__ void bilateral_packed_core(const SrcT* __restrict__ plane, int64_t ssh, int h, int w, int tx0,
                                                      int ty0, float coef, int border, float lo, float rg,
                                                      const SpaceW2& sw, float* smem, float* num, float* den) {
    constexpr int T = 32, R = K / 2, EW = T + 2 * R, EH = T + 2 * R, PITCH = EW | 1;
    for (int i = threadIdx.x; i < EH * EW; i += 256) {
        const int r = i / EW, c = i - r * EW;
        const int sy = border_index(ty0 - R + r, h, border), sx = border_index(tx0 - R + c, w, border);
        smem[r * PITCH + c] = (sy < 0 || sx < 0) ? 0.0f : Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], lo, rg);
    }
    __syncthreads();
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    const float* base = smem + ly0 * PITCH + lx;          // window origin of pixel (ly0, lx)
    const ExpConsts kc = exp_consts();
    const f32x2 coef2 = f2_dup(coef);
    // pairs: (rows ly0, ly0 + 8) and (rows ly0 + 16, ly0 + 24)
    const f32x2 ctrA = f2_pack(base[R * PITCH + R], base[(8 + R) * PITCH + R]);
    const f32x2 ctrB = f2_pack(base[(16 + R) * PITCH + R], base[(24 + R) * PITCH + R]);
    f32x2 numA = f2_dup(0.0f), denA = numA, numB = numA, denB = numA;
#pragma unroll
    for (int dy = 0; dy < K; ++dy) {
#pragma unroll
        for (int dx = 0; dx < K; ++dx) {
            const float ws = sw.w[dy * K + dx];
            const float* p = base + dy * PITCH + dx;
            const f32x2 vA = f2_pack(p[0], p[8 * PITCH]);
            const f32x2 vB = f2_pack(p[16 * PITCH], p[24 * PITCH]);
            const f32x2 dA = f2_sub(vA, ctrA), dB = f2_sub(vB, ctrB);
            const f32x2 wA = weight_x2(f2_mul(coef2, f2_mul(dA, dA)), ws, kc);
            const f32x2 wB = weight_x2(f2_mul(coef2, f2_mul(dB, dB)), ws, kc);
            numA = f2_fma(wA, vA, numA); denA = f2_add(denA, wA);
            numB = f2_fma(wB, vB, numB); denB = f2_add(denB, wB);
        }
    }
    f2_unpack(numA, num[0], num[1]); f2_unpack(numB, num[2], num[3]);
    f2_unpack(denA, den[0], den[1]); f2_unpack(denB, den[2], den[3]);
}

template <typename SrcT, typename DstT, int K>
__global__ void __launch_bounds__(256)
bilateral_packed_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                        int64_t dsh, int h, int w, int tiles_x, int tiles_y, float coef, int border, float lo,
                        float rg, SpaceW2 sw) {
    constexpr int T = 32, R = K / 2, EW = T + 2 * R, EH = T + 2 * R, PITCH = EW | 1;
    __shared__ float smem[EH * PITCH];
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * T, ty0 = (int)((tile / tiles_x) % tiles_y) * T;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    float num[4], den[4];
    bilateral_packed_core<SrcT, K>(src + n * ssn, ssh, h, w, tx0, ty0, coef, border, lo, rg, sw, smem, num, den);
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    const int x = tx0 + lx;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = ty0 + ly0 + 8 * k;
        if (y < h && x < w)
            dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(__fdiv_rn(num[k], den[k]), lo, rg);
    }
}

// Stage A of the fused bilateral -> CLAHE chain (BASELINE.json config 4): the filtered value b never leaves the SM — only
// its CLAHE lookup index trunc(clamp(b * 255)) (one byte per pixel) is written, while its histogram bin floor(b * 256)
// goes into a block histogram that is flushed with one global atomic per occupied bin.  Requires 32-pixel-aligned CLAHE
// tiles without padding (checked on the host), so that a block's 32 x 32 pixels lie in ONE tile.
template <typename SrcT, int K>
__global__ void __launch_bounds__(256)
bilateral_index_kernel(const SrcT* __restrict__ src, uint8_t* __restrict__ idx, uint32_t* __restrict__ hist, int64_t ssn,
                       int64_t ssh, ClaheGeom g, int tiles_x, int tiles_y, float coef, int border, float lo, float rg,
                       SpaceW2 sw) {
    constexpr int T = 32, R = K / 2, EW = T + 2 * R, EH = T + 2 * R, PITCH = EW | 1;
    __shared__ float smem[EH * PITCH];
    __shared__ int s_hist[kBins + 8];
    for (int i = threadIdx.x; i < kBins + 8; i += 256) s_hist[i] = 0;
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * T, ty0 = (int)((tile / tiles_x) % tiles_y) * T;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    float num[4], den[4];
    bilateral_packed_core<SrcT, K>(src + n * ssn, ssh, g.h, g.w, tx0, ty0, coef, border, lo, rg, sw, smem, num, den);
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    uint8_t* ip = idx + n * (int64_t)g.h * g.w + (int64_t)(ty0 + ly0) * g.w + tx0 + lx;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float b = __fdiv_rn(num[k], den[k]);
        ip[(int64_t)8 * k * g.w] = (uint8_t)(fast_idx_bits<false>(b) & 0xFFu);
        hist_add_nobranch(s_hist, fast_bin<false>(b));    // slot 256 swallows what torch.histc would ignore
    }
    __syncthreads();
    uint32_t* gh_ = hist + ((n * g.gh + ty0 / g.th) * (int64_t)g.gw + tx0 / g.tw) * kBins;
    const int v = s_hist[threadIdx.x];
    if (v) atomicAdd(gh_ + threadIdx.x, (uint32_t)v);
}

// ---------------------------------------------------------------- default mode: MUFU.EX2 colour weights
// (MIE_POLICY_BILATERAL_EXACT_EXP selects the reproducible kernels above.)  The colour weight is ONE MUFU.EX2
// (ex2.approx.ftz, max rel err 2^-22) of t = c2 d^2 + log2(ws) — `sw` holds log2 of the spatial weights — so a pixel-tap
// costs five FMA-pipe operations and one XU operation instead of fourteen FMA-pipe operations, and the XU pipe (16
// lanes per clock and SM) becomes the limiter.  The result is within rel 1e-6 of the exact-polynomial kernel — inside
// the north star's 1e-5 for floating-point filters — but not reproducible bit for bit on a CPU: that is what the exact
// mode is kept for.
//
// With the arithmetic that cheap the loads matter, so the tile is laid out for them: P[r][c] = (v(r, c), v(r + 1, c)) as
// one 64-bit word for EVERY r (each value is stored twice), and a thread owns a 2 x 2 block of pixels — two vertical
// pairs.  For a window row dy the ten words P[2 ty + dy][2 tx .. 2 tx + 9] are five conflict-free 16-byte loads and
// already ARE the packed (row, row + 1) operands of all nine taps of both columns: 0.14 loads per pixel-tap instead
// of 1, no register shuffling.  Per 8 x 4096^2 images: exact kernel 5.93 ms, MUFU on the exact kernel's row-strided
// layout 3.27 ms, this kernel 2.90 ms (XU floor: 2.35 ms).  Handing every fourth / fifth / sixth / eighth tap to the
// polynomial to unload the XU pipe was measured and does not pay (3.18 / 3.05 / 2.98 / 2.90 ms).
__device__ __forceinline__ float ex2_approx(float t) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(t));
    return y;
}

template <int K>
struct LeanGeom {
    static constexpr int T = 32, R = K / 2, EW = (T + 2 * R + 2) & ~1, EH = T + 2 * R;   // even pitch: 16-byte rows
    static constexpr int WORDS = (EH - 1) * EW;                                         // 64-bit words
};

// num[k] / den[k] for the thread's pixels (2 ty + (k & 1), 2 tx + (k >> 1)) of the 32 x 32 tile.
template <typename SrcT, int K>
__device__ __forceinline__ void bilateral_lean_core(const SrcT* __restrict__ plane, int64_t ssh, int h, int w, int tx0,
                                                    int ty0, float coef, int border, float lo, float rg,
                                                    const SpaceW2& lsw, float2* P, float* num, float* den) {
    using G = LeanGeom<K>;
    constexpr int R = G::R, EW = G::EW, EH = G::EH, CW = G::T + 2 * R;
    for (int i = threadIdx.x; i < EH * CW; i += 256) {
        const int r = i / CW, c = i - r * CW;
        const int sy = border_index(ty0 - R + r, h, border), sx = border_index(tx0 - R + c, w, border);
        const float v = (sy < 0 || sx < 0) ? 0.0f : Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], lo, rg);
        if (r < EH - 1) P[r * EW + c].x = v;
        if (r > 0) P[(r - 1) * EW + c].y = v;
    }
    __syncthreads();
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const float2* base = P + (2 * ty) * EW + 2 * tx;
    const f32x2 coef2 = f2_dup(coef);
    const ulonglong2 cw = *reinterpret_cast<const ulonglong2*>(base + R * EW + (R & ~1));
    const f32x2 ctrA = (R & 1) ? cw.y : cw.x;
    f32x2 ctrB;
    if (R & 1) ctrB = *reinterpret_cast<const unsigned long long*>(base + R * EW + R + 1);
    else ctrB = cw.y;
    f32x2 numA = f2_dup(0.0f), denA = numA, numB = numA, denB = numA;
#pragma unroll
    for (int dy = 0; dy < K; ++dy) {
        f32x2 win[K + 1];
#pragma unroll
        for (int q = 0; q < (K + 1) / 2; ++q) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(base + dy * EW + 2 * q);
            win[2 * q] = v.x; win[2 * q + 1] = v.y;
        }
#pragma unroll
        for (int dx = 0; dx < K; ++dx) {
            const f32x2 lws2 = f2_dup(lsw.w[dy * K + dx]);
            const f32x2 vA = win[dx], vB = win[dx + 1];
            const f32x2 dA = f2_sub(vA, ctrA), dB = f2_sub(vB, ctrB);
            const f32x2 tA = f2_fma(f2_mul(dA, coef2), dA, lws2), tB = f2_fma(f2_mul(dB, coef2), dB, lws2);
            float a0, a1, b0, b1;
            f2_unpack(tA, a0, a1);
            f2_unpack(tB, b0, b1);
            const f32x2 wA = f2_pack(ex2_approx(a0), ex2_approx(a1));
            const f32x2 wB = f2_pack(ex2_approx(b0), ex2_approx(b1));
            numA = f2_fma(wA, vA, numA); denA = f2_add(denA, wA);
            numB = f2_fma(wB, vB, numB); denB = f2_add(denB, wB);
        }
    }
    f2_unpack(numA, num[0], num[1]); f2_unpack(numB, num[2], num[3]);
    f2_unpack(denA, den[0], den[1]); f2_unpack(denB, den[2], den[3]);
}

template <typename SrcT, typename DstT, int K>
__global__ void __launch_bounds__(256)
bilateral_lean_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                      int64_t dsh, int h, int w, int tiles_x, int tiles_y, float coef, int border, float lo, float rg,
                      SpaceW2 lsw) {
    __shared__ __align__(16) float2 P[LeanGeom<K>::WORDS];
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * 32, ty0 = (int)((tile / tiles_x) % tiles_y) * 32;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    float num[4], den[4];
    bilateral_lean_core<SrcT, K>(src + n * ssn, ssh, h, w, tx0, ty0, coef, border, lo, rg, lsw, P, num, den);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = ty0 + 2 * ty + (k & 1), x = tx0 + 2 * tx + (k >> 1);
        if (y < h && x < w)
            dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(__fdiv_rn(num[k], den[k]), lo, rg);
    }
}

template <typename SrcT, int K>
__global__ void __launch_bounds__(256)
bilateral_lean_index_kernel(const SrcT* __restrict__ src, uint8_t* __restrict__ idx, uint32_t* __restrict__ hist,
                            int64_t ssn, int64_t ssh, ClaheGeom g, int tiles_x, int tiles_y, float coef, int border,
                            float lo, float rg, SpaceW2 lsw) {
    __shared__ __align__(16) float2 P[LeanGeom<K>::WORDS];
    __shared__ int s_hist[kBins + 8];
    for (int i = threadIdx.x; i < kBins + 8; i += 256) s_hist[i] = 0;
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * 32, ty0 = (int)((tile / tiles_x) % tiles_y) * 32;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    float num[4], den[4];
    bilateral_lean_core<SrcT, K>(src + n * ssn, ssh, g.h, g.w, tx0, ty0, coef, border, lo, rg, lsw, P, num, den);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    uint8_t* ip = idx + n * (int64_t)g.h * g.w + (int64_t)(ty0 + 2 * ty) * g.w + tx0 + 2 * tx;
    uint32_t b4[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float b = __fdiv_rn(num[k], den[k]);
        b4[k] = fast_idx_bits<false>(b) & 0xFFu;
        hist_add_nobranch(s_hist, fast_bin<false>(b));    // slot 256 swallows what torch.histc would ignore
    }
    // rows 2 ty and 2 ty + 1, two neighbouring columns each: one 16-bit store per row (tx0 and g.w are even)
    *reinterpret_cast<uint16_t*>(ip) = (uint16_t)(b4[0] | (b4[2] << 8));
    *reinterpret_cast<uint16_t*>(ip + g.w) = (uint16_t)(b4[1] | (b4[3] << 8));
    __syncthreads();
    uint32_t* gh_ = hist + ((n * g.gh + ty0 / g.th) * (int64_t)g.gw + tx0 / g.tw) * kBins;
    const int v = s_hist[threadIdx.x];
    if (v) atomicAdd(gh_ + threadIdx.x, (uint32_t)v);
}

// Tile histograms (global, uint32) -> LUT bytes: one warp per tile, the clip / redistribute / scan of chain_fast.cuh.
__global__ void __launch_bounds__(256)
hist_to_lut_kernel(const uint32_t* __restrict__ hist, uint8_t* __restrict__ luts, LutParams lp, int64_t tiles) {
    __shared__ __align__(16) int s_tot[8][kBins + 8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 8 + warp;
    if (t >= tiles) return;
    const uint4* src = reinterpret_cast<const uint4*>(hist + t * kBins);
    const uint4 a = __ldg(src + 2 * lane), b = __ldg(src + 2 * lane + 1);
    *reinterpret_cast<uint4*>(&s_tot[warp][8 * lane]) = a;
    *reinterpret_cast<uint4*>(&s_tot[warp][8 * lane + 4]) = b;
    __syncwarp();
    warp_build_lut<false>(s_tot[warp], lp, luts + t * kBins, lane);
}

// The approximate-exponential kernels need log2 of every spatial weight: all of them must be positive and normal.
static bool bilateral_approx_ok(const float* wspace, int k) {
    if (kernel_policy(MIE_POLICY_BILATERAL_EXACT_EXP)) return false;
    for (int i = 0; i < k * k; ++i)
        if (!(wspace[i] >= 1.1754944e-38f) || !(wspace[i] < 3.0e38f)) return false;
    return true;
}
static void fill_space_weights(SpaceW2& sw, const float* wspace, int k, bool approx) {
    for (int i = 0; i < 81; ++i) {
        if (i >= k * k) sw.w[i] = 0.f;
        else sw.w[i] = approx ? (float)std::log2((double)wspace[i]) : wspace[i];
    }
}

template <typename SrcT, typename DstT>
static int launch_bilateral_packed(int k, const void* src, void* dst, int64_t ssn, int64_t ssh, int64_t dsn,
                                   int64_t dsh, int h, int w, int tiles_x, int tiles_y, unsigned blocks, float coef,
                                   int border, float lo, float rg, const float* wspace, cudaStream_t st) {
    const bool approx = bilateral_approx_ok(wspace, k);
    SpaceW2 sw;
    fill_space_weights(sw, wspace, k, approx);
#define MIE_BIL(K_)                                                                                          \
    case K_:                                                                                                 \
        if (approx)                                                                                          \
            bilateral_lean_kernel<SrcT, DstT, K_><<<blocks, 256, 0, st>>>((const SrcT*)src, (DstT*)dst, ssn, ssh, dsn, \
                                                                          dsh, h, w, tiles_x, tiles_y, coef, border,   \
                                                                          lo, rg, sw);                       \
        else                                                                                                 \
            bilateral_packed_kernel<SrcT, DstT, K_><<<blocks, 256, 0, st>>>((const SrcT*)src, (DstT*)dst, ssn, ssh, dsn, \
                                                                            dsh, h, w, tiles_x, tiles_y, coef, border, \
                                                                            lo, rg, sw);                     \
        break;
    switch (k) {
        MIE_BIL(3) MIE_BIL(5) MIE_BIL(7) MIE_BIL(9)
        default: return -1;
    }
#undef MIE_BIL
    return check_launch();
}

int bilateral_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
                   int64_t dsn, int64_t dsh, const float* wspace, int ky, int kx, float sigma_color, int border,
                   float lo, float hi, cudaStream_t st) {
    int rc = check_planes({src, sd, ssn, ssh}, {dst, dd, dsn, dsh}, n, h, w);
    if (rc) return rc;
    rc = check_dtypes(sd, dd, lo, hi);
    if (rc) return rc;
    if (!wspace) return MIE_E_NULL;
    if (ky <= 0 || kx <= 0 || !(ky & 1) || !(kx & 1) || ky > kBilMaxK || kx > kBilMaxK) return MIE_E_KERNEL;
    if (border < MIE_BORDER_CONSTANT || border > MIE_BORDER_CIRCULAR) return MIE_E_BORDER;
    if (border == MIE_BORDER_REFLECT && (kx / 2 >= w || ky / 2 >= h)) return MIE_E_BORDER;
    if (border == MIE_BORDER_CIRCULAR && (kx / 2 > w || ky / 2 > h)) return MIE_E_BORDER;
    if (!(sigma_color > 0.0f)) return MIE_E_RANGE;
    if (n == 0) return MIE_OK;
    SpaceW sw;
    for (int i = 0; i < kBilMaxK * kBilMaxK; ++i) sw.w[i] = i < ky * kx ? wspace[i] : 0.0f;
    const float coef = (float)(-0.5 * 1.4426950408889634 / ((double)sigma_color * (double)sigma_color));   // log2 domain
    const int tiles_x = ceil_div(w, 32), tiles_y = ceil_div(h, 32);
    const int64_t blocks = n * tiles_x * tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    const bool no_packed = kernel_policy(MIE_POLICY_GENERIC_BILATERAL);
    if (!no_packed && ky == kx && ky >= 3 && ky <= 9) {   // square 3 / 5 / 7 / 9 windows: packed, fully unrolled kernel
        MIE_DISPATCH_SRC_DST(sd, dd, return (launch_bilateral_packed<SrcT, DstT>(
                                         ky, src, dst, ssn, ssh, dsn, dsh, h, w, tiles_x, tiles_y, (unsigned)blocks,
                                         coef, border, lo, hi - lo, wspace, st)));
    }
    const int ew = 32 + 2 * (kx / 2), eh = 32 + 2 * (ky / 2);
    const size_t smem = (size_t)eh * (ew | 1) * 4;
    MIE_DISPATCH_SRC_DST(sd, dd, (bilateral_kernel<SrcT, DstT><<<(unsigned)blocks, 256, smem, st>>>(
                                     (const SrcT*)src, (DstT*)dst, ssn, ssh, dsn, dsh, h, w, tiles_x, tiles_y, ky, kx,
                                     coef, border, lo, hi - lo, sw)));
    return check_launch();
}

int launch_clahe_apply_index(const uint8_t* idx, const Image& d, int64_t n, const ClaheGeom& g, const uint8_t* luts,
                             void* cells, cudaStream_t st);   // clahe_fast.cu
size_t clahe_cells_bytes(int64_t n, int gh, int gw);

static inline size_t bc_align(size_t v) { return (v + 255) & ~(size_t)255; }

static bool bilateral_clahe_fused_ok(const ClaheGeom& g, int k, int sd, float lo, float hi) {
    if (k != 3 && k != 5 && k != 7 && k != 9) return false;
    if (g.hp != g.h || g.wp != g.w) return false;
    if ((g.th % 32) || (g.tw % 32)) return false;
    if ((g.w & 3) || g.w > 4096 || g.gw > 32) return false;    // interpolation kernel: one block spans a row
    if (!default_range_c(sd, lo, hi)) return false;
    if ((int64_t)g.th * g.tw >= (1 << 24)) return false;
    return true;
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_bilateral_clahe_workspace_bytes(int64_t n, int h, int w, int gh, int gw) {
    if (n <= 0 || h <= 0 || w <= 0 || gh <= 0 || gw <= 0) return 0;
    const size_t tiles = (size_t)n * gh * gw;
    return bc_align(tiles * kBins * sizeof(uint32_t)) + bc_align(tiles * kBins) + bc_align((size_t)n * h * w) +
           bc_align(clahe_cells_bytes(n, gh, gw));
}

int mie_bilateral_clahe_is_fused(int h, int w, int gh, int gw, int k, int dtype) {
    ClaheGeom g;
    if (make_clahe_geom(h, w, gh, gw, MIE_CLAHE_KORNIA, &g)) return 0;
    float lo = 0.f, hi = 1.f;
    if (dtype == MIE_U8) hi = 255.f; else if (dtype == MIE_U16) hi = 65535.f; else if (dtype == MIE_I16) { lo = -32768.f; hi = 32767.f; }
    return bilateral_clahe_fused_ok(g, k, dtype, lo, hi) ? 1 : 0;
}

int mie_bilateral_clahe(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                        int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                        const float* wspace, int k, float sigma_color, int border, int gh, int gw, double clip_limit,
                        float lo, float hi, int stages, void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const Image s{src, src_dtype, src_stride_n, src_stride_h}, d{dst, dst_dtype, dst_stride_n, dst_stride_h};
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    rc = check_dtypes(src_dtype, dst_dtype, lo, hi);
    if (rc) return rc;
    if (!wspace) return MIE_E_NULL;
    if (k <= 0 || !(k & 1) || k > 9) return MIE_E_KERNEL;
    if (border < MIE_BORDER_CONSTANT || border > MIE_BORDER_CIRCULAR) return MIE_E_BORDER;
    if (border == MIE_BORDER_REFLECT && (k / 2 >= w || k / 2 >= h)) return MIE_E_BORDER;
    if (!(sigma_color > 0.0f)) return MIE_E_RANGE;
    if (stages < 1 || stages > 7) return MIE_E_UNSUPPORTED;
    ClaheGeom g;
    rc = make_clahe_geom(h, w, gh, gw, MIE_CLAHE_KORNIA, &g);
    if (rc) return rc;
    if (!bilateral_clahe_fused_ok(g, k, src_dtype, lo, hi)) return MIE_E_UNSUPPORTED;
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < mie_bilateral_clahe_workspace_bytes(n, h, w, gh, gw)) return MIE_E_WORKSPACE;
    const int64_t tiles = n * gh * gw;
    const int tiles_x = w / 32, tiles_y = h / 32;
    const int64_t blocks = n * tiles_x * tiles_y;
    if (blocks > 2147483647LL || tiles > 2147483647LL) return MIE_E_SHAPE;
    uint8_t* ws = (uint8_t*)workspace;
    uint32_t* hist = (uint32_t*)ws;
    uint8_t* luts = ws + bc_align((size_t)tiles * kBins * sizeof(uint32_t));
    uint8_t* idx = luts + bc_align((size_t)tiles * kBins);
    void* cells = idx + bc_align((size_t)n * h * w);
    if (stages & 1) {   // bilateral -> index plane + tile histograms
        cudaError_t e = cudaMemsetAsync(hist, 0, (size_t)tiles * kBins * sizeof(uint32_t), st);
        if (e != cudaSuccess) return (int)e;
        const bool approx = bilateral_approx_ok(wspace, k);
        SpaceW2 sw;
        fill_space_weights(sw, wspace, k, approx);
        const float coef = (float)(-0.5 * 1.4426950408889634 / ((double)sigma_color * (double)sigma_color));
        const float rg = hi - lo;
#define MIE_BIDX(K_)                                                                                                   \
    case K_:                                                                                                           \
        if (approx) {                                                                                                  \
            MIE_DISPATCH_SRC(src_dtype, (bilateral_lean_index_kernel<SrcT, K_><<<(unsigned)blocks, 256, 0, st>>>(     \
                                            (const SrcT*)src, idx, hist, src_stride_n, src_stride_h, g, tiles_x, tiles_y, \
                                            coef, border, lo, rg, sw)));                                                \
        } else {                                                                                                       \
            MIE_DISPATCH_SRC(src_dtype, (bilateral_index_kernel<SrcT, K_><<<(unsigned)blocks, 256, 0, st>>>(    \
                                            (const SrcT*)src, idx, hist, src_stride_n, src_stride_h, g, tiles_x, tiles_y, \
                                            coef, border, lo, rg, sw)));                                                \
        }                                                                                                              \
        break;
        switch (k) {
            MIE_BIDX(3) MIE_BIDX(5) MIE_BIDX(7) MIE_BIDX(9)
            default: return MIE_E_KERNEL;
        }
#undef MIE_BIDX
        rc = check_launch();
        if (rc) return rc;
    }
    if (stages & 2) {   // histograms -> LUTs
        const LutParams lp = make_lut_params(g, clip_limit, MIE_CLAHE_KORNIA);
        hist_to_lut_kernel<<<(unsigned)((tiles + 7) / 8), 256, 0, st>>>(hist, luts, lp, tiles);
        rc = check_launch();
        if (rc) return rc;
    }
    if (stages & 4)     // index plane -> CLAHE blend -> quantise
        return launch_clahe_apply_index(idx, d, n, g, luts, cells, st);
    return MIE_OK;
}

int mie_bilateral(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                             int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                             const float* wspace, int ky, int kx, float sigma_color, int border, float lo, float hi,
                             void* stream) {
    return bilateral_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                          dst_stride_h, wspace, ky, kx, sigma_color, border, lo, hi, (cudaStream_t)stream);
}

}  // extern "C"
