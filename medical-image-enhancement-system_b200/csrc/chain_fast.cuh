// chain_fast.cuh — the tuned fused-chain kernels for the headline geometry
// (BASELINE.json config 2: 64x64-pixel CLAHE tiles, 9-tap Gaussians, integer
// slices with their full dtype range).  Same arithmetic, bit for bit, as the
// generic fused kernels in chain.cu and as oracle/mie_oracle.c; what changes is how
// few instructions each pixel costs:
//
//   * 64/128-bit global loads along x; no haloed input tile in shared memory for
//     chain_a — the horizontal pass runs straight out of registers;
//   * integer -> [0,1] without a divide:  v/65535 == fma(t, c, t) with
//     t = v * 2^-16 (built by OR-ing v into a float's mantissa) and c = RN(1/65535);
//     exact for all 65 536 codes (tests/test_host_logic.py emulates it exhaustively);
//   * floor()/trunc()/rint() by adding 2^23 in the matching rounding mode instead
//     of F2I conversions (which run on the 16-lane conversion pipe);
//   * x/255 as q0 = x*r; q = fma(fma(-255, q0, x), r, q0) (correctly rounded);
//   * histogram: one ATOMS.POPC.INC per pixel into a single block histogram — the
//     hardware aggregates same-address lanes (measured: constant 1.53 cycles per warp
//     instruction for 1..32-way collisions), so no software warp aggregation;
//   * the clip / redistribute / scan -> LUT tail runs in one warp (8 bins per lane);
//   * chain_b packs the four neighbouring LUTs of each interpolation cell into one
//     32-bit word per grey level, so a pixel needs ONE shared-memory lookup.
#pragma once

#include <cuda_fp16.h>

#include "clahe.cuh"
#include "stencil.cuh"

namespace mie {

constexpr int kFastThreads = 288;  // 9 warps: (64+2*4) rows x 8 segments = 2 x 288 row-pass items

// Launch arguments shared by the generic (chain.cu) and tuned (chain_fast.cu) fused kernels.
struct ChainAArgs {
    const void* src;
    int64_t ssn, ssh;
    uint8_t* idx;   // n*h*w lookup indices trunc(G*255)
    uint8_t* luts;  // n*gh*gw*256
    ClaheGeom g;
    LutParams lp;
    int border;
    float lo, rg;
};

struct ChainBArgs {
    const uint8_t* idx;
    const uint8_t* luts;
    void* dst;
    int64_t dsn, dsh;
    ClaheGeom g;
    int tiles_x, tiles_y;
    int border;
    int max_lut_tiles;  // LUT staging capacity (generic kernel)
    float lo, rg;
};

struct WinCvt;   // window.cuh

// Defined in chain_fast.cu.  `fast_chain_mode` returns -1 when the tuned kernels do not cover the request, else
// the range mode of window.cuh: 0 for the dtype's default range, 1 for an integer window the windowed conversion
// can take (*cv filled in).  The destination dtype is the source's or float32.
int fast_chain_mode(const ClaheGeom& g, const Image& s, const Image& d, int kg, int ku, int border, float lo, float hi,
                    WinCvt* cv);
int launch_chain_a_fast(const ChainAArgs& a, int src_dtype, const Taps& wx, const Taps& wy, int R, int64_t n,
                        cudaStream_t st, const WinCvt* win = nullptr);
size_t chain_cells_bytes(int64_t n, int gh, int gw);
// cells[n][gh+1][gw+1][256] (8 bytes each) from luts[n][gh][gw][256]; see chain_fast.cu
int launch_pack_cells(const uint8_t* luts, void* cells, int64_t n, int gh, int gw, cudaStream_t st);
int launch_chain_b_fast(const ChainBArgs& b, int dst_dtype, void* cells, const Taps& wx, const Taps& wy,
                        int64_t n, cudaStream_t st, const WinCvt* win = nullptr);

// low bytes of four words -> one word (3 PRMT)
__device__ __forceinline__ uint32_t pack_low_bytes(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

// Packed f32x2 values held as ONE 64-bit register pair.  The CUDA float2 intrinsics re-pack their
// operands at every call; when the two halves come from different producers (the marching kernels'
// register ring) ptxas then copies them into an aligned pair at every use.  Packing once and keeping
// the 64-bit value costs the two copies once.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_sub(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_dup(float v) { return f2_pack(v, v); }

// ---------------------------------------------------------------- exact default-range pixel mapping
template <typename T>
struct Fast;

template <>
struct Fast<uint16_t> {
    static constexpr float kC = 1.5259021893143654e-05f;  // RN(1/65535)
    static __device__ __forceinline__ float from_bits(uint32_t lo16_in_mantissa) {
        const float t = __fsub_rn(__uint_as_float(lo16_in_mantissa), 128.0f);  // v * 2^-16, exact
        return __fmaf_rn(t, kC, t);
    }
    static __device__ __forceinline__ float one(uint16_t v) { return from_bits(0x43000000u | v); }
    static __device__ __forceinline__ void cvt2(uint32_t w, float* x) {
        x[0] = from_bits(__byte_perm(w, 0x43000000u, 0x7610));
        x[1] = from_bits(__byte_perm(w, 0x43000000u, 0x7632));
    }
    static __device__ __forceinline__ void load4(const uint16_t* p, float* x) {  // p 8-byte aligned
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(p));
        cvt2(a.x, x); cvt2(a.y, x + 2);
    }
    // split form of load4 (the marching kernels issue the load rows ahead of the conversion)
    typedef uint2 raw4;
    static __device__ __forceinline__ raw4 ldg4(const uint16_t* p) { return __ldg(reinterpret_cast<const uint2*>(p)); }
    static __device__ __forceinline__ raw4 zero4() { return make_uint2(0u, 0u); }
    static __device__ __forceinline__ void cvt_raw4(raw4 a, float* x) { cvt2(a.x, x); cvt2(a.y, x + 2); }
    static __device__ __forceinline__ void load8(const uint16_t* p, float* x) {  // p 16-byte aligned
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(p));
        cvt2(b.x, x); cvt2(b.y, x + 2); cvt2(b.z, x + 4); cvt2(b.w, x + 6);
    }
    // rint(clamp(y,0,1)*65535) sits in the low 16 mantissa bits of the returned float's bit pattern
    static __device__ __forceinline__ uint32_t quant(float y) {
        const float c = __saturatef(y);   // == fminf(fmaxf(y, 0), 1) incl. NaN -> 0; folds into the producer as .SAT
        return __float_as_uint(__fadd_rn(__fmul_rn(c, 65535.0f), 8388608.0f));
    }
    // The same for two values at once.  The product is rounded BEFORE the magic add, as in quant(): written as
    // mul.rn.f32x2 followed by fma.rn.f32x2 (m * 1 + 2^23), which ptxas keeps as FMUL2 + FFMA2 — a mul + add pair it
    // would contract into one FFMA2 with a single rounding.
    static __device__ __forceinline__ f32x2 quant2(float y0, float y1) {
        const f32x2 m = f2_mul(f2_pack(__saturatef(y0), __saturatef(y1)), f2_pack(65535.0f, 65535.0f));
        return f2_fma(m, f2_pack(1.0f, 1.0f), f2_pack(8388608.0f, 8388608.0f));
    }
    static __device__ __forceinline__ uint32_t quant2_u16x2(float y0, float y1) {
        float a, b;
        f2_unpack(quant2(y0, y1), a, b);
        return __byte_perm(__float_as_uint(a), __float_as_uint(b), 0x5410);
    }
    static __device__ __forceinline__ void store4(uint16_t* p, const float* y) {
        uint2 o;
        o.x = quant2_u16x2(y[0], y[1]);
        o.y = quant2_u16x2(y[2], y[3]);
        __stcs(reinterpret_cast<uint2*>(p), o);   // streaming: an operator's output is not read again by that operator
    }
    // rows s and s + 1 of the thread's four columns (raw words a, b) -> packed (row s, row s + 1) pairs
    static __device__ __forceinline__ f32x2 from_bits2(uint32_t m0, uint32_t m1) {
        // m - 128 written as fma(m, 1, -128): the same exact difference, but FFMA2 takes broadcast scalar / immediate
        // operands where FADD2 needs both constants materialised as a register pair (two MOVs per use)
        const f32x2 t = f2_fma(f2_pack(__uint_as_float(m0), __uint_as_float(m1)), f2_pack(1.0f, 1.0f), f2_pack(-128.0f, -128.0f));
        return f2_fma(t, f2_pack(kC, kC), t);
    }
    // PRMT takes ONE immediate: with the exponent pattern 0x43000000 and the selector both constant, ptxas keeps the
    // selectors in uniform registers and copies one into a vector register before every PRMT (8 MOVs per row pair in the
    // marching kernels).  exp_magic() hands the pattern over as an opaque register value instead, so that the selectors
    // can be the immediates (ptxas folds a plain `mov` of the constant back in, hence the runtime zero).
    static __device__ __forceinline__ uint32_t exp_magic() {
        return 0x43000000u | (blockDim.y - 1u);   // blockDim.y == 1 for every launch of these kernels: a runtime 0
    }
    static __device__ __forceinline__ void cvt_pair4(raw4 a, raw4 b, f32x2* xp, uint32_t magic = 0x43000000u) {
        xp[0] = from_bits2(__byte_perm(a.x, magic, 0x7610), __byte_perm(b.x, magic, 0x7610));
        xp[1] = from_bits2(__byte_perm(a.x, magic, 0x7632), __byte_perm(b.x, magic, 0x7632));
        xp[2] = from_bits2(__byte_perm(a.y, magic, 0x7610), __byte_perm(b.y, magic, 0x7610));
        xp[3] = from_bits2(__byte_perm(a.y, magic, 0x7632), __byte_perm(b.y, magic, 0x7632));
    }
};

template <>
struct Fast<int16_t> {
    static __device__ __forceinline__ float one(int16_t v) {
        return Fast<uint16_t>::from_bits(0x43000000u | ((uint32_t)(uint16_t)v ^ 0x8000u));
    }
    static __device__ __forceinline__ void load4(const int16_t* p, float* x) {
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(p));
        Fast<uint16_t>::cvt2(a.x ^ 0x80008000u, x); Fast<uint16_t>::cvt2(a.y ^ 0x80008000u, x + 2);  // v + 32768
    }
    typedef uint2 raw4;
    static __device__ __forceinline__ raw4 ldg4(const int16_t* p) { return __ldg(reinterpret_cast<const uint2*>(p)); }
    static __device__ __forceinline__ raw4 zero4() { return make_uint2(0u, 0u); }
    static __device__ __forceinline__ void cvt_raw4(raw4 a, float* x) {
        Fast<uint16_t>::cvt2(a.x ^ 0x80008000u, x); Fast<uint16_t>::cvt2(a.y ^ 0x80008000u, x + 2);
    }
    static __device__ __forceinline__ void load8(const int16_t* p, float* x) {
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(p));
        Fast<uint16_t>::cvt2(b.x ^ 0x80008000u, x); Fast<uint16_t>::cvt2(b.y ^ 0x80008000u, x + 2);
        Fast<uint16_t>::cvt2(b.z ^ 0x80008000u, x + 4); Fast<uint16_t>::cvt2(b.w ^ 0x80008000u, x + 6);
    }
    static __device__ __forceinline__ void store4(int16_t* p, const float* y) {
        uint2 o;
        o.x = Fast<uint16_t>::quant2_u16x2(y[0], y[1]) ^ 0x80008000u;
        o.y = Fast<uint16_t>::quant2_u16x2(y[2], y[3]) ^ 0x80008000u;
        __stcs(reinterpret_cast<uint2*>(p), o);
    }
    static __device__ __forceinline__ uint32_t exp_magic() { return Fast<uint16_t>::exp_magic(); }
    static __device__ __forceinline__ void cvt_pair4(raw4 a, raw4 b, f32x2* xp, uint32_t magic = 0x43000000u) {
        a.x ^= 0x80008000u; a.y ^= 0x80008000u; b.x ^= 0x80008000u; b.y ^= 0x80008000u;   // v + 32768
        Fast<uint16_t>::cvt_pair4(a, b, xp, magic);
    }
};

template <>
struct Fast<uint8_t> {
    static constexpr float kC = 0.003921568859368563f;  // RN(1/255)
    static __device__ __forceinline__ float from_bits(uint32_t lo8_in_mantissa) {
        const float t = __fsub_rn(__uint_as_float(lo8_in_mantissa), 32768.0f);  // v * 2^-8, exact
        return __fmaf_rn(t, kC, t);
    }
    static __device__ __forceinline__ float one(uint8_t v) { return from_bits(0x47000000u | v); }
    static __device__ __forceinline__ void cvt4(uint32_t w, float* x) {
        x[0] = from_bits(__byte_perm(w, 0x47000000u, 0x7650));
        x[1] = from_bits(__byte_perm(w, 0x47000000u, 0x7651));
        x[2] = from_bits(__byte_perm(w, 0x47000000u, 0x7652));
        x[3] = from_bits(__byte_perm(w, 0x47000000u, 0x7653));
    }
    static __device__ __forceinline__ void load4(const uint8_t* p, float* x) {  // p 4-byte aligned
        cvt4(__ldg(reinterpret_cast<const uint32_t*>(p)), x);
    }
    typedef uint32_t raw4;
    static __device__ __forceinline__ raw4 ldg4(const uint8_t* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }
    static __device__ __forceinline__ raw4 zero4() { return 0u; }
    static __device__ __forceinline__ void cvt_raw4(raw4 a, float* x) { cvt4(a, x); }
    static __device__ __forceinline__ void load8(const uint8_t* p, float* x) {  // p 8-byte aligned
        const uint2 b = __ldg(reinterpret_cast<const uint2*>(p));
        cvt4(b.x, x); cvt4(b.y, x + 4);
    }
    static __device__ __forceinline__ uint32_t quant(float y) {  // value in the low byte of the bit pattern
        const float c = __saturatef(y);   // == fminf(fmaxf(y, 0), 1) incl. NaN -> 0; folds into the producer as .SAT
        return __float_as_uint(__fadd_rn(__fmul_rn(c, 255.0f), 8388608.0f));
    }
    static __device__ __forceinline__ void store4(uint8_t* p, const float* y) {
        *reinterpret_cast<uint32_t*>(p) = pack_low_bytes(quant(y[0]), quant(y[1]), quant(y[2]), quant(y[3]));
    }
};

template <>
struct Fast<float> {
    static __device__ __forceinline__ float one(float v) { return v; }
    static __device__ __forceinline__ void load4(const float* p, float* x) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p));
        x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
    }
    static __device__ __forceinline__ void load8(const float* p, float* x) {
        load4(p, x); load4(p + 4, x + 4);
    }
    typedef float4 raw4;
    static __device__ __forceinline__ raw4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
    static __device__ __forceinline__ raw4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ void cvt_raw4(raw4 v, float* x) { x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; }
    static __device__ __forceinline__ void store4(float* p, const float* y) {
        *reinterpret_cast<float4*>(p) = make_float4(y[0], y[1], y[2], y[3]);
    }
};

// ---------------------------------------------------------------- index rules without F2I
// floor(g*256) and trunc(clamp(g*255)): add 2^23 rounding toward -inf and read the mantissa.
// Same values as kornia_bin / kornia_idx (clahe.cuh).
constexpr int kDummyBin = 256;  // histogram slot that swallows pixels torch.histc would ignore
// Word offset into a 257-entry histogram: min(floor(g*256), 255), or kDummyBin outside [0,1] / NaN.
// NONNEG: the caller guarantees g >= 0 and not NaN (Gaussian of normalised integer pixels).
template <bool NONNEG>
__device__ __forceinline__ int fast_bin(float g) {
    float f = fminf(__fmaf_rd(g, 256.0f, 8388608.0f), 8388608.0f + 255.0f);
    const bool ok = NONNEG ? (g <= 1.0f) : (g >= 0.0f && g <= 1.0f);
    f = ok ? f : 8388608.0f + (float)kDummyBin;
    return (int)(__float_as_uint(f) - 0x4B000000u);
}
// Bit pattern whose low byte is trunc(clamp(g*255, 0, 255)) (NaN -> 0).
template <bool NONNEG>
__device__ __forceinline__ uint32_t fast_idx_bits(float g) {
    float f = __fmul_rn(g, 255.0f);
    if (!NONNEG) f = fmaxf(f, 0.0f);     // first, so that NaN -> 0 as in fminf(fmaxf(f, 0), 255) (clahe.cuh, oracle)
    f = fminf(f, 255.0f);
    return __float_as_uint(__fadd_rd(f, 8388608.0f));
}

// Vertical correlation of 4 adjacent columns with packed fma.rn.f32x2 (same per-lane rounding as
// four scalar fmas; one issue slot per two results).  win[k] = row k of the window, result row j.
template <int R>
__device__ __forceinline__ void col4_f32x2(const float4* win, int j, const Taps& wy, float* g) {
    const float2 w0 = make_float2(wy.w[0], wy.w[0]);
    float2 a = __fmul2_rn(w0, make_float2(win[j].x, win[j].y));
    float2 b = __fmul2_rn(w0, make_float2(win[j].z, win[j].w));
#pragma unroll
    for (int t = 1; t <= 2 * R; ++t) {
        const float2 wt = make_float2(wy.w[t], wy.w[t]);
        a = __ffma2_rn(wt, make_float2(win[j + t].x, win[j + t].y), a);
        b = __ffma2_rn(wt, make_float2(win[j + t].z, win[j + t].w), b);
    }
    g[0] = a.x; g[1] = a.y; g[2] = b.x; g[3] = b.y;
}

// x / 255, correctly rounded (Markstein: y = RN(1/b), q0 = RN(a*y), r = a - b*q0 exact, RN(q0 + r*y)).
__device__ __forceinline__ float div255(float x) {
    constexpr float r = 0.003921568859368563f;
    const float q0 = __fmul_rn(x, r);
    return __fmaf_rn(__fmaf_rn(-255.0f, q0, x), r, q0);
}

// x / 255 on a packed pair in TWO operations: 1/255 = r + r2 with r = RN(1/255), r2 = RN(1/255 - r); q = fma(x, r,
// RN(x * r2)).  Equal to the correctly rounded quotient for EVERY float with 7.7e-34 < |x| <= 256 and for 0
// (exhaustive host check: profiles/microbench/div255_check.c, 1 132 462 081 inputs; the failures of the two-operation
// form all lie in [1.2e-38, 7.7e-34], where x * r2 underflows).  A CLAHE blend is 0 or at least 2^-60 in magnitude: its
// operands are multiples of 2^-30 (integers times k/63 weights).
__device__ __forceinline__ f32x2 div255_x2(f32x2 x) {
    const f32x2 r = f2_dup(0.003921568859368563f), r2 = f2_dup(-2.3191758240217e-10f);
    return f2_fma(x, r, f2_mul(x, r2));
}

// Histogram increment.  atomicAdd(p, 1) with an unused result compiles to ATOMS.POPC.INC.32, which
// aggregates same-address lanes in hardware: measured on B200 at 1.53 cycles per warp instruction
// per SM for every same-address multiplicity from 1 to 32 (profiles/microbench/hist_prims_b200_r1.log),
// whereas software aggregation costs far more issue slots (MATCH.ANY: 64 cycles for 32 distinct
// values; a shfl/ballot/popc peel loop: ~14 instructions per distinct bin).  So constant images
// ("air") and noise cost the same, and no per-warp sub-histograms are needed.
__device__ __forceinline__ void hist_add(int* s_h, int bin) {
    if (bin >= 0) atomicAdd(&s_h[bin], 1);
}
// Branch-free form for histograms with a dummy slot (bin from fast_bin, always in range).
__device__ __forceinline__ void hist_add_nobranch(int* s_h, int bin) { atomicAdd(&s_h[bin], 1); }

// Histogram increment for values proven to lie in [0, 1] (integer pixels blurred with weights whose
// fp32 sum, accumulated in kernel order, does not exceed 1: gauss_of_ones_le1 on the host).  Then
// floor(g*256) is in [0, 256] with 256 <=> g == 1.0, which torch.histc counts in the last bin: slot 256
// is merged into bin 255 when the LUT is built (warp_build_lut<true>).  Three instructions per pixel:
// FFMA.RM (mantissa of g*256 + 2^23 rounded down = the bin), LEA (bin*4 + base) and ATOMS.POPC.INC.
// hist_base32 = shared-window address of slot 0 minus 4 * 0x4B000000 (mod 2^32).
__device__ __forceinline__ uint32_t hist_base32(const int* s_h) {
    return (uint32_t)__cvta_generic_to_shared(s_h) - (0x4B000000u << 2);
}
__device__ __forceinline__ void hist_add_le1(uint32_t base32, float g) {
    const uint32_t addr = base32 + (__float_as_uint(__fmaf_rd(g, 256.0f, 8388608.0f)) << 2);
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
}
// Bit pattern whose low byte is trunc(g*255) for g in [0, 1].
__device__ __forceinline__ uint32_t fast_idx_bits_le1(float g) {
    return __float_as_uint(__fadd_rd(__fmul_rn(g, 255.0f), 8388608.0f));
}
// The two LE1 rules on a packed pair of blurred values (same per-lane operations and rounding modes as
// fast_idx_bits_le1 / hist_add_le1; ptxas keeps mul.rn + add.rm apart because the rounding modes differ).
__device__ __forceinline__ f32x2 f2_add_rm(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_fma_rm(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rm.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ void idx_bits_le1_x2(f32x2 g, uint32_t& b0, uint32_t& b1) {
    float a, b;
    // RD(RN(g * 255) * 1 + 2^23): the add written as an fma with multiplicand 1 (exact), see from_bits2
    f2_unpack(f2_fma_rm(f2_mul(g, f2_pack(255.0f, 255.0f)), f2_pack(1.0f, 1.0f), f2_pack(8388608.0f, 8388608.0f)), a, b);
    b0 = __float_as_uint(a); b1 = __float_as_uint(b);
}
__device__ __forceinline__ void hist_add_le1_x2(uint32_t base32, f32x2 g) {
    float a, b;
    f2_unpack(f2_fma_rm(g, f2_pack(256.0f, 256.0f), f2_pack(8388608.0f, 8388608.0f)), a, b);
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(base32 + (__float_as_uint(a) << 2)) : "memory");
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(base32 + (__float_as_uint(b) << 2)) : "memory");
}

// Clip / redistribute / cumulate -> 256 LUT bytes, computed by ONE warp from the
// block-total histogram in shared memory (lane L owns bins 8L..8L+7).
// MERGE256: slot 256 holds pixels whose value is exactly 1.0 (see hist_add_le1) and belongs to bin 255.
template <bool MERGE256 = false>
__device__ __forceinline__ void warp_build_lut(const int* s_tot, const LutParams& p, uint8_t* lut_out, int lane) {
    int hv[8];
    {
        const int4 a = *reinterpret_cast<const int4*>(s_tot + 8 * lane);
        const int4 b = *reinterpret_cast<const int4*>(s_tot + 8 * lane + 4);
        hv[0] = a.x; hv[1] = a.y; hv[2] = a.z; hv[3] = a.w; hv[4] = b.x; hv[5] = b.y; hv[6] = b.z; hv[7] = b.w;
        if (MERGE256 && lane == 31) hv[7] += s_tot[256];
    }
    if (p.clip > 0) {
        int local = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { hv[k] = min(hv[k], p.clip); local += hv[k]; }
        const int clipped = p.pixels - warp_sum(local);
        const int resid = clipped & 255;
        const int redist = (clipped - resid) >> 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) hv[k] += redist + ((8 * lane + k) < resid ? 1 : 0);
    }
#pragma unroll
    for (int k = 1; k < 8; ++k) hv[k] += hv[k - 1];
    int incl = hv[7];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const int excl = incl - hv[7];
    uint32_t w0 = 0, w1 = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float f = __fmul_rn((float)(hv[k] + excl), p.lut_scale);
        f = floorf(fminf(fmaxf(f, 0.0f), 255.0f));
        const uint32_t b = (uint32_t)(int)f;
        if (k < 4) w0 |= b << (8 * k); else w1 |= b << (8 * (k - 4));
    }
    *reinterpret_cast<uint2*>(lut_out + 8 * lane) = make_uint2(w0, w1);
}

// 24 converted pixels x[0..23] = image columns c0-4 .. c0+19 of one row (16 outputs + halo 4);
// columns outside the image (left edge: c0 == 0, right edge: c0 + 16 == w) are filled from the
// registers already loaded, so edge tiles cost no extra loads.
template <typename SrcT>
__device__ __forceinline__ void load_row24(const SrcT* row, int c0, int w, int border, float* x) {
    Fast<SrcT>::load8(row + c0, x + 4);
    Fast<SrcT>::load8(row + c0 + 8, x + 12);
    if (c0 != 0) {
        Fast<SrcT>::load4(row + c0 - 4, x);
    } else if (border == MIE_BORDER_REFLECT) {
        x[0] = x[8]; x[1] = x[7]; x[2] = x[6]; x[3] = x[5];
    } else {
        const float e = border == MIE_BORDER_REPLICATE ? x[4] : 0.0f;
        x[0] = e; x[1] = e; x[2] = e; x[3] = e;
    }
    if (c0 + 16 != w) {
        Fast<SrcT>::load4(row + c0 + 16, x + 20);
    } else if (border == MIE_BORDER_REFLECT) {
        x[20] = x[18]; x[21] = x[17]; x[22] = x[16]; x[23] = x[15];
    } else {
        const float e = border == MIE_BORDER_REPLICATE ? x[19] : 0.0f;
        x[20] = e; x[21] = e; x[22] = e; x[23] = e;
    }
}

// s_mid row layout of the tuned chain_a kernel: the 16 column quads of a row are stored even quads
// first (quad q at word 4*(q/2)), odd quads from word 48 (4*(12 + q/2)), rows 84 words apart.  With
// it, the row pass (4 lanes of a row x 2 rows per quarter-warp, STS.128 each) and the column pass
// (8 lanes of a row per quarter-warp, LDS.128 each) both touch 32 distinct banks.
constexpr int kPMa = 84;
__device__ __forceinline__ int quad_off(int q) { return 4 * ((q >> 1) + ((q & 1) ? 12 : 0)); }

// Cell-table entry: four integers of magnitude <= 255 stored as the UPPER 16 bits of their fp32
// encodings (exact: 8 significant bits), e.x = hi16(tl - tr) | hi16(tr) << 16, e.y the same for the
// bottom pair.  Decoding is one PRMT / LOP3 per value on the integer pipe (an fp16 table would cost
// one HADD2.F32 per value on the FMA pipe, which is the busier one).
__device__ __forceinline__ uint32_t cell_word(int diff, int base) {
    return (__float_as_uint((float)diff) >> 16) | (__float_as_uint((float)base) & 0xFFFF0000u);
}
// CLAHE output of one pixel from its cell-table entry:
// t = tr + wx (tl - tr); b = br + wx (bl - br); out = (b + wy (t - b)) / 255, one fma per lerp.
__device__ __forceinline__ float clahe_px(uint2 e, float wxv, float wyv) {
    const float dt = __uint_as_float(__byte_perm(e.x, 0u, 0x1044)), tr = __uint_as_float(e.x & 0xFFFF0000u);
    const float db = __uint_as_float(__byte_perm(e.y, 0u, 0x1044)), br = __uint_as_float(e.y & 0xFFFF0000u);
    const float t = __fmaf_rn(wxv, dt, tr);
    const float b = __fmaf_rn(wxv, db, br);
    return div255(__fmaf_rn(wyv, __fsub_rn(t, b), b));
}

// The same for the pixels of rows s and s + 1 of one column as a packed pair (entries e0, e1; column weight wx2 =
// (wx, wx), row weights wy2 = (wy_s, wy_s+1)): one packed instruction per step instead of two scalar ones — the same
// IEEE operations per lane, so the same bits as clahe_px.
__device__ __forceinline__ f32x2 clahe_px2(uint2 e0, uint2 e1, f32x2 wx2, f32x2 wy2) {
    const f32x2 dt = f2_pack(__uint_as_float(__byte_perm(e0.x, 0u, 0x1044)), __uint_as_float(__byte_perm(e1.x, 0u, 0x1044)));
    const f32x2 tr = f2_pack(__uint_as_float(e0.x & 0xFFFF0000u), __uint_as_float(e1.x & 0xFFFF0000u));
    const f32x2 db = f2_pack(__uint_as_float(__byte_perm(e0.y, 0u, 0x1044)), __uint_as_float(__byte_perm(e1.y, 0u, 0x1044)));
    const f32x2 br = f2_pack(__uint_as_float(e0.y & 0xFFFF0000u), __uint_as_float(e1.y & 0xFFFF0000u));
    const f32x2 t = f2_fma(wx2, dt, tr);
    const f32x2 b = f2_fma(wx2, db, br);
    return div255_x2(f2_fma(wy2, f2_sub(t, b), b));
}

// Interpolation weight of the upper / left tile for haloed index k (tile position p = k - 4):
// kornia_axis() of any pixel at that position, identical for every interior tile; in the border
// half-tiles both neighbours are the same tile, so the value there is irrelevant.
struct AxisWeights {
    float w[kTile + 8];
};
inline void fill_axis_weights(AxisWeights& aw) {
    for (int k = 0; k < kTile + 8; ++k) {
        const int p = k - 4;                                          // position relative to the tile origin
        const int r = p < kTile / 2 ? p + kTile / 2 : p - kTile / 2;  // offset from the previous tile centre
        aw.w[k] = (float)(kTile - 1 - r) / (float)(kTile - 1);
    }
}

// Marching kernels (chain_march.cu): full-width 64-row bands, 9-tap Gaussians, W % 128 == 0, W <= 1024.
bool march_chain_ok(const ClaheGeom& g, int kg, int ku);
int launch_chain_a_march(const ChainAArgs& a, int src_dtype, const Taps& wx, const Taps& wy, int64_t n,
                         cudaStream_t st, const WinCvt* win = nullptr);
int launch_chain_b_march(const ChainBArgs& b, int dst_dtype, void* cells, const Taps& wx, const Taps& wy, int64_t n,
                         cudaStream_t st, const WinCvt* win = nullptr);

}  // namespace mie
