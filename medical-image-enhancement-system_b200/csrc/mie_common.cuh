// mie_common.cuh — shared device/host helpers for the sm_100a enhancement kernels.
//
// Pixel <-> [0,1] mapping, border index rules and launch plumbing.  The fp32
// operation order written here is the one oracle/mie_oracle.c restates; every
// float op that must match bit for bit uses an explicit-rounding intrinsic so
// that nvcc's -fmad contraction cannot reassociate it.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/mie.h"

namespace mie {

constexpr int kBins = 256;

struct Taps {
    float w[MIE_MAX_TAPS];
};

// ---------------------------------------------------------------- pixel traits
template <typename T>
struct Px;

template <>
struct Px<float> {
    static constexpr int code = MIE_F32;
    static __device__ __forceinline__ float to01(float v, float, float) { return v; }
    static __device__ __forceinline__ float from01(float y, float, float) { return y; }
};

template <typename T, int LO, int HI>
struct PxInt {
    static __device__ __forceinline__ float to01(T v, float lo, float rg) {
        return __fdiv_rn(__fsub_rn((float)v, lo), rg);
    }
    static __device__ __forceinline__ T from01(float y, float lo, float rg) {
        float c = __saturatef(y);   // == fminf(fmaxf(y, 0), 1) incl. NaN -> 0
        float q = __fadd_rn(rintf(__fmul_rn(c, rg)), lo);
        q = fminf(fmaxf(q, (float)LO), (float)HI);
        return (T)__float2int_rn(q);
    }
};
template <>
struct Px<uint8_t> : PxInt<uint8_t, 0, 255> {
    static constexpr int code = MIE_U8;
};
template <>
struct Px<uint16_t> : PxInt<uint16_t, 0, 65535> {
    static constexpr int code = MIE_U16;
};
template <>
struct Px<int16_t> : PxInt<int16_t, -32768, 32767> {
    static constexpr int code = MIE_I16;
};

// skimage.util.img_as_float of an integer code (float64): unsigned v / max, int16 (2 v + 1) / 65535.
template <typename T>
__device__ __forceinline__ double skb_as_float(int v) {
    if constexpr (sizeof(T) == 1) return __ddiv_rn((double)v, 255.0);
    else if constexpr (T(-1) > T(0)) return __ddiv_rn((double)v, 65535.0);
    else return __ddiv_rn(__dadd_rn(__dmul_rn((double)v, 2.0), 1.0), 65535.0);
}

// One correctly rounded operation each, never contracted to fma: the scikit-image kernels follow numpy's element-wise
// order with them, in the image's float type SkFloat<T> (float64 for integer images, float32 for float32 images).
__device__ __forceinline__ float rn_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double rn_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float rn_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double rn_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float rn_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double rn_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float rn_div(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double rn_div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float rn_sqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double rn_sqrt(double a) { return __dsqrt_rn(a); }

template <typename T>
using SkFloat = typename std::conditional<std::is_same<T, float>::value, float, double>::type;

// Fixed-order sums: a warp butterfly, then the 8 warp totals of a 256-thread block in index order (thread 0 holds the
// block's sum), so a reduction gives the same bits on every run.
template <typename A>
__device__ __forceinline__ A warp_tree(A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <typename A>
__device__ __forceinline__ A block_tree_256(A v, A* s8) {
    v = warp_tree(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s8[threadIdx.x >> 5] = v;
    __syncthreads();
    A t = 0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) t += s8[i];
    }
    return t;
}

// ---------------------------------------------------------------- borders
// Returns the source index for coordinate i of an axis of length n, or -1 for
// MIE_BORDER_CONSTANT outside the image.  Reflect = mirror without repeating
// the edge sample (torch 'reflect', cv2 BORDER_REFLECT_101, scipy 'mirror').
__host__ __device__ __forceinline__ int border_index(int i, int n, int mode) {
    if (i >= 0 && i < n) return i;
    switch (mode) {
        case MIE_BORDER_REFLECT: {
            if (n == 1) return 0;
            int p = 2 * (n - 1);
            int m = i % p;
            if (m < 0) m += p;
            return m < n ? m : p - m;
        }
        case MIE_BORDER_REPLICATE:
            return i < 0 ? 0 : n - 1;
        case MIE_BORDER_CIRCULAR: {
            int m = i % n;
            return m < 0 ? m + n : m;
        }
        case MIE_BORDER_SYMMETRIC: {   // period 2n: 0..n-1, n-1..0
            int p = 2 * n;
            int m = i % p;
            if (m < 0) m += p;
            return m < n ? m : p - 1 - m;
        }
        default:
            return -1;
    }
}

__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// ---------------------------------------------------------------- CLAHE geometry
struct ClaheGeom {
    int h, w;      // image
    int gh, gw;    // grid
    int th, tw;    // tile size in pixels
    int hp, wp;    // padded image (th*gh, tw*gw)
};

// kornia: tile = ceil(dim/grid), +1 if odd; pad bottom/right with 'reflect'.
// opencv: pad to the next multiple of the grid with BORDER_REFLECT_101 — BOTH axes by tiles - dim % tiles as soon
// as either is not divisible, so an evenly dividing axis then grows by a full `tiles` pixels (cv::CLAHE::apply).
inline int make_clahe_geom(int h, int w, int gh, int gw, int semantics, ClaheGeom* g) {
    if (h <= 0 || w <= 0) return MIE_E_SHAPE;
    if (gh <= 0 || gw <= 0) return MIE_E_GRID;
    g->h = h; g->w = w; g->gh = gh; g->gw = gw;
    if (semantics == MIE_CLAHE_KORNIA) {
        g->th = (h + gh - 1) / gh; g->tw = (w + gw - 1) / gw;
        g->th += g->th & 1; g->tw += g->tw & 1;
    } else if (semantics == MIE_CLAHE_OPENCV) {
        if (h % gh == 0 && w % gw == 0) { g->th = h / gh; g->tw = w / gw; }
        else { g->th = (h + gh - h % gh) / gh; g->tw = (w + gw - w % gw) / gw; }
    } else {
        return MIE_E_UNSUPPORTED;
    }
    g->hp = g->th * gh; g->wp = g->tw * gw;
    // torch.nn.functional.pad(mode='reflect') needs pad < dim; kornia raises
    // ValueError when pad > dim and torch raises for pad == dim.  OpenCV's
    // copyMakeBorder mirrors repeatedly, so any pad is legal there.
    if (semantics == MIE_CLAHE_KORNIA && (g->hp - h >= h || g->wp - w >= w)) return MIE_E_PAD;
    return MIE_OK;
}

// ---------------------------------------------------------------- host plumbing
// Process-wide kernel-selection mask set through mie_set_kernel_policy (include/mie.h): a verification hook that
// routes a request to the generic kernel although a tuned one covers it, so that tests can compare both on the
// same input.  Defined in mie_abi.cu; never read from the environment.
extern unsigned g_kernel_policy;
inline bool kernel_policy(unsigned bit) { return (g_kernel_policy & bit) != 0; }

inline int check_launch() {
    cudaError_t e = cudaPeekAtLastError();
    return e == cudaSuccess ? MIE_OK : (int)e;
}

// One image operand of a C-ABI call: plane i at p + i*sn, row y at + y*sh (strides in elements, include/mie.h).
// bytes() and aligned() need a valid dtype code.
struct Image {
    const void* p;
    int dtype;
    int64_t sn, sh;
    int bytes() const {
        static const int kEsz[4] = {1, 2, 2, 4};
        return kEsz[dtype];
    }
    // base, plane stride and row stride all multiples of b bytes (vector loads and stores of b bytes)
    bool aligned(int b) const { return (uintptr_t)p % b == 0 && sn * bytes() % b == 0 && sh * bytes() % b == 0; }
    void* out() const { return const_cast<void*>(p); }
};

// Rows no shorter than the width, and plane i + 1 starting after plane i's last row.
inline bool plane_strides_ok(const Image& x, int64_t n, int h, int w) {
    return x.sh >= w && (n <= 1 || x.sn >= (int64_t)(h - 1) * x.sh + w);
}

inline int check_planes(const Image& s, const Image& d, int64_t n, int h, int w) {
    if (n < 0 || h <= 0 || w <= 0) return MIE_E_SHAPE;
    if (n > 0 && (!s.p || !d.p)) return MIE_E_NULL;  // empty batches carry null pointers
    if (!plane_strides_ok(s, n, h, w) || !plane_strides_ok(d, n, h, w)) return MIE_E_STRIDE;
    return MIE_OK;
}

// Batches of volumes: sn is the volume stride, slice z of a volume starts at + z*slice_stride.
inline bool volume_strides_ok(const Image& x, int64_t slice_stride, int64_t n, int depth, int h, int w) {
    const int64_t slice = (int64_t)(h - 1) * x.sh + w;
    return x.sh >= w && (depth <= 1 || slice_stride >= slice) &&
           (n <= 1 || x.sn >= (int64_t)(depth - 1) * slice_stride + slice);
}

inline int check_volumes(const Image& s, int64_t ssd, const Image& d, int64_t dsd, int64_t n, int depth, int h, int w) {
    if (n < 0 || depth <= 0 || h <= 0 || w <= 0) return MIE_E_SHAPE;
    if (n > 0 && (!s.p || !d.p)) return MIE_E_NULL;
    if (!volume_strides_ok(s, ssd, n, depth, h, w) || !volume_strides_ok(d, dsd, n, depth, h, w)) return MIE_E_STRIDE;
    return MIE_OK;
}

inline bool valid_dtype(int d) { return d >= MIE_U8 && d <= MIE_F32; }

inline int check_dtypes(int sd, int dd, float lo, float hi) {
    if (!valid_dtype(sd) || !valid_dtype(dd)) return MIE_E_DTYPE;
    if (dd != sd && dd != MIE_F32) return MIE_E_DTYPE;
    if (sd != MIE_F32 && !(hi > lo)) return MIE_E_RANGE;
    return MIE_OK;
}

// Opt a kernel in to > 48 KB of dynamic shared memory once per device.
#define MIE_ENSURE_SMEM(kernel, bytes)                                                              \
    do {                                                                                            \
        static unsigned long long done_ = 0;                                                        \
        int dev_ = 0;                                                                               \
        cudaGetDevice(&dev_);                                                                       \
        if (!((done_ >> (dev_ & 63)) & 1ull)) {                                                     \
            cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)); \
            done_ |= 1ull << (dev_ & 63);                                                           \
        }                                                                                           \
    } while (0)

// Dispatch on (src dtype, dst dtype) with dst in {src, F32}.
#define MIE_DISPATCH_SRC(sd, ...)                                                   \
    switch (sd) {                                                                   \
        case MIE_U8: { using SrcT = uint8_t; __VA_ARGS__; } break;                  \
        case MIE_U16: { using SrcT = uint16_t; __VA_ARGS__; } break;                \
        case MIE_I16: { using SrcT = int16_t; __VA_ARGS__; } break;                 \
        case MIE_F32: { using SrcT = float; __VA_ARGS__; } break;                   \
        default: return MIE_E_DTYPE;                                                \
    }

#define MIE_DISPATCH_SRC_DST(sd, dd, ...)                                           \
    MIE_DISPATCH_SRC(sd, if ((dd) == MIE_F32) { using DstT = float; __VA_ARGS__; }  \
                         else { using DstT = SrcT; __VA_ARGS__; })

}  // namespace mie
