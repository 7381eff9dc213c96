// metrics.cu — full-reference quality metrics on device (SURVEY.md §8(f) F4): the reductions behind
// sewar.full_ref.mse / rmse / psnr / ssim (reference pyproject.toml:13, pin uv.lock:692-700; sewar 0.4.6
// is not installable here, semantics RECALLED — see oracle/oracle.py:sewar_*).
//
//   mie_sqdiff_sums : per plane  sum (a-b)^2  and  sum |a-b|            -> mse, rmse, psnr, mae
//   mie_ssim_sums   : per plane  sum ssim_map  and  sum cs_map over the 'valid' ws x ws uniform windows
//
// Pixels are used RAW (sewar works on pixel values, MAX = dtype maximum), not mapped to [0,1].
// Integer planes: every window / plane sum is accumulated in 64-bit integers, i.e. exactly; the only
// floating-point arithmetic is the float64 SSIM formula per window and the float64 sum of the maps.
// Float planes accumulate in float64.  All reductions run in a fixed order (per-thread, warp tree,
// block tree, then one block per plane over the block partials), so results are reproducible run to run.
#include <type_traits>

#include "mie_common.cuh"

namespace mie {

template <typename T> struct MetAcc { using type = long long; };
template <> struct MetAcc<float> { using type = double; };

template <typename A>
__device__ __forceinline__ A warp_tree(A v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Sum over the 256 threads of a block, fixed order; result valid in thread 0.
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

// ---------------------------------------------------------------- sum (a-b)^2, sum |a-b|
template <typename T>
__global__ void __launch_bounds__(256)
sqdiff_partial_kernel(const T* __restrict__ a, const T* __restrict__ b, int64_t asn, int64_t ash, int64_t bsn,
                      int64_t bsh, int h, int w, int rows_per_block, typename MetAcc<T>::type* __restrict__ part) {
    using A = typename MetAcc<T>::type;
    __shared__ A s8[8];
    const int64_t n = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    A s2 = 0, s1 = 0;
    for (int y = y0 + (threadIdx.x >> 5); y < y1; y += 8) {
        const T* ra = a + n * asn + (int64_t)y * ash;
        const T* rb = b + n * bsn + (int64_t)y * bsh;
        for (int x = threadIdx.x & 31; x < w; x += 32) {
            const A d = (A)ra[x] - (A)rb[x];
            s2 += d * d;
            s1 += d < 0 ? -d : d;
        }
    }
    const A t2 = block_tree_256(s2, s8);
    const A t1 = block_tree_256(s1, s8);
    if (threadIdx.x == 0) {
        A* o = part + (n * gridDim.x + blockIdx.x) * 2;
        o[0] = t2; o[1] = t1;
    }
}

// The same for 8 / 16-bit planes whose rows are 16-byte aligned multiples of 16 bytes: one 128-bit load per image and
// lane, (a - b)^2 accumulated exactly by 32 x 32 + 64-bit multiply-adds (|a - b| <= 65535, so the square fits 32 bits).
// Integer sums are exact in any order: the result is the one of the scalar kernel, bit for bit.
template <typename T>
__global__ void __launch_bounds__(256)
sqdiff_vec_kernel(const T* __restrict__ a, const T* __restrict__ b, int64_t asn, int64_t ash, int64_t bsn, int64_t bsh,
                  int h, int w, int rows_per_block, long long* __restrict__ part) {
    constexpr int PER = 16 / (int)sizeof(T);          // pixels per 128-bit load
    __shared__ long long s8[8];
    const int64_t n = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    const int vecs = w / PER, total = vecs * (y1 - y0);
    unsigned long long s2 = 0ull, s1 = 0ull;
    auto one = [&](int va, int vb) {
        const int d = va - vb;
        const unsigned ad = (unsigned)(d < 0 ? -d : d);
        s2 += (unsigned long long)ad * ad;
        s1 += ad;
    };
    (void)total;
    for (int r = threadIdx.x >> 5; r < y1 - y0; r += 8) {
        const uint4* ra = reinterpret_cast<const uint4*>(a + n * asn + (int64_t)(y0 + r) * ash);
        const uint4* rb = reinterpret_cast<const uint4*>(b + n * bsn + (int64_t)(y0 + r) * bsh);
#pragma unroll 4
        for (int c = threadIdx.x & 31; c < vecs; c += 32) {
        const uint4 qa = __ldg(ra + c);
        const uint4 qb = __ldg(rb + c);
        const uint32_t wa[4] = {qa.x, qa.y, qa.z, qa.w}, wb[4] = {qb.x, qb.y, qb.z, qb.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if constexpr (sizeof(T) == 1) {
#pragma unroll
                for (int j = 0; j < 4; ++j) one((int)((wa[k] >> (8 * j)) & 0xFFu), (int)((wb[k] >> (8 * j)) & 0xFFu));
            } else if constexpr (std::is_signed<T>::value) {
                one((int)(short)(wa[k] & 0xFFFFu), (int)(short)(wb[k] & 0xFFFFu));
                one((int)wa[k] >> 16, (int)wb[k] >> 16);
            } else {
                one((int)(wa[k] & 0xFFFFu), (int)(wb[k] & 0xFFFFu));
                one((int)(wa[k] >> 16), (int)(wb[k] >> 16));
            }
        }
        }
    }
    const long long t2 = block_tree_256((long long)s2, s8);
    const long long t1 = block_tree_256((long long)s1, s8);
    if (threadIdx.x == 0) {
        long long* o = part + (n * gridDim.x + blockIdx.x) * 2;
        o[0] = t2; o[1] = t1;
    }
}

// one block per plane: partials[n][count][2] -> out[n][2] (float64)
template <typename A>
__global__ void __launch_bounds__(256)
metric_finish_kernel(const A* __restrict__ part, int count, double* __restrict__ out) {
    __shared__ A s8[8];
    const int64_t n = blockIdx.x;
    A v0 = 0, v1 = 0;
    for (int i = threadIdx.x; i < count; i += 256) {
        v0 += part[(n * count + i) * 2];
        v1 += part[(n * count + i) * 2 + 1];
    }
    const A t0 = block_tree_256(v0, s8);
    const A t1 = block_tree_256(v1, s8);
    if (threadIdx.x == 0) { out[n * 2] = (double)t0; out[n * 2 + 1] = (double)t1; }
}

// ---------------------------------------------------------------- SSIM, uniform ws x ws window, 'valid'
constexpr int kSsimTile = 32;
constexpr int kSsimMaxWs = 16;

template <typename T> struct SsimRaw { using type = int; };
template <> struct SsimRaw<float> { using type = float; };

// Block = 32x32 windows.  Phase 1: raw tile (32+ws-1)^2 of both images in shared memory.  Phase 2: the five
// horizontal ws-sums (a, b, a^2, b^2, ab) for every tile row.  Phase 3: vertical ws-sums, the float64
// SSIM / CS formulas, block reduction.
template <typename T>
__global__ void __launch_bounds__(256)
ssim_partial_kernel(const T* __restrict__ a, const T* __restrict__ b, int64_t asn, int64_t ash, int64_t bsn,
                    int64_t bsh, int h, int w, int ws, int tiles_x, int tiles_y, double c1, double c2,
                    double* __restrict__ part) {
    using A = typename MetAcc<T>::type;
    using R = typename SsimRaw<T>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int e = kSsimTile + ws - 1;                       // tile edge with halo
    R* sa = reinterpret_cast<R*>(smem_raw);
    R* sb = sa + e * e;
    A* hs = reinterpret_cast<A*>(smem_raw + (((size_t)2 * e * e * sizeof(R) + 15) & ~(size_t)15));  // [5][e][32]
    __shared__ double s8[8];
    const int64_t n = blockIdx.y;
    const int tx0 = (int)(blockIdx.x % tiles_x) * kSsimTile, ty0 = (int)(blockIdx.x / tiles_x) * kSsimTile;
    const int oh = h - ws + 1, ow = w - ws + 1;
    const T* pa = a + n * asn;
    const T* pb = b + n * bsn;
    for (int i = threadIdx.x; i < e * e; i += 256) {
        const int r = i / e, c = i - r * e;
        const int y = min(ty0 + r, h - 1), x = min(tx0 + c, w - 1);   // clamped reads feed masked windows only
        sa[i] = (R)pa[(int64_t)y * ash + x];
        sb[i] = (R)pb[(int64_t)y * bsh + x];
    }
    __syncthreads();
    // Phase 2: horizontal ws-sums as RUNNING sums — a thread owns 8 consecutive windows of one tile row: the first sum in
    // full, then one sample in and one out per window (integer planes: exact; float planes: float64, 8 steps).
    for (int job = threadIdx.x; job < e * 4; job += 256) {
        const int r = job >> 2, l0 = (job & 3) * 8;
        const R* ra = sa + r * e + l0;
        const R* rb = sb + r * e + l0;
        A s_a = 0, s_b = 0, s_aa = 0, s_bb = 0, s_ab = 0;
        auto add = [&](R xa, R xb, int sign) {
            if constexpr (std::is_same<A, long long>::value) {
                const int va = xa, vb = xb;
                const long long aa = (long long)((unsigned)va * (unsigned)va), bb = (long long)((unsigned)vb * (unsigned)vb);
                const long long ab = (long long)va * vb;
                if (sign > 0) { s_a += va; s_b += vb; s_aa += aa; s_bb += bb; s_ab += ab; }
                else { s_a -= va; s_b -= vb; s_aa -= aa; s_bb -= bb; s_ab -= ab; }
            } else {
                const A va = (A)xa, vb = (A)xb;
                if (sign > 0) { s_a += va; s_b += vb; s_aa += va * va; s_bb += vb * vb; s_ab += va * vb; }
                else { s_a -= va; s_b -= vb; s_aa -= va * va; s_bb -= vb * vb; s_ab -= va * vb; }
            }
        };
        for (int k = 0; k < ws; ++k) add(ra[k], rb[k], 1);
        A* o = hs + r * 32 + l0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j) { add(ra[j + ws - 1], rb[j + ws - 1], 1); add(ra[j - 1], rb[j - 1], -1); }
            o[j] = s_a; o[e * 32 + j] = s_b; o[2 * e * 32 + j] = s_aa; o[3 * e * 32 + j] = s_bb; o[4 * e * 32 + j] = s_ab;
        }
    }
    __syncthreads();
    // Phase 3: vertical ws-sums, again running: a thread owns 4 consecutive windows of one column.
    const int lx = threadIdx.x & 31, r0 = (threadIdx.x >> 5) * 4;
    const double inv_n = 1.0 / (double)(ws * ws);
    double acc_s = 0.0, acc_c = 0.0;
    {
        A s_a = 0, s_b = 0, s_aa = 0, s_bb = 0, s_ab = 0;
        for (int k = 0; k < ws; ++k) {
            const A* p = hs + (r0 + k) * 32 + lx;
            s_a += p[0]; s_b += p[e * 32]; s_aa += p[2 * e * 32]; s_bb += p[3 * e * 32]; s_ab += p[4 * e * 32];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j) {
                const A* pi = hs + (r0 + j + ws - 1) * 32 + lx;
                const A* po = hs + (r0 + j - 1) * 32 + lx;
                s_a += pi[0] - po[0]; s_b += pi[e * 32] - po[e * 32]; s_aa += pi[2 * e * 32] - po[2 * e * 32];
                s_bb += pi[3 * e * 32] - po[3 * e * 32]; s_ab += pi[4 * e * 32] - po[4 * e * 32];
            }
            if (ty0 + r0 + j >= oh || tx0 + lx >= ow) continue;
            const double mu_a = (double)s_a * inv_n, mu_b = (double)s_b * inv_n;
            const double mu_aa = mu_a * mu_a, mu_bb = mu_b * mu_b, mu_ab = mu_a * mu_b;
            const double var_a = (double)s_aa * inv_n - mu_aa, var_b = (double)s_bb * inv_n - mu_bb;
            const double cov = (double)s_ab * inv_n - mu_ab;
            const double cs = (2.0 * cov + c2) / (var_a + var_b + c2);
            acc_c += cs;
            acc_s += ((2.0 * mu_ab + c1) * (2.0 * cov + c2)) / ((mu_aa + mu_bb + c1) * (var_a + var_b + c2));
        }
    }
    const double ts = block_tree_256(acc_s, s8);
    const double tc = block_tree_256(acc_c, s8);
    if (threadIdx.x == 0) {
        double* o = part + (n * gridDim.x + blockIdx.x) * 2;
        o[0] = ts; o[1] = tc;
    }
}

static size_t ssim_smem_bytes(int ws, int esz_raw, int esz_acc) {
    const int e = kSsimTile + ws - 1;
    return (((size_t)2 * e * e * esz_raw + 15) & ~(size_t)15) + (size_t)5 * e * 32 * esz_acc;
}

static int sqdiff_rows_per_block(int64_t n, int h) {
    int bpp = (int)((8 * 148 + n - 1) / n);
    int rows = ceil_div(h, bpp < 1 ? 1 : bpp);
    return rows < 8 ? 8 : rows;
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_metric_workspace_bytes(int64_t n, int h, int w, int ws) {
    if (n <= 0 || h <= 0 || w <= 0) return 0;
    size_t blocks;
    if (ws <= 0) {
        blocks = (size_t)ceil_div(h, sqdiff_rows_per_block(n, h));
    } else {
        if (ws > h || ws > w) return 0;
        blocks = (size_t)ceil_div(w - ws + 1, kSsimTile) * ceil_div(h - ws + 1, kSsimTile);
    }
    return (size_t)n * blocks * 2 * 8;
}

int mie_sqdiff_sums(const void* a, const void* b, int dtype, int64_t n, int h, int w, int64_t a_stride_n,
                    int64_t a_stride_h, int64_t b_stride_n, int64_t b_stride_h, double* out, void* workspace,
                    size_t workspace_bytes, void* stream) {
    const Image A{a, dtype, a_stride_n, a_stride_h}, B{b, dtype, b_stride_n, b_stride_h};
    int rc = check_planes(A, B, n, h, w);
    if (rc) return rc;
    if (!valid_dtype(dtype)) return MIE_E_DTYPE;
    if (n == 0) return MIE_OK;
    if (n > 65535) return MIE_E_SHAPE;
    if (!out || !workspace) return MIE_E_NULL;
    if (workspace_bytes < mie_metric_workspace_bytes(n, h, w, 0)) return MIE_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int rows = sqdiff_rows_per_block(n, h);
    const int count = ceil_div(h, rows);
    dim3 grid((unsigned)count, (unsigned)n);
    const bool vec = dtype != MIE_F32 && ((int64_t)w * A.bytes()) % 16 == 0 && A.aligned(16) && B.aligned(16);
#define MIE_SQDIFF(T)                                                                                          \
    if (vec && sizeof(T) != 4)                                                                                 \
        sqdiff_vec_kernel<T><<<grid, 256, 0, st>>>((const T*)a, (const T*)b, a_stride_n, a_stride_h, b_stride_n,   \
                                                   b_stride_h, h, w, rows, (long long*)workspace);             \
    else                                                                                                       \
        sqdiff_partial_kernel<T><<<grid, 256, 0, st>>>((const T*)a, (const T*)b, a_stride_n, a_stride_h, b_stride_n, \
                                                       b_stride_h, h, w, rows, (MetAcc<T>::type*)workspace);    \
    rc = check_launch();                                                                                       \
    if (rc) return rc;                                                                                         \
    metric_finish_kernel<MetAcc<T>::type><<<(unsigned)n, 256, 0, st>>>((const MetAcc<T>::type*)workspace, count, out)
    switch (dtype) {
        case MIE_U8: MIE_SQDIFF(uint8_t); break;
        case MIE_U16: MIE_SQDIFF(uint16_t); break;
        case MIE_I16: MIE_SQDIFF(int16_t); break;
        default:
            sqdiff_partial_kernel<float><<<grid, 256, 0, st>>>((const float*)a, (const float*)b, a_stride_n, a_stride_h,
                                                                b_stride_n, b_stride_h, h, w, rows, (double*)workspace);
            rc = check_launch();
            if (rc) return rc;
            metric_finish_kernel<double><<<(unsigned)n, 256, 0, st>>>((const double*)workspace, count, out);
            break;
    }
#undef MIE_SQDIFF
    return check_launch();
}

int mie_ssim_sums(const void* a, const void* b, int dtype, int64_t n, int h, int w, int64_t a_stride_n,
                  int64_t a_stride_h, int64_t b_stride_n, int64_t b_stride_h, int ws, double c1, double c2,
                  double* out, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_planes({a, dtype, a_stride_n, a_stride_h}, {b, dtype, b_stride_n, b_stride_h}, n, h, w);
    if (rc) return rc;
    if (!valid_dtype(dtype)) return MIE_E_DTYPE;
    if (ws < 1 || ws > kSsimMaxWs || ws > h || ws > w) return MIE_E_KERNEL;
    if (n == 0) return MIE_OK;
    if (n > 65535) return MIE_E_SHAPE;
    if (!out || !workspace) return MIE_E_NULL;
    if (workspace_bytes < mie_metric_workspace_bytes(n, h, w, ws)) return MIE_E_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int tiles_x = ceil_div(w - ws + 1, kSsimTile), tiles_y = ceil_div(h - ws + 1, kSsimTile);
    const int count = tiles_x * tiles_y;
    dim3 grid((unsigned)count, (unsigned)n);
#define MIE_SSIM(T)                                                                                         \
    {                                                                                                       \
        const size_t smem = ssim_smem_bytes(ws, 4, 8);                                                      \
        MIE_ENSURE_SMEM(ssim_partial_kernel<T>, ssim_smem_bytes(kSsimMaxWs, 4, 8));                         \
        ssim_partial_kernel<T><<<grid, 256, smem, st>>>((const T*)a, (const T*)b, a_stride_n, a_stride_h,   \
                                                        b_stride_n, b_stride_h, h, w, ws, tiles_x, tiles_y, c1, \
                                                        c2, (double*)workspace);                            \
    }
    switch (dtype) {
        case MIE_U8: MIE_SSIM(uint8_t); break;
        case MIE_U16: MIE_SSIM(uint16_t); break;
        case MIE_I16: MIE_SSIM(int16_t); break;
        default: MIE_SSIM(float); break;
    }
#undef MIE_SSIM
    rc = check_launch();
    if (rc) return rc;
    metric_finish_kernel<double><<<(unsigned)n, 256, 0, st>>>((const double*)workspace, count, out);
    return check_launch();
}

}  // extern "C"
