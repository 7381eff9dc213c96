// sk_exposure.cu — scikit-image exposure functions on the GPU (SURVEY.md §8(f) F3, Appendix B3):
//   skimage.exposure.equalize_adapthist  and  skimage.exposure.equalize_hist   (reference pyproject.toml:12).
// Both differ algorithmically from their kornia counterparts (clahe.cu / equalize.cu): 2^14 grey levels after a
// per-image min-max normalisation, an iterative clip redistribution, contextual regions anchored at the image
// origin with block-corner centred interpolation, and a final min-max rescale; the global equalisation maps every
// pixel through the image's own CDF in float64.
//
// RECALLED semantics (scikit-image is not on disk): the kernels follow the per-pixel restatement in
// oracle/mie_oracle.c (orc_sk_*), which is bit-identical to the array-level numpy twin oracle/skimage_twin.py.
// Arithmetic is the upstream's: float64 for integer images (explicit __d*_rn so that nothing is contracted into an
// fma), float32 for float32 images; histograms and the clip redistribution are integer work and bit-exact.
//
// Launches of mie_sk_equalize_adapthist (per batch of n planes):
//   sk_minmax_kernel        per-image min / max of the input codes (atomics on ordered ints)
//   sk_adapt_hist_kernel    one block per contextual region: grey level -> bin -> shared-memory histogram
//                           (ATOMS.POPC.INC), then warp 0 clips / redistributes / cumulates -> 16-bit mapping
//   sk_adapt_apply_kernel   per pixel: 4 mapping lookups, float64 coefficients, float32 accumulation in upstream's
//                           order, truncation to uint16; block-reduced min / max of the result
//   sk_rescale01_kernel     (c - min) / (max - min) in float64 -> float64 or float32 output
// mie_sk_equalize_adapthist3d (one image per (d, h, w) volume) runs the same stages on volumes: sk_minmax3d_kernel,
// sk_bin_table_kernel (integer codes -> bin), sk_adapt3d_hist_kernel (one cluster per 3-D region), sk_adapt3d_apply_kernel
// (8 lookups, trilinear), sk_rescale01_3d_kernel; the clip / map, min / max and rescale arithmetic is shared device code.
// Their per-voxel restatement is orc_sk_clahe3d in tests/sk_adapthist3d_oracle.c (built on oracle/mie_oracle.c).
#include <climits>

#include <cooperative_groups.h>

#include "mie_common.cuh"

namespace mie {

constexpr int kSkGray = 16384;       // NR_OF_GRAY
constexpr int kSkMaxBins = 4096;     // shared-memory histogram capacity of the region kernel

struct SkRange {     // per-image input range (workspace): ordered-int min / max
    int mn, mx;
};

__device__ __forceinline__ int float_order(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float float_unorder(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

template <typename T>
__device__ __forceinline__ int sk_key(T v) {
    if constexpr (sizeof(T) == 4) return float_order(v);
    else return (int)v;
}

// img_as_float of one integer code (unsigned: v / max; int16: (2 v + 1) / 65535)
template <typename T>
__device__ __forceinline__ double sk_as_float(int v) {
    if constexpr (sizeof(T) == 1) return __ddiv_rn((double)v, 255.0);
    else if constexpr (T(-1) > T(0)) return __ddiv_rn((double)v, 65535.0);
    else return __ddiv_rn(__dadd_rn(__dmul_rn((double)v, 2.0), 1.0), 65535.0);
}

__global__ void sk_init_ranges_kernel(SkRange* r, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { r[i].mn = INT_MAX; r[i].mx = INT_MIN; }
}

// min / max of one row's ordered keys, strided over the 256 threads of a block
template <typename T>
__device__ __forceinline__ void sk_row_minmax(const T* __restrict__ row, int w, int& mn, int& mx) {
    for (int x = threadIdx.x; x < w; x += 256) {
        const int k = sk_key<T>(row[x]);
        mn = min(mn, k); mx = max(mx, k);
    }
}

// warp-reduce a thread's (mn, mx) and fold it into *out with one pair of atomics per warp
__device__ __forceinline__ void sk_commit_minmax(int mn, int mx, SkRange* out) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0 && mn <= mx) { atomicMin(&out->mn, mn); atomicMax(&out->mx, mx); }
}

template <typename T>
__global__ void __launch_bounds__(256)
sk_minmax_kernel(const T* __restrict__ src, int64_t ssn, int64_t ssh, int h, int w, int rows_per_block, SkRange* out) {
    const int64_t n = blockIdx.y;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    int mn = INT_MAX, mx = INT_MIN;
    for (int y = y0; y < y1; ++y) sk_row_minmax<T>(src + n * ssn + (int64_t)y * ssh, w, mn, mx);
    sk_commit_minmax(mn, mx, &out[n]);
}

// The 2^14-level grey value CLAHE sees: round(rescale_intensity(img_as_float(v), out_range=(0, 16383))).
template <typename T>
struct SkGrey {
    double f_lo, span;   // integer images: float64
    float mn32, span32;  // float32 images: float32
    bool flat;
    __device__ __forceinline__ void init(const SkRange& r) {
        flat = r.mn == r.mx;
        if constexpr (sizeof(T) == 4) {
            mn32 = float_unorder(r.mn);
            span32 = __fsub_rn(float_unorder(r.mx), mn32);
        } else {
            f_lo = sk_as_float<T>(r.mn);
            span = __dsub_rn(sk_as_float<T>(r.mx), f_lo);
        }
    }
    __device__ __forceinline__ int grey(T v) const {
        if constexpr (sizeof(T) == 4) {
            float g;
            if (!flat) g = __fadd_rn(__fmul_rn(__fdiv_rn(__fsub_rn(v, mn32), span32), 16383.0f), 0.0f);
            else g = fminf(fmaxf(v, 0.0f), 16383.0f);
            return (int)(uint16_t)(long long)rintf(g);
        } else {
            const double f = sk_as_float<T>((int)v);
            double g;
            if (!flat) g = __dadd_rn(__dmul_rn(__ddiv_rn(__dsub_rn(f, f_lo), span), 16383.0), 0.0);
            else g = fmin(fmax(f, 0.0), 16383.0);
            return (int)(uint16_t)(long long)rint(g);
        }
    }
};

// numpy.pad(mode='reflect') index
__device__ __forceinline__ int sk_reflect(int i, int n) {
    if (i >= 0 && i < n) return i;
    if (n == 1) return 0;
    const int p = 2 * (n - 1);
    int m = i % p;
    if (m < 0) m += p;
    return m < n ? m : p - m;
}

__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct SkAdaptArgs {
    int h, w, kr, kc, nbr, nbc, nbins, bin_size;
    int clim;
    double scale;   // 16383 / (kr * kc)
};

// clip_histogram + map_histogram of one region's shared-memory histogram s_hist[0 .. nb), run by one full warp; the
// 16-bit mapping goes to out[0 .. nb).  Integer work except the final float64 scale.
__device__ __forceinline__ void sk_clip_map_warp(int* s_hist, int nb, int clim, double scale, uint16_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    // ---- clip_histogram (lane L owns bins L, L + 32, ...)
    int n_excess = 0;
    for (int b = lane; b < nb; b += 32) {
        const int v = s_hist[b];
        if (v > clim) { n_excess += v - clim; s_hist[b] = clim; }
    }
    n_excess = warp_sum_i(n_excess);
    const int bin_incr = n_excess / nb;
    const int upper = clim - bin_incr;
    int d = 0;
    for (int b = lane; b < nb; b += 32)
        if (s_hist[b] < upper) { d -= bin_incr; s_hist[b] += bin_incr; }
    // mid mask on the UPDATED histogram (own bins only: no cross-lane dependency)
    for (int b = lane; b < nb; b += 32) {
        const int v = s_hist[b];
        if (v >= upper && v < clim) { d += v - clim; s_hist[b] = clim; }
    }
    n_excess += warp_sum_i(d);
    __syncwarp();
    while (n_excess > 0) {
        const int prev = n_excess;
        for (int index = 0; index < nb; ++index) {
            int under = 0;
            for (int b = lane; b < nb; b += 32) under += s_hist[b] < clim;
            under = warp_sum_i(under);
            int step = under / n_excess;
            if (step < 1) step = 1;
            const int npos = (nb - index + step - 1) / step;
            int given = 0;
            for (int j = lane; j < npos; j += 32) {
                const int b = index + j * step;
                if (s_hist[b] < clim) { s_hist[b] += 1; ++given; }
            }
            __syncwarp();
            n_excess -= warp_sum_i(given);
            if (n_excess <= 0) break;
        }
        if (prev == n_excess) break;
    }
    __syncwarp();
    // ---- map_histogram: int(min(cumsum * scale + 0, 16383)); chunked warp scan over the bins in order
    int carry = 0;
    for (int b0 = 0; b0 < nb; b0 += 32) {
        const int b = b0 + lane;
        int v = b < nb ? s_hist[b] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        const int cum = carry + v;
        if (b < nb) {
            double m = __dadd_rn(__dmul_rn((double)cum, scale), 0.0);
            m = m > 16383.0 ? 16383.0 : m;
            out[b] = (uint16_t)(long long)m;
        }
        carry = __shfl_sync(0xffffffffu, cum, 31);
    }
}

// One block per contextual region (bj, bi, n).
template <typename T>
__global__ void __launch_bounds__(256)
sk_adapt_hist_kernel(const T* __restrict__ src, int64_t ssn, int64_t ssh, SkAdaptArgs a, const SkRange* __restrict__ ranges,
                     uint16_t* __restrict__ maps) {
    extern __shared__ int s_hist[];
    const int tid = threadIdx.x;
    const int bj = blockIdx.x, bi = blockIdx.y;
    const int64_t n = blockIdx.z;
    for (int b = tid; b < a.nbins; b += 256) s_hist[b] = 0;
    SkGrey<T> G;
    G.init(ranges[n]);
    __syncthreads();
    const T* plane = src + n * ssn;
    const int total = a.kr * a.kc;
    for (int i = tid; i < total; i += 256) {
        const int r = i / a.kc, c = i - r * a.kc;
        const int sy = sk_reflect(bi * a.kr + r, a.h), sx = sk_reflect(bj * a.kc + c, a.w);
        atomicAdd(&s_hist[G.grey(plane[(int64_t)sy * ssh + sx]) / a.bin_size], 1);
    }
    __syncthreads();
    if (tid >= 32) return;
    sk_clip_map_warp(s_hist, a.nbins, a.clim, a.scale, maps + (((int64_t)n * a.nbr + bi) * a.nbc + bj) * a.nbins);
}

// Interpolation pass: 256 threads = 32 columns x 8 rows per step; a block covers 32 x 32 pixels.
template <typename T>
__global__ void __launch_bounds__(256)
sk_adapt_apply_kernel(const T* __restrict__ src, int64_t ssn, int64_t ssh, SkAdaptArgs a, const SkRange* __restrict__ ranges,
                      const uint16_t* __restrict__ maps, uint16_t* __restrict__ cplane, SkRange* __restrict__ out_ranges) {
    const int64_t n = blockIdx.z;
    SkGrey<T> G;
    G.init(ranges[n]);
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int r0 = a.kr / 2, c0 = a.kc / 2;
    int mn = INT_MAX, mx = INT_MIN;
    const uint16_t* m0 = maps + (int64_t)n * a.nbr * a.nbc * a.nbins;
    if (x < a.w) {
        const int px = x + c0, bx = px / a.kc, rx = px - bx * a.kc;
        const double cx = __ddiv_rn((double)rx, (double)a.kc);
        const double wx0 = __dsub_rn(1.0, cx), wx1 = cx;
        const int hc0 = min(max(bx - 1, 0), a.nbc - 1), hc1 = min(max(bx, 0), a.nbc - 1);
        for (int k = 0; k < 4; ++k) {
            const int y = blockIdx.y * 32 + (threadIdx.x >> 5) + 8 * k;
            if (y >= a.h) break;
            const int py = y + r0, by = py / a.kr, ry = py - by * a.kr;
            const double cy = __ddiv_rn((double)ry, (double)a.kr);
            const double wy0 = __dsub_rn(1.0, cy), wy1 = cy;
            const int hr0 = min(max(by - 1, 0), a.nbr - 1), hr1 = min(max(by, 0), a.nbr - 1);
            const int bin = G.grey(src[n * ssn + (int64_t)y * ssh + x]) / a.bin_size;
            const uint16_t* t0 = m0 + (int64_t)hr0 * a.nbc * a.nbins + bin;
            const uint16_t* t1 = m0 + (int64_t)hr1 * a.nbc * a.nbins + bin;
            float acc = 0.0f;
            acc = __fadd_rn(acc, (float)__dmul_rn((double)__ldg(t0 + hc0 * a.nbins), __dmul_rn(wx0, wy0)));
            acc = __fadd_rn(acc, (float)__dmul_rn((double)__ldg(t0 + hc1 * a.nbins), __dmul_rn(wx1, wy0)));
            acc = __fadd_rn(acc, (float)__dmul_rn((double)__ldg(t1 + hc0 * a.nbins), __dmul_rn(wx0, wy1)));
            acc = __fadd_rn(acc, (float)__dmul_rn((double)__ldg(t1 + hc1 * a.nbins), __dmul_rn(wx1, wy1)));
            const int c = (int)(uint16_t)(int)acc;
            cplane[(n * a.h + y) * (int64_t)a.w + x] = (uint16_t)c;
            mn = min(mn, c); mx = max(mx, c);
        }
    }
    sk_commit_minmax(mn, mx, &out_ranges[n]);
}

// rescale_intensity(out_range=(0, 1)) of one uint16 CLAHE value.  F32MATH: float32 images keep float32 arithmetic.
template <typename DstT, bool F32MATH>
__device__ __forceinline__ DstT sk_rescale01_value(int v, const SkRange& r) {
    if constexpr (F32MATH) {
        float q;
        if (r.mn != r.mx) q = __fadd_rn(__fmul_rn(__fdiv_rn(__fsub_rn((float)v, (float)r.mn), __fsub_rn((float)r.mx, (float)r.mn)), 1.0f), 0.0f);
        else q = fminf(fmaxf((float)v, 0.0f), 1.0f);
        return (DstT)q;
    } else {
        double q;
        if (r.mn != r.mx) q = __dadd_rn(__dmul_rn(__ddiv_rn(__dsub_rn((double)v, (double)r.mn), __dsub_rn((double)r.mx, (double)r.mn)), 1.0), 0.0);
        else q = fmin(fmax((double)v, 0.0), 1.0);
        return (DstT)q;
    }
}

template <typename DstT, bool F32MATH>
__global__ void __launch_bounds__(256)
sk_rescale01_kernel(const uint16_t* __restrict__ c, DstT* __restrict__ dst, int64_t dsn, int64_t dsh, int h, int w,
                    const SkRange* __restrict__ ranges) {
    const int64_t n = blockIdx.z;
    const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    dst[n * dsn + (int64_t)y * dsh + x] = sk_rescale01_value<DstT, F32MATH>(c[(n * h + y) * (int64_t)w + x], ranges[n]);
}

// ---------------------------------------------------------------- equalize_adapthist on volumes (skimage on a 3-D array)
// Same stages as above with one (D, H, W) volume as the image: min / max over the volume, 3-D contextual regions of
// (kd, kr, kc) voxels anchored at the origin, trilinear blend of 8 mappings, min-max rescale over the volume.  Voxel
// offsets are int64 and every grid is flat in x (a volume has d * h rows and can have more than 65 535 regions).
constexpr int kSkCodes = 65536;          // per-volume stride of the code -> bin tables (uint16 / int16 codes)
constexpr int kSkVoxelsPerCta = 16384;   // a region larger than this is counted by a cluster of up to 8 CTAs

struct SkAdapt3Args {
    int d, h, w, kd, kr, kc, nbz, nby, nbx, nbins, bin_size, clim;
    int rows_per_cta;   // (z, y) rows of a region counted by one CTA of its cluster
    int tpr;            // threads per region row in the histogram pass: a power of two >= min(kc, 32)
    double scale;       // 16383 / (kd * kr * kc)
    int64_t ssn, ssd, ssh;
};

// Grey bin of a voxel.  Integer images: the bin depends on the code alone, so it is looked up in the per-volume table
// that sk_bin_table_kernel fills with SkGrey::grey(code) / bin_size (no float64 division per voxel).  float32 images
// keep the per-voxel float32 arithmetic of SkGrey.
template <typename T>
struct SkBin {
    const uint16_t* table;
    SkGrey<T> G;
    int bin_size;
    __device__ __forceinline__ void init(const SkRange* ranges, const uint16_t* tables, int64_t n, int bs) {
        if constexpr (sizeof(T) == 4) { G.init(ranges[n]); bin_size = bs; }
        else table = tables + n * kSkCodes;
    }
    __device__ __forceinline__ int operator()(T v) const {
        if constexpr (sizeof(T) == 4) return G.grey(v) / bin_size;
        else if constexpr (T(-1) > T(0)) return __ldg(table + (int)v);
        else return __ldg(table + (int)v + 32768);
    }
};

template <typename T>
__global__ void __launch_bounds__(256)
sk_bin_table_kernel(const SkRange* __restrict__ ranges, int bin_size, int ncodes, uint16_t* __restrict__ tables) {
    const int64_t n = blockIdx.y;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= ncodes) return;
    SkGrey<T> G;
    G.init(ranges[n]);
    const int v = T(-1) > T(0) ? i : i - 32768;
    tables[n * kSkCodes + i] = (uint16_t)(G.grey((T)v) / bin_size);
}

// rows_per_block (z, y) rows of volume blockIdx.y per block
template <typename T>
__global__ void __launch_bounds__(256)
sk_minmax3d_kernel(const T* __restrict__ src, SkAdapt3Args a, int rows_per_block, SkRange* out) {
    const int64_t n = blockIdx.y;
    const int r0 = blockIdx.x * rows_per_block, r1 = min(r0 + rows_per_block, a.d * a.h);
    int mn = INT_MAX, mx = INT_MIN;
    for (int r = r0; r < r1; ++r) {
        const int z = r / a.h, y = r - z * a.h;
        sk_row_minmax<T>(src + n * a.ssn + z * a.ssd + y * a.ssh, a.w, mn, mx);
    }
    sk_commit_minmax(mn, mx, &out[n]);
}

// One thread-block cluster per contextual region (region = blockIdx.x / cluster size; regions in (n, bz, by, bx) order).
// CTA `rank` counts the (z, y) rows [rank * rows_per_cta, ...) of the region into its own shared histogram; the leader
// adds the peers' histograms through DSMEM, then its warp 0 clips and maps like the 2-D kernel.
template <typename T>
__global__ void __launch_bounds__(256)
sk_adapt3d_hist_kernel(const T* __restrict__ src, SkAdapt3Args a, const SkRange* __restrict__ ranges,
                       const uint16_t* __restrict__ tables, uint16_t* __restrict__ maps) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ int s_hist[];
    const int tid = threadIdx.x;
    const unsigned cs = cluster.num_blocks(), rank = cluster.block_rank();
    const int64_t region = blockIdx.x / cs;
    const int64_t per_vol = (int64_t)a.nbz * a.nby * a.nbx;
    const int64_t n = region / per_vol;
    const int64_t rem = region - n * per_vol;
    const int bz = (int)(rem / ((int64_t)a.nby * a.nbx));
    const int rem2 = (int)(rem - (int64_t)bz * a.nby * a.nbx);
    const int by = rem2 / a.nbx, bx = rem2 - by * a.nbx;
    for (int b = tid; b < a.nbins; b += 256) s_hist[b] = 0;
    SkBin<T> B;
    B.init(ranges, tables, n, a.bin_size);
    __syncthreads();
    const T* vol = src + n * a.ssn;
    const int lane = tid & (a.tpr - 1), sub = tid / a.tpr, step = 256 / a.tpr;
    const int q1 = (int)min((int64_t)(rank + 1) * a.rows_per_cta, (int64_t)a.kd * a.kr);
    for (int q = (int)rank * a.rows_per_cta + sub; q < q1; q += step) {
        const int dz = q / a.kr, r = q - dz * a.kr;
        const T* row = vol + sk_reflect(bz * a.kd + dz, a.d) * a.ssd + sk_reflect(by * a.kr + r, a.h) * a.ssh;
        for (int c = lane; c < a.kc; c += a.tpr) atomicAdd(&s_hist[B(row[sk_reflect(bx * a.kc + c, a.w)])], 1);
    }
    cluster.sync();
    if (rank == 0)
        for (int b = tid; b < a.nbins; b += 256) {
            int s = s_hist[b];
            for (unsigned r = 1; r < cs; ++r) s += *cluster.map_shared_rank(&s_hist[b], r);
            s_hist[b] = s;
        }
    cluster.sync();   // the peers' shared memory stays alive until the leader has read it
    if (rank != 0 || tid >= 32) return;
    sk_clip_map_warp(s_hist, a.nbins, a.clim, a.scale, maps + region * a.nbins);
}

// Interpolation pass on volumes: a block covers 32 x 32 voxels of one slice z (blockIdx.x = ((n * d + z) * tiles_y + ty)
// * tiles_x + tx).  Per voxel 8 mapping lookups; coefficient of edge (ez, ey, ex) = (wx[ex] * wy[ey]) * wz[ez] in
// float64 (np.prod over the axes, x first); float32 accumulation in np.ndindex(2, 2, 2) order (z outermost, x
// innermost); truncation to uint16; block-reduced min / max of the result.
template <typename T>
__global__ void __launch_bounds__(256)
sk_adapt3d_apply_kernel(const T* __restrict__ src, SkAdapt3Args a, int tiles_x, int tiles_y, const SkRange* __restrict__ ranges,
                        const uint16_t* __restrict__ tables, const uint16_t* __restrict__ maps, uint16_t* __restrict__ cvol,
                        SkRange* __restrict__ out_ranges) {
    int t = blockIdx.x;
    const int tx = t % tiles_x; t /= tiles_x;
    const int ty = t % tiles_y; t /= tiles_y;
    const int z = t % a.d;
    const int64_t n = t / a.d;
    SkBin<T> B;
    B.init(ranges, tables, n, a.bin_size);
    const int pz = z + a.kd / 2, bz = pz / a.kd, rz = pz - bz * a.kd;
    const double cz = __ddiv_rn((double)rz, (double)a.kd);
    const double wz[2] = {__dsub_rn(1.0, cz), cz};
    const int64_t zplane = (int64_t)a.nby * a.nbx * a.nbins;
    const uint16_t* m0 = maps + n * a.nbz * zplane;
    const uint16_t* mz[2] = {m0 + min(max(bz - 1, 0), a.nbz - 1) * zplane, m0 + min(max(bz, 0), a.nbz - 1) * zplane};
    const int x = tx * 32 + (threadIdx.x & 31);
    int mn = INT_MAX, mx = INT_MIN;
    if (x < a.w) {
        const int px = x + a.kc / 2, bx = px / a.kc, rx = px - bx * a.kc;
        const double cx = __ddiv_rn((double)rx, (double)a.kc);
        const double wx[2] = {__dsub_rn(1.0, cx), cx};
        const int64_t hx[2] = {(int64_t)min(max(bx - 1, 0), a.nbx - 1) * a.nbins, (int64_t)min(max(bx, 0), a.nbx - 1) * a.nbins};
        const T* srow = src + n * a.ssn + z * a.ssd + x;
        uint16_t* crow = cvol + (n * a.d + z) * a.h * (int64_t)a.w + x;
        for (int k = 0; k < 4; ++k) {
            const int y = ty * 32 + (threadIdx.x >> 5) + 8 * k;
            if (y >= a.h) break;
            const int py = y + a.kr / 2, by = py / a.kr, ry = py - by * a.kr;
            const double cy = __ddiv_rn((double)ry, (double)a.kr);
            const double wy[2] = {__dsub_rn(1.0, cy), cy};
            const int64_t hy[2] = {(int64_t)min(max(by - 1, 0), a.nby - 1) * a.nbx * a.nbins,
                                   (int64_t)min(max(by, 0), a.nby - 1) * a.nbx * a.nbins};
            const int bin = B(srow[y * a.ssh]);
            float acc = 0.0f;
#pragma unroll
            for (int ez = 0; ez < 2; ++ez)
#pragma unroll
                for (int ey = 0; ey < 2; ++ey)
#pragma unroll
                    for (int ex = 0; ex < 2; ++ex) {
                        const double coef = __dmul_rn(__dmul_rn(wx[ex], wy[ey]), wz[ez]);
                        acc = __fadd_rn(acc, (float)__dmul_rn((double)__ldg(mz[ez] + hy[ey] + hx[ex] + bin), coef));
                    }
            const int c = (int)(uint16_t)(int)acc;
            crow[(int64_t)y * a.w] = (uint16_t)c;
            mn = min(mn, c); mx = max(mx, c);
        }
    }
    sk_commit_minmax(mn, mx, &out_ranges[n]);
}

// one row of 256 voxels per block: blockIdx.x = ((n * d + z) * h + y) * tiles_x + tx
template <typename DstT, bool F32MATH>
__global__ void __launch_bounds__(256)
sk_rescale01_3d_kernel(const uint16_t* __restrict__ c, DstT* __restrict__ dst, int64_t dsn, int64_t dsd, int64_t dsh,
                       int d, int h, int w, int tiles_x, const SkRange* __restrict__ ranges) {
    const int row = blockIdx.x / tiles_x;
    const int x = (blockIdx.x - row * tiles_x) * 256 + threadIdx.x;
    if (x >= w) return;
    const int vz = row / h, y = row - vz * h;
    const int n = vz / d, z = vz - n * d;
    dst[(int64_t)n * dsn + z * dsd + y * dsh + x] = sk_rescale01_value<DstT, F32MATH>(c[(int64_t)row * w + x], ranges[n]);
}

template <typename T>
static int sk_adapthist3d_launch(const T* src, void* dst, int src_dtype, int dst_dtype, int64_t n, const SkAdapt3Args& a,
                                 int cs, int64_t dsn, int64_t dsd, int64_t dsh, SkRange* rin, SkRange* rout,
                                 uint16_t* tables, uint16_t* maps, uint16_t* cvol, cudaStream_t st) {
    const int rpb = 8;
    sk_minmax3d_kernel<T><<<dim3((unsigned)ceil_div(a.d * a.h, rpb), (unsigned)n), 256, 0, st>>>(src, a, rpb, rin);
    if constexpr (sizeof(T) != 4) {
        const int ncodes = sizeof(T) == 1 ? 256 : 65536;
        sk_bin_table_kernel<T><<<dim3((unsigned)(ncodes / 256), (unsigned)n), 256, 0, st>>>(rin, a.bin_size, ncodes, tables);
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(n * a.nbz * a.nby * a.nbx * cs));
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = (size_t)a.nbins * sizeof(int);
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, sk_adapt3d_hist_kernel<T>, src, a, (const SkRange*)rin, (const uint16_t*)tables, maps);
    if (e != cudaSuccess) return (int)e;
    const int tiles_x = ceil_div(a.w, 32), tiles_y = ceil_div(a.h, 32);
    sk_adapt3d_apply_kernel<T><<<(unsigned)(n * a.d * tiles_y * tiles_x), 256, 0, st>>>(src, a, tiles_x, tiles_y, rin, tables, maps,
                                                                                       cvol, rout);
    const int rx = ceil_div(a.w, 256);
    const unsigned gres = (unsigned)(n * a.d * a.h * rx);
    const bool f32 = src_dtype == MIE_F32;
    if (dst_dtype == MIE_F32) {
        if (f32) sk_rescale01_3d_kernel<float, true><<<gres, 256, 0, st>>>(cvol, (float*)dst, dsn, dsd, dsh, a.d, a.h, a.w, rx, rout);
        else sk_rescale01_3d_kernel<float, false><<<gres, 256, 0, st>>>(cvol, (float*)dst, dsn, dsd, dsh, a.d, a.h, a.w, rx, rout);
    } else {
        if (f32) sk_rescale01_3d_kernel<double, true><<<gres, 256, 0, st>>>(cvol, (double*)dst, dsn, dsd, dsh, a.d, a.h, a.w, rx, rout);
        else sk_rescale01_3d_kernel<double, false><<<gres, 256, 0, st>>>(cvol, (double*)dst, dsn, dsd, dsh, a.d, a.h, a.w, rx, rout);
    }
    return check_launch();
}

// ---------------------------------------------------------------- equalize_hist (integer images)
template <typename T>
__global__ void __launch_bounds__(256)
sk_eqhist_count_kernel(const T* __restrict__ src, int64_t ssn, int64_t ssh, int h, int w, int rows_per_block,
                       const SkRange* __restrict__ ranges, unsigned* __restrict__ hist, int bins_cap) {
    const int64_t n = blockIdx.y;
    const int vmin = ranges[n].mn;
    unsigned* hh = hist + n * bins_cap;
    const int y0 = blockIdx.x * rows_per_block, y1 = min(y0 + rows_per_block, h);
    for (int y = y0; y < y1; ++y) {
        const T* row = src + n * ssn + (int64_t)y * ssh;
        for (int x = threadIdx.x; x < w; x += 256) atomicAdd(&hh[(int)row[x] - vmin], 1u);
    }
}
// in-place inclusive prefix sum of hist[0 .. vmax - vmin] (one block per image)
__global__ void __launch_bounds__(1024)
sk_eqhist_scan_kernel(unsigned* __restrict__ hist, int bins_cap, const SkRange* __restrict__ ranges) {
    __shared__ unsigned s_part[1024];
    const int64_t n = blockIdx.x;
    unsigned* hh = hist + n * bins_cap;
    const int nb = ranges[n].mx - ranges[n].mn + 1;
    const int per = (nb + 1023) / 1024;
    const int b0 = threadIdx.x * per, b1 = min(b0 + per, nb);
    unsigned s = 0;
    for (int b = b0; b < b1; ++b) s += hh[b];
    s_part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const unsigned t = threadIdx.x >= o ? s_part[threadIdx.x - o] : 0u;
        __syncthreads();
        s_part[threadIdx.x] += t;
        __syncthreads();
    }
    unsigned run = threadIdx.x ? s_part[threadIdx.x - 1] : 0u;
    for (int b = b0; b < b1; ++b) { run += hh[b]; hh[b] = run; }
}
template <typename T, typename DstT>
__global__ void __launch_bounds__(256)
sk_eqhist_apply_kernel(const T* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                       int h, int w, const SkRange* __restrict__ ranges, const unsigned* __restrict__ hist, int bins_cap) {
    const int64_t n = blockIdx.z;
    const int x = blockIdx.x * 256 + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const SkRange r = ranges[n];
    const unsigned* hh = hist + n * bins_cap;
    const double total = (double)hh[r.mx - r.mn];
    const int v = (int)src[n * ssn + (int64_t)y * ssh + x];
    dst[n * dsn + (int64_t)y * dsh + x] = (DstT)__ddiv_rn((double)hh[v - r.mn], total);
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_sk_adapthist_workspace_bytes(int64_t n, int h, int w, int kr, int kc, int nbins) {
    if (n <= 0 || h <= 0 || w <= 0 || kr <= 0 || kc <= 0 || nbins <= 0) return 0;
    const size_t nbr = (size_t)ceil_div(h, kr), nbc = (size_t)ceil_div(w, kc);
    return align256((size_t)n * 2 * sizeof(SkRange)) + align256((size_t)n * nbr * nbc * nbins * sizeof(uint16_t)) +
           align256((size_t)n * h * w * sizeof(uint16_t));
}

int mie_sk_equalize_adapthist(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                              int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                              int kr, int kc, double clip_limit, int nbins, void* workspace, size_t workspace_bytes,
                              void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h}, n, h, w);
    if (rc) return rc;
    if (!valid_dtype(src_dtype) || (dst_dtype != MIE_F32 && dst_dtype != MIE_F64)) return MIE_E_DTYPE;
    if (kr <= 0 || kc <= 0) return MIE_E_KERNEL;
    if (nbins <= 0 || nbins > kSkMaxBins) return MIE_E_UNSUPPORTED;
    if ((int64_t)kr * kc > 2147483647LL || n > 65535) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < mie_sk_adapthist_workspace_bytes(n, h, w, kr, kc, nbins)) return MIE_E_WORKSPACE;
    SkAdaptArgs a;
    a.h = h; a.w = w; a.kr = kr; a.kc = kc; a.nbr = ceil_div(h, kr); a.nbc = ceil_div(w, kc); a.nbins = nbins;
    a.bin_size = 1 + kSkGray / nbins;
    const int64_t elems = (int64_t)kr * kc;
    if (clip_limit > 0.0) {
        double c = clip_limit * (double)elems;
        if (c < 1.0) c = 1.0;
        a.clim = c >= 2147483647.0 ? 2147483647 : (int)c;
    } else {
        a.clim = 65535;   // np.iinfo(uint16).max: upstream's "do not clip"
    }
    a.scale = 16383.0 / (double)elems;
    if (a.nbr > 65535 || a.nbc > 2147483647) return MIE_E_SHAPE;
    uint8_t* ws = (uint8_t*)workspace;
    SkRange* rin = (SkRange*)ws;
    SkRange* rout = rin + n;
    uint16_t* maps = (uint16_t*)(ws + align256((size_t)n * 2 * sizeof(SkRange)));
    uint16_t* cplane = (uint16_t*)((uint8_t*)maps + align256((size_t)n * a.nbr * a.nbc * nbins * sizeof(uint16_t)));
    sk_init_ranges_kernel<<<(unsigned)((2 * n + 255) / 256), 256, 0, st>>>(rin, 2 * n);
    const int rpb = 8;
    const dim3 gmm((unsigned)ceil_div(h, rpb), (unsigned)n);
    const dim3 ghist((unsigned)a.nbc, (unsigned)a.nbr, (unsigned)n);
    const dim3 gapp((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 32), (unsigned)n);
    const size_t smem = (size_t)nbins * sizeof(int);
    MIE_DISPATCH_SRC(src_dtype, {
        sk_minmax_kernel<SrcT><<<gmm, 256, 0, st>>>((const SrcT*)src, src_stride_n, src_stride_h, h, w, rpb, rin);
        sk_adapt_hist_kernel<SrcT><<<ghist, 256, smem, st>>>((const SrcT*)src, src_stride_n, src_stride_h, a, rin, maps);
        sk_adapt_apply_kernel<SrcT><<<gapp, 256, 0, st>>>((const SrcT*)src, src_stride_n, src_stride_h, a, rin, maps, cplane, rout);
    });
    const dim3 gres((unsigned)ceil_div(w, 256), (unsigned)h, (unsigned)n);
    if (h > 65535) return MIE_E_SHAPE;
    if (src_dtype == MIE_F32) {
        if (dst_dtype == MIE_F32) sk_rescale01_kernel<float, true><<<gres, 256, 0, st>>>(cplane, (float*)dst, dst_stride_n, dst_stride_h, h, w, rout);
        else sk_rescale01_kernel<double, true><<<gres, 256, 0, st>>>(cplane, (double*)dst, dst_stride_n, dst_stride_h, h, w, rout);
    } else {
        if (dst_dtype == MIE_F32) sk_rescale01_kernel<float, false><<<gres, 256, 0, st>>>(cplane, (float*)dst, dst_stride_n, dst_stride_h, h, w, rout);
        else sk_rescale01_kernel<double, false><<<gres, 256, 0, st>>>(cplane, (double*)dst, dst_stride_n, dst_stride_h, h, w, rout);
    }
    return check_launch();
}

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

size_t mie_sk_adapthist3d_workspace_bytes(int64_t n, int d, int h, int w, int kd, int kr, int kc, int nbins) {
    if (n <= 0 || d <= 0 || h <= 0 || w <= 0 || kd <= 0 || kr <= 0 || kc <= 0 || nbins <= 0) return 0;
    const size_t regions = (size_t)ceil_div64(d, kd) * (size_t)ceil_div64(h, kr) * (size_t)ceil_div64(w, kc);
    return align256((size_t)n * 2 * sizeof(SkRange)) + align256((size_t)n * kSkCodes * sizeof(uint16_t)) +
           align256((size_t)n * regions * nbins * sizeof(uint16_t)) + align256((size_t)n * d * h * w * sizeof(uint16_t));
}

int mie_sk_equalize_adapthist3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                                int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                                int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                                int kd, int kr, int kc, double clip_limit, int nbins, void* workspace, size_t workspace_bytes,
                                void* stream) {
    const int rc = check_volumes({src, src_dtype, src_stride_n, src_stride_h}, src_stride_d,
                                 {dst, dst_dtype, dst_stride_n, dst_stride_h}, dst_stride_d, n, d, h, w);
    if (rc) return rc;
    if (!valid_dtype(src_dtype) || (dst_dtype != MIE_F32 && dst_dtype != MIE_F64)) return MIE_E_DTYPE;
    if (kd <= 0 || kr <= 0 || kc <= 0) return MIE_E_KERNEL;
    if (nbins <= 0 || nbins > kSkMaxBins) return MIE_E_UNSUPPORTED;
    const int64_t elems = (int64_t)kd * kr * kc;
    if (elems > INT_MAX || n > 65535) return MIE_E_SHAPE;
    // every index below stays in int: rows of a volume, padded coordinates, flat grids
    if ((int64_t)d * h > INT_MAX || (int64_t)d + kd > INT_MAX || (int64_t)h + kr > INT_MAX || (int64_t)w + kc > INT_MAX)
        return MIE_E_SHAPE;
    SkAdapt3Args a;
    a.d = d; a.h = h; a.w = w; a.kd = kd; a.kr = kr; a.kc = kc;
    a.nbz = ceil_div(d, kd); a.nby = ceil_div(h, kr); a.nbx = ceil_div(w, kc);
    a.nbins = nbins;
    a.bin_size = 1 + kSkGray / nbins;
    if (clip_limit > 0.0) {
        double c = clip_limit * (double)elems;
        if (c < 1.0) c = 1.0;
        a.clim = c >= 2147483647.0 ? 2147483647 : (int)c;
    } else {
        a.clim = 65535;   // np.iinfo(uint16).max: upstream's "do not clip" (ASSUMED, as in 2-D)
    }
    a.scale = 16383.0 / (double)elems;
    a.ssn = src_stride_n; a.ssd = src_stride_d; a.ssh = src_stride_h;
    // cluster size from the region's size: up to 8 CTAs, each counting >= kSkVoxelsPerCta voxels and >= 1 row
    const int rows = kd * kr;
    int cs = 1;
    while (cs < 8 && elems > (int64_t)cs * kSkVoxelsPerCta && rows >= 2 * cs) cs <<= 1;
    a.rows_per_cta = ceil_div(rows, cs);
    a.tpr = 32;
    while (a.tpr > 1 && a.tpr / 2 >= kc) a.tpr >>= 1;
    const int64_t regions = (int64_t)a.nbz * a.nby * a.nbx;
    if (n * regions * cs > INT_MAX || n * d * ceil_div64(h, 32) * ceil_div64(w, 32) > INT_MAX ||
        n * d * h * ceil_div64(w, 256) > INT_MAX)
        return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < mie_sk_adapthist3d_workspace_bytes(n, d, h, w, kd, kr, kc, nbins)) return MIE_E_WORKSPACE;
    uint8_t* ws = (uint8_t*)workspace;
    SkRange* rin = (SkRange*)ws;
    SkRange* rout = rin + n;
    ws += align256((size_t)n * 2 * sizeof(SkRange));
    uint16_t* tables = (uint16_t*)ws;
    ws += align256((size_t)n * kSkCodes * sizeof(uint16_t));
    uint16_t* maps = (uint16_t*)ws;
    ws += align256((size_t)n * regions * nbins * sizeof(uint16_t));
    uint16_t* cvol = (uint16_t*)ws;
    cudaStream_t st = (cudaStream_t)stream;
    sk_init_ranges_kernel<<<(unsigned)((2 * n + 255) / 256), 256, 0, st>>>(rin, 2 * n);
    MIE_DISPATCH_SRC(src_dtype, {
        return sk_adapthist3d_launch<SrcT>((const SrcT*)src, dst, src_dtype, dst_dtype, n, a, cs, dst_stride_n, dst_stride_d,
                                           dst_stride_h, rin, rout, tables, maps, cvol, st);
    });
    return MIE_OK;
}

size_t mie_sk_equalize_hist_workspace_bytes(int64_t n, int src_dtype) {
    if (n <= 0) return 0;
    const size_t cap = src_dtype == MIE_U8 ? 256 : 65536;
    return align256((size_t)n * sizeof(SkRange)) + (size_t)n * cap * sizeof(unsigned);
}

int mie_sk_equalize_hist(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                         int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                         void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h}, n, h, w);
    if (rc) return rc;
    if (src_dtype != MIE_U8 && src_dtype != MIE_U16 && src_dtype != MIE_I16) return MIE_E_DTYPE;
    if (dst_dtype != MIE_F32 && dst_dtype != MIE_F64) return MIE_E_DTYPE;
    if (n > 65535 || h > 65535) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < mie_sk_equalize_hist_workspace_bytes(n, src_dtype)) return MIE_E_WORKSPACE;
    const int cap = src_dtype == MIE_U8 ? 256 : 65536;
    SkRange* rin = (SkRange*)workspace;
    unsigned* hist = (unsigned*)((uint8_t*)workspace + align256((size_t)n * sizeof(SkRange)));
    sk_init_ranges_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rin, n);
    cudaError_t e = cudaMemsetAsync(hist, 0, (size_t)n * cap * sizeof(unsigned), st);
    if (e != cudaSuccess) return (int)e;
    const int rpb = 8;
    const dim3 gmm((unsigned)ceil_div(h, rpb), (unsigned)n);
    const dim3 gapp((unsigned)ceil_div(w, 256), (unsigned)h, (unsigned)n);
#define MIE_SK_EQ(T_)                                                                                                  \
    sk_minmax_kernel<T_><<<gmm, 256, 0, st>>>((const T_*)src, src_stride_n, src_stride_h, h, w, rpb, rin);              \
    sk_eqhist_count_kernel<T_><<<gmm, 256, 0, st>>>((const T_*)src, src_stride_n, src_stride_h, h, w, rpb, rin, hist, cap); \
    sk_eqhist_scan_kernel<<<(unsigned)n, 1024, 0, st>>>(hist, cap, rin);                                               \
    if (dst_dtype == MIE_F32)                                                                                          \
        sk_eqhist_apply_kernel<T_, float><<<gapp, 256, 0, st>>>((const T_*)src, (float*)dst, src_stride_n, src_stride_h,   \
                                                                 dst_stride_n, dst_stride_h, h, w, rin, hist, cap);    \
    else                                                                                                               \
        sk_eqhist_apply_kernel<T_, double><<<gapp, 256, 0, st>>>((const T_*)src, (double*)dst, src_stride_n, src_stride_h, \
                                                                  dst_stride_n, dst_stride_h, h, w, rin, hist, cap)
    switch (src_dtype) {
        case MIE_U8: MIE_SK_EQ(uint8_t); break;
        case MIE_U16: MIE_SK_EQ(uint16_t); break;
        default: MIE_SK_EQ(int16_t); break;
    }
#undef MIE_SK_EQ
    return check_launch();
}

}  // extern "C"
