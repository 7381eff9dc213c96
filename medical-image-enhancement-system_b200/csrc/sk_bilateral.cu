// sk_bilateral.cu — skimage.restoration.denoise_bilateral on single-channel planes (SURVEY.md §8(f) F3, Appendix B4;
// reference pyproject.toml:12).  Not kornia's bilateral_blur (bilateral.cu): the colour weight comes from a LUT of
// `bins` entries over the image's dynamic range, indexed by min(int(|c - v| * bins / max_value), bins - 1); the spatial
// weight from a win x win Gaussian LUT; the default border is mode='constant' (outside pixels have value cval and DO take
// part in the weighted mean); images with negative values are shifted by their minimum and shifted back.
//
// RECALLED semantics; the kernel follows oracle/mie_oracle.c:orc_sk_bilateral (bit-identical to the numpy twin
// oracle/skimage_twin.py): float64 arithmetic in upstream's order with explicit __d*_rn (no fma contraction).  Both LUTs
// are built by the caller exactly as upstream builds them in Python (numpy exp) and passed in as device arrays.
#include "mie_common.cuh"

namespace mie {

// mode: 0 constant, 1 edge, 2 symmetric, 3 reflect, 4 wrap (numpy.pad names)
__device__ __forceinline__ int skb_border(int i, int n, int mode) {
    if (i >= 0 && i < n) return i;
    switch (mode) {
        case 1: return i < 0 ? 0 : n - 1;
        case 2: { const int p = 2 * n; int m = i % p; if (m < 0) m += p; return m < n ? m : p - 1 - m; }
        case 3: { if (n == 1) return 0; const int p = 2 * (n - 1); int m = i % p; if (m < 0) m += p; return m < n ? m : p - m; }
        case 4: { int m = i % n; return m < 0 ? m + n : m; }
        default: return -1;
    }
}

// 32 x 32 output pixels per block; the haloed tile is staged as float64 in shared memory, followed by the colour LUT
// when it fits (LUT_SMEM), which it does for the default 10 000 bins.
template <typename T, typename DstT, bool LUT_SMEM>
__global__ void __launch_bounds__(256)
sk_bilateral_kernel(const T* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                    int h, int w, int win, int bins, int mode, double cval, const double* __restrict__ color_luts,
                    const double* __restrict__ range_lut, const int* __restrict__ ranges) {
    extern __shared__ __align__(16) double s_mem[];
    const int ext = (win - 1) / 2, ew = 32 + 2 * ext, pitch = ew | 1;
    double* s_tile = s_mem;
    double* s_rng = s_tile + (32 + 2 * ext) * pitch;
    double* s_col = s_rng + win * win;
    const int64_t n = blockIdx.z;
    const int tx0 = blockIdx.x * 32, ty0 = blockIdx.y * 32;
    const int vmin = ranges[2 * n], vmax = ranges[2 * n + 1];
    const double min_value = skb_as_float<T>(vmin);
    double max_value = skb_as_float<T>(vmax);
    const bool shift = min_value < 0.0;
    if (shift) max_value = __dsub_rn(max_value, min_value);
    const T* plane = src + n * ssn;
    for (int i = threadIdx.x; i < ew * ew; i += 256) {
        const int r = i / ew, c = i - r * ew;
        const int sy = skb_border(ty0 - ext + r, h, mode), sx = skb_border(tx0 - ext + c, w, mode);
        double v;
        if (sy < 0 || sx < 0) v = cval;
        else { v = skb_as_float<T>((int)plane[(int64_t)sy * ssh + sx]); if (shift) v = __dsub_rn(v, min_value); }
        s_tile[r * pitch + c] = v;
    }
    for (int i = threadIdx.x; i < win * win; i += 256) s_rng[i] = range_lut[i];
    const double* col = color_luts + n * (int64_t)bins;
    if (LUT_SMEM) {
        for (int i = threadIdx.x; i < bins; i += 256) s_col[i] = col[i];
        col = s_col;
    }
    __syncthreads();
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    const int x = tx0 + lx;
    if (x >= w) return;
    if (vmin == vmax) {   // flat image: upstream returns the float image unchanged
        for (int k = 0; k < 4; ++k) {
            const int y = ty0 + ly0 + 8 * k;
            if (y < h) dst[n * dsn + (int64_t)y * dsh + x] = (DstT)min_value;
        }
        return;
    }
    const double dist_scale = __ddiv_rn((double)bins, max_value);
    const long long last = bins - 1;
    for (int k = 0; k < 4; ++k) {
        const int ly = ly0 + 8 * k, y = ty0 + ly;
        if (y >= h) break;
        const double centre = s_tile[(ly + ext) * pitch + lx + ext];
        double total_v = 0.0, total_w = 0.0;
        for (int kr = 0; kr < win; ++kr) {
            const double* trow = s_tile + (ly + kr) * pitch + lx;
            const double* rrow = s_rng + kr * win;
            for (int kc = 0; kc < win; ++kc) {
                const double v = trow[kc];
                const double t = __dsub_rn(centre, v);
                const double dist = __dsqrt_rn(__dmul_rn(t, t));
                long long b = (long long)__dmul_rn(dist, dist_scale);
                b = b > last ? last : b;
                const double weight = __dmul_rn(rrow[kc], LUT_SMEM ? col[b] : __ldg(col + b));
                total_v = __dadd_rn(total_v, __dmul_rn(v, weight));
                total_w = __dadd_rn(total_w, weight);
            }
        }
        double o = __ddiv_rn(total_v, total_w);
        if (shift) o = __dadd_rn(o, min_value);
        dst[n * dsn + (int64_t)y * dsh + x] = (DstT)o;
    }
}

}  // namespace mie

using namespace mie;

extern "C" int mie_sk_denoise_bilateral(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                                        int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n,
                                        int64_t dst_stride_h, int win_size, int bins, int mode, double cval,
                                        const double* color_luts, const double* range_lut, const int* ranges,
                                        void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h}, n, h, w);
    if (rc) return rc;
    if (src_dtype != MIE_U8 && src_dtype != MIE_U16 && src_dtype != MIE_I16) return MIE_E_DTYPE;
    if (dst_dtype != MIE_F32 && dst_dtype != MIE_F64) return MIE_E_DTYPE;
    if (win_size <= 0 || !(win_size & 1) || win_size > 63) return MIE_E_KERNEL;
    if (bins <= 0) return MIE_E_SHAPE;
    if (mode < 0 || mode > 4) return MIE_E_BORDER;
    if (n > 65535 || ceil_div(h, 32) > 65535) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (!color_luts || !range_lut || !ranges) return MIE_E_NULL;
    const int ext = (win_size - 1) / 2, ew = 32 + 2 * ext;
    const size_t base = ((size_t)ew * (ew | 1) + (size_t)win_size * win_size) * sizeof(double);
    const bool lut_smem = base + (size_t)bins * sizeof(double) <= 200 * 1024;
    const size_t smem = base + (lut_smem ? (size_t)bins * sizeof(double) : 0);
    if (smem > 200 * 1024) return MIE_E_KERNEL;
    const dim3 grid((unsigned)ceil_div(w, 32), (unsigned)ceil_div(h, 32), (unsigned)n);
#define MIE_SKB(T_, D_)                                                                                              \
    do {                                                                                                             \
        if (lut_smem) {                                                                                              \
            MIE_ENSURE_SMEM((sk_bilateral_kernel<T_, D_, true>), 200 * 1024);                                        \
            sk_bilateral_kernel<T_, D_, true><<<grid, 256, smem, st>>>((const T_*)src, (D_*)dst, src_stride_n, src_stride_h, \
                dst_stride_n, dst_stride_h, h, w, win_size, bins, mode, cval, color_luts, range_lut, ranges);        \
        } else {                                                                                                     \
            MIE_ENSURE_SMEM((sk_bilateral_kernel<T_, D_, false>), 200 * 1024);                                       \
            sk_bilateral_kernel<T_, D_, false><<<grid, 256, smem, st>>>((const T_*)src, (D_*)dst, src_stride_n, src_stride_h, \
                dst_stride_n, dst_stride_h, h, w, win_size, bins, mode, cval, color_luts, range_lut, ranges);        \
        }                                                                                                            \
    } while (0)
    switch (src_dtype) {
        case MIE_U8: if (dst_dtype == MIE_F32) MIE_SKB(uint8_t, float); else MIE_SKB(uint8_t, double); break;
        case MIE_U16: if (dst_dtype == MIE_F32) MIE_SKB(uint16_t, float); else MIE_SKB(uint16_t, double); break;
        default: if (dst_dtype == MIE_F32) MIE_SKB(int16_t, float); else MIE_SKB(int16_t, double); break;
    }
#undef MIE_SKB
    return check_launch();
}
