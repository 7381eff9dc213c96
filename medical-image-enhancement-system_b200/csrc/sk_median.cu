// sk_median.cu — skimage.filters.median with any footprint (scipy.ndimage.median_filter(x, footprint=fp, mode, cval)) on
// planes and whole volumes (SURVEY.md §8(a) A6; reference pyproject.toml:12).  Pure selection: element count / 2 of the
// sorted window, so every output is one of the window's samples (or the cval) and equals scipy's value.
//
// One kernel serves both entry points: a plane is a volume of depth 1.  A block of 256 threads owns 4 outputs per
// thread: 32 x 8 x 4 (z) of a volume, or 32 x 32 of a plane.  It stages the haloed tile once in shared memory as
// unsigned ORDERED keys (u8 / u16 as they are, i16 ^ 0x8000, f32 bits with the sign flipped or every bit flipped when
// negative), with the borders resolved while staging (border_index; 'constant' stores the caller's cval key), and
// decodes the footprint's bit mask into a list of tile offsets next to it.  Selection is MSB-first radix counting: for
// bit b, count the samples below res | 1 << b, and keep that bit when the count is <= rank.  The final res is the
// largest key with at most `rank` samples below it, i.e. the rank-th smallest.  8, 16 or 32 passes, one code path for
// every dtype; the 4 outputs of a thread share each offset load.
#include "mie_common.cuh"

namespace mie {

constexpr int kSkmOut = 4;                                          // outputs per thread
constexpr int kSkmCells = MIE_SK_MEDIAN3D_MAX_EXTENT * MIE_SK_MEDIAN3D_MAX_EXTENT * MIE_SK_MEDIAN3D_MAX_EXTENT;
constexpr int kSkmWords = (kSkmCells + 31) / 32;
static_assert(MIE_SK_MEDIAN_MAX_EXTENT * MIE_SK_MEDIAN_MAX_EXTENT <= kSkmCells, "2-D footprints share the 3-D mask");

// The footprint travels in the kernel parameters (no __constant__ symbol, no copy): row-major bit mask over
// (fz, fy, fx) plus the number of set cells before each word, so that every word decodes independently.
struct SkmFootprint {
    uint32_t mask[kSkmWords];
    uint16_t first[kSkmWords];
    int fz, fy, fx, count;
};

template <typename T> struct SkmKey;
template <> struct SkmKey<uint8_t> {
    using K = uint8_t;
    static __host__ __device__ __forceinline__ K to(uint8_t v) { return v; }
    static __device__ __forceinline__ uint8_t from(uint32_t k) { return (uint8_t)k; }
};
template <> struct SkmKey<uint16_t> {
    using K = uint16_t;
    static __host__ __device__ __forceinline__ K to(uint16_t v) { return v; }
    static __device__ __forceinline__ uint16_t from(uint32_t k) { return (uint16_t)k; }
};
template <> struct SkmKey<int16_t> {
    using K = uint16_t;
    static __host__ __device__ __forceinline__ K to(int16_t v) { return (uint16_t)((uint16_t)v ^ 0x8000u); }
    static __device__ __forceinline__ int16_t from(uint32_t k) { return (int16_t)(uint16_t)(k ^ 0x8000u); }
};
template <> struct SkmKey<float> {
    using K = uint32_t;
    static __host__ __device__ __forceinline__ K to(float v) {
        uint32_t u;
        memcpy(&u, &v, 4);
        return u ^ ((uint32_t)((int32_t)u >> 31) | 0x80000000u);
    }
    static __device__ __forceinline__ float from(uint32_t k) {
        return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
    }
};

__host__ __device__ __forceinline__ size_t skm_keys_bytes(int tile, int esz) { return ((size_t)tile * esz + 15) & ~(size_t)15; }

template <typename T>
__global__ void __launch_bounds__(256)
sk_median_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t n, int d, int h, int w, int64_t ssn,
                 int64_t ssd, int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, const SkmFootprint fp, int rz,
                 int tiles_x, int tiles_y, int mode, uint32_t cval_key) {
    using Key = SkmKey<T>;
    using K = typename Key::K;
    constexpr int kBits = 8 * (int)sizeof(K);
    extern __shared__ __align__(16) unsigned char s_mem[];
    const int ry = kSkmOut / rz;
    const int tsx = 32 + fp.fx - 1, tsy = 8 * ry + fp.fy - 1, tsz = rz + fp.fz - 1;
    const int plane = tsx * tsy, tile = plane * tsz;
    K* s_key = reinterpret_cast<K*>(s_mem);
    uint16_t* s_off = reinterpret_cast<uint16_t*>(s_mem + skm_keys_bytes(tile, sizeof(K)));

    const int fyx = fp.fy * fp.fx, nwords = (fp.fz * fyx + 31) / 32;
    for (int wd = threadIdx.x; wd < nwords; wd += blockDim.x) {
        uint32_t m = fp.mask[wd];
        int pos = fp.first[wd];
        while (m) {
            const int c = wd * 32 + __ffs(m) - 1;
            m &= m - 1;
            const int cz = c / fyx, rem = c - cz * fyx, cy = rem / fp.fx, cx = rem - cy * fp.fx;
            s_off[pos++] = (uint16_t)((cz * tsy + cy) * tsx + cx);
        }
    }

    const int bx = (int)(blockIdx.x % (unsigned)tiles_x), rest = (int)(blockIdx.x / (unsigned)tiles_x);
    const int by = rest % tiles_y, bz = rest / tiles_y;
    const int x0 = bx * 32, y0 = by * 8 * ry, z0 = bz * rz;
    const int oz = z0 - fp.fz / 2, oy = y0 - fp.fy / 2, ox = x0 - fp.fx / 2;   // the footprint's centre: extent // 2
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;
    int base[kSkmOut];
#pragma unroll
    for (int r = 0; r < kSkmOut; ++r) base[r] = ((r % rz) * tsy + ly + 8 * (r / rz)) * tsx + lx;
    const uint32_t rank = (uint32_t)(fp.count >> 1);

    for (int64_t img = blockIdx.y; img < n; img += gridDim.y) {
        const T* s = src + img * ssn;
        __syncthreads();   // the previous image's selection has finished with the tile (and s_off is complete)
        for (int i = threadIdx.x; i < tile; i += blockDim.x) {
            const int lz = i / plane, ri = i - lz * plane, lyy = ri / tsx, lxx = ri - lyy * tsx;
            const int gz = border_index(oz + lz, d, mode), gy = border_index(oy + lyy, h, mode),
                      gx = border_index(ox + lxx, w, mode);
            K k = (K)cval_key;
            if ((gz | gy | gx) >= 0) k = Key::to(s[gz * ssd + gy * ssh + gx]);
            s_key[i] = k;
        }
        __syncthreads();
        uint32_t res[kSkmOut];
#pragma unroll
        for (int r = 0; r < kSkmOut; ++r) res[r] = 0;
        for (int b = kBits - 1; b >= 0; --b) {
            uint32_t piv[kSkmOut], cnt[kSkmOut];
#pragma unroll
            for (int r = 0; r < kSkmOut; ++r) { piv[r] = res[r] | (1u << b); cnt[r] = 0; }
#pragma unroll 4
            for (int j = 0; j < fp.count; ++j) {
                const int o = s_off[j];
#pragma unroll
                for (int r = 0; r < kSkmOut; ++r) cnt[r] += (uint32_t)s_key[base[r] + o] < piv[r] ? 1u : 0u;
            }
#pragma unroll
            for (int r = 0; r < kSkmOut; ++r) res[r] = cnt[r] <= rank ? piv[r] : res[r];
        }
        const int x = x0 + lx;
#pragma unroll
        for (int r = 0; r < kSkmOut; ++r) {
            const int z = z0 + r % rz, y = y0 + ly + 8 * (r / rz);
            if (x < w && y < h && z < d) dst[img * dsn + z * dsd + y * dsh + x] = Key::from(res[r]);
        }
    }
}

// The caller's cval as a key of the image dtype: it must be exactly representable (integers in range, or the float32
// it already is; NaN is accepted for float32, whose results are unspecified as for NaN pixels).
inline int skm_cval_key(int dtype, double cval, uint32_t* key) {
    switch (dtype) {
        case MIE_U8:
            if (!(cval >= 0.0 && cval <= 255.0 && cval == (double)(int)cval)) return MIE_E_RANGE;
            *key = SkmKey<uint8_t>::to((uint8_t)(int)cval);
            return MIE_OK;
        case MIE_U16:
            if (!(cval >= 0.0 && cval <= 65535.0 && cval == (double)(int)cval)) return MIE_E_RANGE;
            *key = SkmKey<uint16_t>::to((uint16_t)(int)cval);
            return MIE_OK;
        case MIE_I16:
            if (!(cval >= -32768.0 && cval <= 32767.0 && cval == (double)(int)cval)) return MIE_E_RANGE;
            *key = SkmKey<int16_t>::to((int16_t)(int)cval);
            return MIE_OK;
        default: {
            const float f = (float)cval;
            if (cval == cval && (double)f != cval) return MIE_E_RANGE;
            *key = SkmKey<float>::to(f);
            return MIE_OK;
        }
    }
}

inline int skm_footprint(const uint8_t* footprint, int fz, int fy, int fx, int max_extent, SkmFootprint* fp) {
    if (fz < 1 || fy < 1 || fx < 1 || fz > max_extent || fy > max_extent || fx > max_extent) return MIE_E_KERNEL;
    if (!footprint) return MIE_E_NULL;
    memset(fp, 0, sizeof(*fp));
    fp->fz = fz; fp->fy = fy; fp->fx = fx;
    const int cells = fz * fy * fx;
    for (int c = 0; c < cells; ++c)
        if (footprint[c]) fp->mask[c >> 5] |= 1u << (c & 31);
    int count = 0;
    for (int wd = 0; wd < kSkmWords; ++wd) {
        fp->first[wd] = (uint16_t)count;
        count += __builtin_popcount(fp->mask[wd]);
    }
    fp->count = count;
    return count ? MIE_OK : MIE_E_KERNEL;
}

template <typename T>
int skm_launch(const void* src, void* dst, int64_t n, int d, int h, int w, int64_t ssn, int64_t ssd, int64_t ssh,
               int64_t dsn, int64_t dsd, int64_t dsh, const SkmFootprint& fp, int mode, uint32_t cval_key,
               cudaStream_t st) {
    const int rz = d > 1 ? kSkmOut : 1, ry = kSkmOut / rz;
    const int64_t tiles_x = ceil_div(w, 32), tiles_y = (h + 8 * ry - 1) / (8 * ry), tiles_z = (d + rz - 1) / rz;
    const int64_t blocks = tiles_x * tiles_y * tiles_z;
    if (blocks > 0x7fffffff) return MIE_E_SHAPE;
    const int tile = (32 + fp.fx - 1) * (8 * ry + fp.fy - 1) * (rz + fp.fz - 1);
    const size_t smem = skm_keys_bytes(tile, sizeof(typename SkmKey<T>::K)) + (size_t)fp.count * sizeof(uint16_t);
    MIE_ENSURE_SMEM(sk_median_kernel<T>, 227 * 1024);
    const dim3 grid((unsigned)blocks, (unsigned)(n < 65535 ? n : 65535));
    sk_median_kernel<T><<<grid, 256, smem, st>>>((const T*)src, (T*)dst, n, d, h, w, ssn, ssd, ssh, dsn, dsd, dsh, fp, rz,
                                                 (int)tiles_x, (int)tiles_y, mode, cval_key);
    return check_launch();
}

inline int skm_run(const void* src, void* dst, int dtype, int64_t n, int d, int h, int w, int64_t ssn, int64_t ssd,
                   int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, const uint8_t* footprint, int fz, int fy, int fx,
                   int max_extent, int border, double cval, void* stream) {
    SkmFootprint fp;
    int rc = skm_footprint(footprint, fz, fy, fx, max_extent, &fp);
    if (rc) return rc;
    if (border < MIE_BORDER_CONSTANT || border > MIE_BORDER_SYMMETRIC) return MIE_E_BORDER;
    uint32_t key = 0;
    if ((rc = skm_cval_key(dtype, cval, &key))) return rc;
    if (n == 0) return MIE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    MIE_DISPATCH_SRC(dtype, return skm_launch<SrcT>(src, dst, n, d, h, w, ssn, ssd, ssh, dsn, dsd, dsh, fp, border, key,
                                                    st));
    return MIE_OK;
}

}  // namespace mie

using namespace mie;

extern "C" int mie_sk_median(const void* src, void* dst, int dtype, int64_t n, int h, int w, int64_t src_stride_n,
                             int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h, const uint8_t* footprint,
                             int fy, int fx, int border, double cval, void* stream) {
    if (!valid_dtype(dtype)) return MIE_E_DTYPE;
    int rc = check_planes({src, dtype, src_stride_n, src_stride_h}, {dst, dtype, dst_stride_n, dst_stride_h}, n, h, w);
    if (rc) return rc;
    return skm_run(src, dst, dtype, n, 1, h, w, src_stride_n, 0, src_stride_h, dst_stride_n, 0, dst_stride_h, footprint,
                   1, fy, fx, MIE_SK_MEDIAN_MAX_EXTENT, border, cval, stream);
}

extern "C" int mie_sk_median3d(const void* src, void* dst, int dtype, int64_t n, int d, int h, int w,
                               int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h, int64_t dst_stride_n,
                               int64_t dst_stride_d, int64_t dst_stride_h, const uint8_t* footprint, int fz, int fy,
                               int fx, int border, double cval, void* stream) {
    if (!valid_dtype(dtype)) return MIE_E_DTYPE;
    int rc = check_volumes({src, dtype, src_stride_n, src_stride_h}, src_stride_d, {dst, dtype, dst_stride_n, dst_stride_h},
                           dst_stride_d, n, d, h, w);
    if (rc) return rc;
    return skm_run(src, dst, dtype, n, d, h, w, src_stride_n, src_stride_d, src_stride_h, dst_stride_n, dst_stride_d,
                   dst_stride_h, footprint, fz, fy, fx, MIE_SK_MEDIAN3D_MAX_EXTENT, border, cval, stream);
}
