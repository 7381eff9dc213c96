// median.cu — 2-D K x K and 3-D 3x3x3 median filters (pure selection, bit-exact).
//
// Kernels, fastest first:
//   median3x3_packed_kernel / median5x5_packed_kernel  8 / 16-bit pixels, rows a multiple of 8 pixels: two pixels
//       per lane on min/max.{u,s}16x2, marching rows in registers, neighbours by shuffle, no shared memory;
//   median3x3_f32_kernel     float planes, rows a multiple of 4 pixels: the same marching schedule, one pixel per register;
//   median3d_direct_kernel   16-bit volumes of even width: sorted 9-lists of three planes in registers,
//       rank 13 of 27 by column sorts + pruning + merges;
//   median3d_packed_kernel   16-bit volumes of any width (planes staged in shared memory), same selection;
//   median2d_kernel<KY,KX> / median3d_kernel   every other size / dtype: shared-memory tiles, forgetful selection.
//
// mie_median2d replaces kornia.filters.median_blur (zero padding, lower median ==
// true median for odd window sizes) and skimage.filters.median on 2-D input
// ('nearest' border); SURVEY.md §8(a) A5.
// mie_median3d replaces skimage.filters.median on a volume ->
// scipy.ndimage.median_filter(footprint=ones((3,3,3)), mode='nearest'), rank
// 27//2 = 13 (site-packages/scipy/ndimage/_filters.py:1961-1962); §8(a) A6.
//
// Selection is done in registers with "forgetful selection": keep a working set
// of N/2+2 candidates, repeatedly drop its minimum and maximum (neither can be
// the median) and insert the next sample.  All indices are compile-time, so the
// whole network is min/max instructions on registers.

#include "mie_common.cuh"

#define MIE_HAVE_MEDIAN 1

namespace mie {

template <typename C>
__device__ __forceinline__ void cswap(C& a, C& b) {
    C lo = a < b ? a : b;
    C hi = a < b ? b : a;
    a = lo; b = hi;
}
template <>
__device__ __forceinline__ void cswap<int>(int& a, int& b) {
    int lo = min(a, b), hi = max(a, b);
    a = lo; b = hi;
}
template <>
__device__ __forceinline__ void cswap<float>(float& a, float& b) {
    float lo = fminf(a, b), hi = fmaxf(a, b);
    a = lo; b = hi;
}

// Moves the minimum of a[0..CNT) to a[0] and the maximum to a[CNT-1].
template <int CNT, typename C>
__device__ __forceinline__ void minmax_to_ends(C* a) {
#pragma unroll
    for (int i = 0; i < CNT / 2; ++i) cswap(a[i], a[CNT - 1 - i]);
#pragma unroll
    for (int i = 1; i < (CNT + 1) / 2; ++i) cswap(a[0], a[i]);
#pragma unroll
    for (int i = CNT / 2; i < CNT - 1; ++i) cswap(a[i], a[CNT - 1]);
}

template <int CNT, int NEXT, int N, typename C>
struct Forget {
    static __device__ __forceinline__ C run(C* a, const C* v) {
        minmax_to_ends<CNT>(a);
        if constexpr (NEXT < N) {
            // drop max (slot CNT-1) and replace min (slot 0) with the next sample
            a[0] = v[NEXT];
            return Forget<CNT - 1, NEXT + 1, N, C>::run(a, v);
        } else if constexpr (CNT == 3) {
            return a[1];
        } else {
            // no samples left: drop both ends and continue on the interior
            return Forget<CNT - 2, NEXT, N, C>::run(a + 1, v);
        }
    }
};
template <int NEXT, int N, typename C>
struct Forget<1, NEXT, N, C> {
    static __device__ __forceinline__ C run(C* a, const C*) { return a[0]; }
};
template <int NEXT, int N, typename C>
struct Forget<2, NEXT, N, C> {
    static __device__ __forceinline__ C run(C* a, const C*) { return a[0] < a[1] ? a[0] : a[1]; }
};

// Median (rank N/2, 0-based, of the sorted samples) of v[0..N), N odd.
template <int N, typename C>
__device__ __forceinline__ C median_of(const C* v) {
    constexpr int M = N / 2 + 2 < N ? N / 2 + 2 : N;
    C a[M];
#pragma unroll
    for (int i = 0; i < M; ++i) a[i] = v[i];
    return Forget<M, M, N, C>::run(a, v);
}

template <typename T> struct Cmp { using type = int; };
template <> struct Cmp<float> { using type = float; };

// ---------------------------------------------------------------- 2-D
template <typename T, int KY, int KX>
__global__ void __launch_bounds__(256)
median2d_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                int h, int w, int tiles_x, int tiles_y, int border) {
    using C = typename Cmp<T>::type;
    constexpr int TW = 32, TH = 32, RY = KY / 2, RX = KX / 2, EW = TW + 2 * RX, EH = TH + 2 * RY;
    __shared__ C s[EH][EW + 1];
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % tiles_x) * TW, ty0 = (int)((tile / tiles_x) % tiles_y) * TH;
    const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
    const T* plane = src + n * ssn;
    for (int i = threadIdx.x; i < EH * EW; i += 256) {
        const int r = i / EW, c = i - r * EW;
        const int sy = border_index(ty0 - RY + r, h, border), sx = border_index(tx0 - RX + c, w, border);
        s[r][c] = (sy < 0 || sx < 0) ? (C)0 : (C)plane[(int64_t)sy * ssh + sx];
    }
    __syncthreads();
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
#pragma unroll 1
    for (int ly = ly0; ly < TH; ly += 8) {
        const int y = ty0 + ly, x = tx0 + lx;
        if (y >= h || x >= w) continue;
        C v[KY * KX];
#pragma unroll
        for (int dy = 0; dy < KY; ++dy)
#pragma unroll
            for (int dx = 0; dx < KX; ++dx) v[dy * KX + dx] = s[ly + dy][lx + dx];
        dst[n * dsn + (int64_t)y * dsh + x] = (T)median_of<KY * KX, C>(v);
    }
}

template <typename T, int KY, int KX>
static int launch_median2d(const void* src, void* dst, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int64_t dsn,
                           int64_t dsh, int border, cudaStream_t st) {
    const int tiles_x = ceil_div(w, 32), tiles_y = ceil_div(h, 32);
    const int64_t blocks = n * tiles_x * tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    median2d_kernel<T, KY, KX><<<(unsigned)blocks, 256, 0, st>>>((const T*)src, (T*)dst, ssn, ssh, dsn, dsh, h, w,
                                                                tiles_x, tiles_y, border);
    return check_launch();
}

template <typename T>
static int dispatch_median2d(int ky, int kx, const void* src, void* dst, int64_t n, int h, int w, int64_t ssn,
                             int64_t ssh, int64_t dsn, int64_t dsh, int border, cudaStream_t st) {
#define MIE_M2D(KY_, KX_) \
    if (ky == KY_ && kx == KX_) return launch_median2d<T, KY_, KX_>(src, dst, n, h, w, ssn, ssh, dsn, dsh, border, st);
    MIE_M2D(3, 3) MIE_M2D(5, 5) MIE_M2D(7, 7) MIE_M2D(1, 3) MIE_M2D(3, 1) MIE_M2D(3, 5) MIE_M2D(5, 3) MIE_M2D(1, 1)
#undef MIE_M2D
    return MIE_E_KERNEL;
}

// ---------------------------------------------------------------- 3-D, 3x3x3
// One block owns a 32x8 (x,y) tile and walks a chunk of z with a rolling ring of
// three haloed planes in shared memory, so each plane is read once per block.
template <typename T>
__global__ void __launch_bounds__(256)
median3d_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssd, int64_t ssh, int64_t dsd, int64_t dsh,
                int d, int h, int w, int tiles_x, int tiles_y, int zchunk, const T* __restrict__ halo_lo,
                const T* __restrict__ halo_hi, int border) {
    using C = typename Cmp<T>::type;
    constexpr int TW = 32, TH = 8, EW = TW + 2, EH = TH + 2;
    __shared__ C ring[3][EH][EW + 1];
    const int tx0 = (int)(blockIdx.x % tiles_x) * TW, ty0 = (int)(blockIdx.x / tiles_x) * TH;
    const int z0 = blockIdx.y * zchunk, z1 = min(z0 + zchunk, d);
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;

    auto load_plane = [&](int z) {
        // z in [-1, d]: -1 / d come from the neighbouring slab's halo plane or the border rule
        const T* p = nullptr;
        int64_t rs = ssh;
        if (z < 0) {
            if (halo_lo) { p = halo_lo; rs = w; }
            else if (border == MIE_BORDER_REPLICATE) p = src;
        } else if (z >= d) {
            if (halo_hi) { p = halo_hi; rs = w; }
            else if (border == MIE_BORDER_REPLICATE) p = src + (int64_t)(d - 1) * ssd;
        } else {
            p = src + (int64_t)z * ssd;
        }
        C(*slot)[EW + 1] = ring[(z + 3) % 3];
        for (int i = threadIdx.x; i < EH * EW; i += 256) {
            const int r = i / EW, c = i - r * EW;
            const int sy = border_index(ty0 - 1 + r, h, border), sx = border_index(tx0 - 1 + c, w, border);
            slot[r][c] = (!p || sy < 0 || sx < 0) ? (C)0 : (C)p[(int64_t)sy * rs + sx];
        }
    };

    load_plane(z0 - 1);
    load_plane(z0);
    for (int z = z0; z < z1; ++z) {
        load_plane(z + 1);
        __syncthreads();
        const int y = ty0 + ly, x = tx0 + lx;
        if (y < h && x < w) {
            C v[27];
#pragma unroll
            for (int dz = 0; dz < 3; ++dz) {
                C(*slot)[EW + 1] = ring[(z + dz + 2) % 3];  // planes z-1, z, z+1
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) v[dz * 9 + dy * 3 + dx] = slot[ly + dy][lx + dx];
            }
            dst[(int64_t)z * dsd + (int64_t)y * dsh + x] = (T)median_of<27, C>(v);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- 3-D, 3x3x3, 16-bit voxels, two per lane
// Packed variant for uint16 / int16 volumes: a lane owns TWO x-adjacent voxels held in one 32-bit word and
// runs the same forgetful selection on min.{u,s}16x2 / max.{u,s}16x2 (VIMNMX.U16 / .S16), which issue at
// the rate of the scalar min/max (profiles/microbench/minmax_rates_b200_r1.log: 2.0 warp instructions per
// clock per SM) — so the ~300 min/max of a 27-sample median serve two voxels.  The three z-planes of the
// window live in registers as 3x3 packed words each; a z-step loads one new plane (nine 32-bit
// shared-memory loads + six PRMT to form the x-1 / x+1 neighbours), the other two are carried over.
struct PackedU16 {
    uint32_t v;
};
struct PackedS16 {
    uint32_t v;
};
// min and max are separate (non-volatile) asm statements so that halves of a compare-exchange whose
// result is never read are removed by the compiler (the pruned selection networks below rely on it).
__device__ __forceinline__ PackedU16 pmin(PackedU16 a, PackedU16 b) {
    PackedU16 r;
    asm("min.u16x2 %0, %1, %2;" : "=r"(r.v) : "r"(a.v), "r"(b.v));
    return r;
}
__device__ __forceinline__ PackedU16 pmax(PackedU16 a, PackedU16 b) {
    PackedU16 r;
    asm("max.u16x2 %0, %1, %2;" : "=r"(r.v) : "r"(a.v), "r"(b.v));
    return r;
}
__device__ __forceinline__ PackedS16 pmin(PackedS16 a, PackedS16 b) {
    PackedS16 r;
    asm("min.s16x2 %0, %1, %2;" : "=r"(r.v) : "r"(a.v), "r"(b.v));
    return r;
}
__device__ __forceinline__ PackedS16 pmax(PackedS16 a, PackedS16 b) {
    PackedS16 r;
    asm("max.s16x2 %0, %1, %2;" : "=r"(r.v) : "r"(a.v), "r"(b.v));
    return r;
}
__device__ __forceinline__ void cswap(PackedU16& a, PackedU16& b) {
    const PackedU16 lo = pmin(a, b), hi = pmax(a, b);
    a = lo; b = hi;
}
__device__ __forceinline__ void cswap(PackedS16& a, PackedS16& b) {
    const PackedS16 lo = pmin(a, b), hi = pmax(a, b);
    a = lo; b = hi;
}
__device__ __forceinline__ bool operator<(const PackedU16& a, const PackedU16& b) { return a.v < b.v; }  // unused
__device__ __forceinline__ bool operator<(const PackedS16& a, const PackedS16& b) { return a.v < b.v; }  // unused
template <typename P>
__device__ __forceinline__ P packed_min(P a, P b) { cswap(a, b); return a; }

template <int NEXT, int N>
struct Forget<2, NEXT, N, PackedU16> {
    static __device__ __forceinline__ PackedU16 run(PackedU16* a, const PackedU16*) { return packed_min(a[0], a[1]); }
};
template <int NEXT, int N>
struct Forget<2, NEXT, N, PackedS16> {
    static __device__ __forceinline__ PackedS16 run(PackedS16* a, const PackedS16*) { return packed_min(a[0], a[1]); }
};

// ---- rank 13 of 27 from three SORTED 9-lists (the 3x3 neighbourhoods of planes z-1, z, z+1)
// A z-step sorts only the incoming plane's nine samples (25 compare-exchanges, Dobbelaere's optimal
// 9-input network) and reuses the sorted lists of the other two planes, i.e. one sort per output.
// Selection: write the lists as the rows of a 3x9 matrix and sort its columns — rows stay sorted, so
// element (r,c) has (r+1)(c+1)-1 others below it and (3-r)(9-c)-1 above; 14 or more on either side
// rules it out.  Seven entries drop out as too small, seven as too large, and the median of 27 is
// the median (rank 6) of the remaining 13: row0[5..8], row1[2..6], row2[0..3] — three sorted runs.
// Merge the two 4-runs (Batcher odd-even merge, 9 compare-exchanges) into W and finish with
// rank_r(W u Y) = min(w_r, min_{i+j=r-1} max(w_i, y_j)).  ~110 min/max per voxel PAIR instead of the
// ~350 of the forgetful selection (verified exhaustively on 0/1 inputs and on random ties:
// tests/test_host_logic.py::test_median27_selection_network).
template <typename P>
__device__ __forceinline__ void sort9(P* a) {
#define MIE_CS(i, j) cswap(a[i], a[j]);
    MIE_CS(0, 3) MIE_CS(1, 7) MIE_CS(2, 5) MIE_CS(4, 8)
    MIE_CS(0, 7) MIE_CS(2, 4) MIE_CS(3, 8) MIE_CS(5, 6)
    MIE_CS(0, 2) MIE_CS(1, 3) MIE_CS(4, 5) MIE_CS(7, 8)
    MIE_CS(1, 4) MIE_CS(3, 6) MIE_CS(5, 7)
    MIE_CS(0, 1) MIE_CS(2, 4) MIE_CS(3, 5) MIE_CS(6, 8)
    MIE_CS(2, 3) MIE_CS(4, 5) MIE_CS(6, 7)
    MIE_CS(1, 2) MIE_CS(3, 4) MIE_CS(5, 6)
#undef MIE_CS
}
template <typename P>
__device__ __forceinline__ P select27_sorted(const P* A, const P* B, const P* C) {
    P W[8], Y[5];
    // columns 5..8 -> minimum (row 0), columns 0..3 -> maximum (row 2), columns 2..6 -> middle (row 1)
#pragma unroll
    for (int c = 0; c < 9; ++c) {
        const P lo = pmin(A[c], B[c]), hi = pmax(A[c], B[c]);
        if (c >= 5) W[c - 5] = pmin(lo, C[c]);
        if (c <= 3) W[4 + c] = pmax(hi, C[c]);
        if (c >= 2 && c <= 6) Y[c - 2] = c <= 4 ? pmax(lo, pmin(hi, C[c])) : pmin(hi, pmax(lo, C[c]));
    }
    cswap(W[0], W[4]); cswap(W[1], W[5]); cswap(W[2], W[6]); cswap(W[3], W[7]);
    cswap(W[2], W[4]); cswap(W[3], W[5]);
    cswap(W[1], W[2]); cswap(W[3], W[4]); cswap(W[5], W[6]);
    P m = W[6];
#pragma unroll
    for (int j = 0; j < 5; ++j) m = pmin(m, pmax(W[5 - j], Y[j]));
    return m;
}

template <typename T> struct PackedOf;
template <> struct PackedOf<uint16_t> { using type = PackedU16; };
template <> struct PackedOf<int16_t> { using type = PackedS16; };
template <> struct PackedOf<uint8_t> { using type = PackedU16; };   // 8-bit pixels widened to 16-bit lanes on load

template <typename T>
__global__ void __launch_bounds__(256)
median3d_packed_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssd, int64_t ssh, int64_t dsd,
                       int64_t dsh, int d, int h, int w, int tiles_x, int tiles_y, int zchunk,
                       const T* __restrict__ halo_lo, const T* __restrict__ halo_hi, int border) {
    using P = typename PackedOf<T>::type;
    constexpr int TW = 64, TH = 8, EW = TW + 4, EH = TH + 2;   // haloed x range tx0-2 .. tx0+65 (aligned words)
    constexpr int PITCH = EW + 2;                              // 70 voxels = 35 words per row
    __shared__ __align__(4) T ring[3][EH][PITCH];
    const int tx0 = (int)(blockIdx.x % tiles_x) * TW, ty0 = (int)(blockIdx.x / tiles_x) * TH;
    const int z0 = blockIdx.y * zchunk, z1 = min(z0 + zchunk, d);
    const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;

    auto load_plane = [&](int z) {
        const T* p = nullptr;
        int64_t rs = ssh;
        if (z < 0) {
            if (halo_lo) { p = halo_lo; rs = w; }
            else if (border == MIE_BORDER_REPLICATE) p = src;
        } else if (z >= d) {
            if (halo_hi) { p = halo_hi; rs = w; }
            else if (border == MIE_BORDER_REPLICATE) p = src + (int64_t)(d - 1) * ssd;
        } else {
            p = src + (int64_t)z * ssd;
        }
        T(*slot)[PITCH] = ring[(z + 3) % 3];
        for (int i = threadIdx.x; i < EH * EW; i += 256) {
            const int r = i / EW, c = i - r * EW;
            // columns beyond the image + 1 only feed masked outputs: clamp them into border_index's domain
            const int sy = border_index(ty0 - 1 + r, h, border), sx = border_index(min(tx0 - 2 + c, w), w, border);
            slot[r][c] = (!p || sy < 0 || sx < 0) ? (T)0 : p[(int64_t)sy * rs + sx];
        }
    };
    // nine packed words of one plane around this lane's voxel pair: rows ly..ly+2, x-1 / x / x+1 neighbours
    auto plane_words = [&](int z, P* out) {
        const T(*slot)[PITCH] = ring[(z + 3) % 3];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const uint32_t* row = reinterpret_cast<const uint32_t*>(&slot[ly + dy][0]) + lx;
            const uint32_t w0 = row[0], w1 = row[1], w2 = row[2];   // voxels (x-2,x-1) (x,x+1) (x+2,x+3)
            out[dy * 3 + 0].v = __byte_perm(w0, w1, 0x5432);        // (x-1, x)
            out[dy * 3 + 1].v = w1;                                 // (x, x+1)
            out[dy * 3 + 2].v = __byte_perm(w1, w2, 0x5432);        // (x+1, x+2)
        }
    };

    load_plane(z0 - 1);
    load_plane(z0);
    __syncthreads();
    P win[3][9];   // win[k] = SORTED 3x3 neighbourhood of plane z - 1 + k (rotated by register renaming below)
    plane_words(z0 - 1, win[0]);
    plane_words(z0, win[1]);
    sort9(win[0]);
    sort9(win[1]);
    const int y = ty0 + ly, x = tx0 + 2 * lx;
    for (int zb = z0; zb < z1; zb += 3) {
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int z = zb + u;
            if (z < z1) {   // uniform
                load_plane(z + 1);
                __syncthreads();
                plane_words(z + 1, win[(u + 2) % 3]);
                sort9(win[(u + 2) % 3]);
                const uint32_t m = select27_sorted(win[u % 3], win[(u + 1) % 3], win[(u + 2) % 3]).v;
                if (y < h && x < w) {
                    T* o = dst + (int64_t)z * dsd + (int64_t)y * dsh + x;
                    if (x + 1 < w && ((reinterpret_cast<uintptr_t>(o) & 3) == 0)) {
                        *reinterpret_cast<uint32_t*>(o) = m;
                    } else {
                        o[0] = (T)(m & 0xFFFFu);
                        if (x + 1 < w) o[1] = (T)(m >> 16);
                    }
                }
                // no second barrier: the next step writes ring slot (z + 2) % 3, and only slot (z + 1) % 3
                // is still being read (the other two planes of the window are held in registers)
            }
        }
    }
}

// ---------------------------------------------------------------- 3-D, 3x3x3, 16-bit, register marching, no smem
// Even widths with 4-byte-aligned rows: a lane owns one voxel pair and reads the nine packed words of the
// incoming plane (rows y-1..y+1, pairs x-2, x, x+2) straight from global memory — every word is fetched
// by nine lanes of the same block, so the loads hit L1 — instead of staging planes in shared memory:
// no per-voxel index arithmetic, no barriers.  The two older planes stay in registers as sorted 9-lists.
template <typename T, bool EDGE>
__device__ __forceinline__ void median3d_direct_body(const T* __restrict__ src, T* __restrict__ dst, int64_t ssd,
                                                     int64_t ssh, int64_t dsd, int64_t dsh, int d, int h, int w, int x,
                                                     int y, int z0, int z1, const T* __restrict__ halo_lo,
                                                     const T* __restrict__ halo_hi, bool rep) {
    using P = typename PackedOf<T>::type;
    // Rows / pairs outside the volume are read from a clamped (always valid) address and replaced by the
    // border value with a select, so the nine loads of a plane are independent and issue back to back;
    // interior tiles (EDGE == false) need no selects at all.
    const int yc[3] = {EDGE ? max(y - 1, 0) : y - 1, y, EDGE ? min(y + 1, h - 1) : y + 1};
    const bool row_zero[3] = {EDGE && !rep && y == 0, false, EDGE && !rep && y + 1 >= h};
    const bool has_l = !EDGE || x >= 2, has_r = !EDGE || x + 2 < w;
    const int64_t xl = has_l ? -1 : 0, xr = has_r ? 1 : 0;

    auto plane_words = [&](int z, P* out) {
        const T* p = src + (int64_t)min(max(z, 0), d - 1) * ssd;   // replicate rule
        int64_t rs = ssh;
        bool plane_zero = false;
        if (z < 0) {
            if (halo_lo) { p = halo_lo; rs = w; }
            else plane_zero = !rep;
        } else if (z >= d) {
            if (halo_hi) { p = halo_hi; rs = w; }
            else plane_zero = !rep;
        }
        if (plane_zero) {                                          // uniform: constant rule beyond the volume
#pragma unroll
            for (int k = 0; k < 9; ++k) out[k].v = 0u;
            return;
        }
        uint32_t w0[3], w1[3], w2[3];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const uint32_t* row = reinterpret_cast<const uint32_t*>(p + (int64_t)yc[dy] * rs + x);
            w1[dy] = __ldg(row);
            w0[dy] = __ldg(row + xl);
            w2[dy] = __ldg(row + xr);
        }
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const uint32_t c = row_zero[dy] ? 0u : w1[dy];
            const uint32_t l = has_l ? (row_zero[dy] ? 0u : w0[dy]) : (rep ? c << 16 : 0u);   // voxel x-1, high half
            const uint32_t r = has_r ? (row_zero[dy] ? 0u : w2[dy]) : (rep ? c >> 16 : 0u);   // voxel x+2, low half
            out[dy * 3 + 0].v = __byte_perm(l, c, 0x5432);                                    // (x-1, x)
            out[dy * 3 + 1].v = c;                                                            // (x, x+1)
            out[dy * 3 + 2].v = __byte_perm(c, r, 0x5432);                                    // (x+1, x+2)
        }
        sort9(out);
    };

    P win[3][9];   // win[k] = SORTED 3x3 neighbourhood of plane z - 1 + k (rotated by register renaming)
    plane_words(z0 - 1, win[0]);
    plane_words(z0, win[1]);
    T* o = dst + (int64_t)y * dsh + x;
    for (int zb = z0; zb < z1; zb += 3) {
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int z = zb + u;
            if (z < z1) {   // uniform
                plane_words(z + 1, win[(u + 2) % 3]);
                const uint32_t m = select27_sorted(win[u % 3], win[(u + 1) % 3], win[(u + 2) % 3]).v;
                *reinterpret_cast<uint32_t*>(o + (int64_t)z * dsd) = m;
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
median3d_direct_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssd, int64_t ssh, int64_t dsd,
                       int64_t dsh, int d, int h, int w, int tiles_x, int zchunk, const T* __restrict__ halo_lo,
                       const T* __restrict__ halo_hi, int border) {
    const int tx0 = (int)(blockIdx.x % tiles_x) * 64, ty0 = (int)(blockIdx.x / tiles_x) * 8;
    const int z0 = blockIdx.y * zchunk, z1 = min(z0 + zchunk, d);
    const int x = tx0 + 2 * (threadIdx.x & 31), y = ty0 + (threadIdx.x >> 5);
    if (x >= w || y >= h) return;                  // no barriers below
    const bool rep = border == MIE_BORDER_REPLICATE;
    const bool interior = tx0 > 0 && tx0 + 64 < w && ty0 > 0 && ty0 + 8 < h;   // block-uniform
    if (interior) median3d_direct_body<T, false>(src, dst, ssd, ssh, dsd, dsh, d, h, w, x, y, z0, z1, halo_lo, halo_hi, rep);
    else median3d_direct_body<T, true>(src, dst, ssd, ssh, dsd, dsh, d, h, w, x, y, z0, z1, halo_lo, halo_hi, rep);
}

// ---------------------------------------------------------------- 2-D 3x3, 8 / 16-bit pixels, marching rows
// A lane owns 8 consecutive columns (one 128-bit load per row = four packed pixel pairs) and marches
// down a band of rows with the last three rows in registers; the pair to the left / right comes from the
// neighbouring lane by shuffle (from global memory or the border rule at the ends of the warp's 256-column
// strip).  Per row the three vertical samples of every packed word are sorted once (3 compare-exchanges,
// shared by the three windows that contain the column); the x-1 / x+1 neighbours of the sorted triples are
// byte permutes of adjacent words (sorting columns commutes with shifting them).  Then the classic
// median-of-9 identity: med3(max of the column minima, med3 of the column medians, min of the column
// maxima).  ~27 integer-pipe instructions per pixel pair, no shared memory.
template <typename T>
__global__ void __launch_bounds__(256, 4)
median3x3_packed_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                        int64_t dsh, int64_t nplanes, int h, int w, int strips, int bands, int rows_per_band,
                        int border) {
    using P = typename PackedOf<T>::type;
    const int lane = threadIdx.x & 31;
    const int64_t wg = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int strip = (int)(wg % strips), band = (int)((wg / strips) % bands);
    const int64_t n = wg / ((int64_t)strips * bands);
    if (n >= nplanes) return;                      // warp-uniform
    const int x0 = strip * 256 + lane * 8;
    const bool active = x0 < w;
    const int y0 = band * rows_per_band, y1 = min(y0 + rows_per_band, h);
    const T* plane = src + n * ssn;
    T* oplane = dst + n * dsn;

    // Row y arrives in two steps so that the loads of row y + 2 are in flight while row y + 1 is consumed
    // (with the load issued where it is used the kernel sat on the scoreboard: 6.8 stalled warps per issue,
    // profiles/r1_ncu_full_standalone_ops2.txt).  issue_row: the global loads only — the lane's 8 pixels plus
    // the pair across the strip boundary for lanes 0 / 31.  finish_row: widening, neighbour shuffles and the
    // border rule, giving six packed words [pair left of x0 | four own pairs | pair right of x0 + 7].
    struct Raw { uint4 q; uint32_t l, r; };
    auto issue_row = [&](int y, Raw& t) {
        const int sy = border_index(y, h, border);
        t.q = make_uint4(0u, 0u, 0u, 0u); t.l = 0u; t.r = 0u;
        if (sy >= 0 && active) {
            const T* row = plane + (int64_t)sy * ssh;
            if constexpr (sizeof(T) == 1) {
                const uint2 raw = __ldg(reinterpret_cast<const uint2*>(row + x0));
                t.q.x = raw.x; t.q.y = raw.y;
                if (lane == 0 && x0 != 0) t.l = (uint32_t)__ldg(row + x0 - 1) << 16;
                if (lane == 31 && x0 + 8 != w) t.r = (uint32_t)__ldg(row + x0 + 8);
            } else {
                t.q = __ldg(reinterpret_cast<const uint4*>(row + x0));
                if (lane == 0 && x0 != 0) t.l = __ldg(reinterpret_cast<const uint32_t*>(row + x0 - 2));
                if (lane == 31 && x0 + 8 != w) t.r = __ldg(reinterpret_cast<const uint32_t*>(row + x0 + 8));
            }
        }
    };
    auto finish_row = [&](int y, const Raw& t, P* r) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        uint32_t left = 0u, right = 0u;
        if (border_index(y, h, border) >= 0) {      // uniform
            if constexpr (sizeof(T) == 1) {         // 8 bytes -> four (pixel, pixel) words of 16-bit lanes
                v.x = __byte_perm(t.q.x, 0u, 0x4140); v.y = __byte_perm(t.q.x, 0u, 0x4342);
                v.z = __byte_perm(t.q.y, 0u, 0x4140); v.w = __byte_perm(t.q.y, 0u, 0x4342);
            } else {
                v = t.q;
            }
            left = __shfl_up_sync(0xffffffffu, v.w, 1);
            right = __shfl_down_sync(0xffffffffu, v.x, 1);
            if (active) {
                if (x0 == 0) {                      // pixel -1 sits in the high half
                    left = border == MIE_BORDER_REFLECT ? (v.x & 0xFFFF0000u)
                         : (border == MIE_BORDER_REPLICATE || border == MIE_BORDER_SYMMETRIC) ? (v.x << 16) : 0u;
                } else if (lane == 0) {
                    left = t.l;
                }
                if (x0 + 8 == w) {                  // pixel w sits in the low half
                    right = border == MIE_BORDER_REFLECT ? (v.w & 0xFFFFu)
                          : (border == MIE_BORDER_REPLICATE || border == MIE_BORDER_SYMMETRIC) ? (v.w >> 16) : 0u;
                } else if (lane == 31) {
                    right = t.r;
                }
            }
        }
        r[0].v = left; r[1].v = v.x; r[2].v = v.y; r[3].v = v.z; r[4].v = v.w; r[5].v = right;
    };

    P ring[3][6];
    Raw nxt;
    {
        Raw t0, t1;
        issue_row(y0 - 1, t0); issue_row(y0, t1); issue_row(y0 + 1, nxt);
        finish_row(y0 - 1, t0, ring[0]); finish_row(y0, t1, ring[1]);
    }
    for (int yb = y0; yb < y1; yb += 3) {
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int y = yb + u;
            if (y < y1) {                           // uniform
                const Raw cur = nxt;
                if (y + 1 < y1) issue_row(y + 2, nxt);   // uniform; consumed by the next output row
                finish_row(y + 1, cur, ring[(u + 2) % 3]);
                P lo[6], mi[6], hi[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    P a = ring[u % 3][c], b = ring[(u + 1) % 3][c], cc = ring[(u + 2) % 3][c];
                    cswap(a, b); cswap(b, cc); cswap(a, b);
                    lo[c] = a; mi[c] = b; hi[c] = cc;
                }
                uint32_t o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    P Llo, Lmi, Lhi, Rlo, Rmi, Rhi;
                    Llo.v = __byte_perm(lo[k].v, lo[k + 1].v, 0x5432); Rlo.v = __byte_perm(lo[k + 1].v, lo[k + 2].v, 0x5432);
                    Lmi.v = __byte_perm(mi[k].v, mi[k + 1].v, 0x5432); Rmi.v = __byte_perm(mi[k + 1].v, mi[k + 2].v, 0x5432);
                    Lhi.v = __byte_perm(hi[k].v, hi[k + 1].v, 0x5432); Rhi.v = __byte_perm(hi[k + 1].v, hi[k + 2].v, 0x5432);
                    const P maxlo = pmax(pmax(Llo, lo[k + 1]), Rlo);
                    const P minhi = pmin(pmin(Lhi, hi[k + 1]), Rhi);
                    const P a = pmin(Lmi, mi[k + 1]), b = pmax(Lmi, mi[k + 1]);
                    const P medmi = pmax(a, pmin(b, Rmi));
                    const P c = pmin(maxlo, medmi), d = pmax(maxlo, medmi);
                    o[k] = pmax(c, pmin(d, minhi)).v;
                }
                if (active) {
                    if constexpr (sizeof(T) == 1)
                        *reinterpret_cast<uint2*>(oplane + (int64_t)y * dsh + x0) =
                            make_uint2(__byte_perm(o[0], o[1], 0x6420), __byte_perm(o[2], o[3], 0x6420));
                    else
                        *reinterpret_cast<uint4*>(oplane + (int64_t)y * dsh + x0) = make_uint4(o[0], o[1], o[2], o[3]);
                }
            }
        }
    }
}

// ---------------------------------------------------------------- 2-D 5x5, 8 / 16-bit pixels, marching rows
// Same schedule as the 3x3 kernel (8 columns per lane, neighbours by shuffle, five rows in registers).
// Per row the five vertical samples of every packed word are sorted once (9 compare-exchanges, shared by
// the five windows that contain the column; the x-1 / x+1 shifted columns are byte permutes of the sorted
// words).  The window is then a 5x5 matrix with sorted columns; sorting its ROWS keeps the columns sorted,
// so element (r, c) has (r+1)(c+1)-1 samples below and (5-r)(5-c)-1 above: 13 or more on either side rules
// it out.  Six entries drop out on each side and the median of 25 is the median (rank 6) of the remaining 13
// — five sorted runs of 2, 3, 3, 3, 2 — found by three small merges (3 + 6 + 8 compare-exchanges) and
// rank_r(W u Y) = min(w_r, min_{i+j=r-1} max(w_i, y_j)).  Unused halves of the row sorts are dead code.
// Verified on 0/1 inputs and random ties: tests/test_host_logic.py::test_median25_selection_network.
template <typename P>
__device__ __forceinline__ void sort5(P& a, P& b, P& c, P& d, P& e) {
    cswap(a, d); cswap(b, e); cswap(a, c); cswap(b, d); cswap(a, b); cswap(c, e); cswap(b, c); cswap(d, e); cswap(c, d);
}
// col[c][r]: column c of the window (c = 0..4), vertical rank r (0..4)
template <typename P>
__device__ __forceinline__ P select25_sorted_columns(const P (&A)[5], const P (&B)[5], const P (&C)[5],
                                                     const P (&D)[5], const P (&E)[5]) {
    P R[5][5];
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        R[r][0] = A[r]; R[r][1] = B[r]; R[r][2] = C[r]; R[r][3] = D[r]; R[r][4] = E[r];
        sort5(R[r][0], R[r][1], R[r][2], R[r][3], R[r][4]);
    }
    // candidates: R0[3..4], R1[2..4], R2[1..3], R3[0..2], R4[0..1]
    P xz[4] = {R[0][3], R[0][4], R[4][0], R[4][1]};
    cswap(xz[0], xz[2]); cswap(xz[1], xz[3]); cswap(xz[1], xz[2]);                        // merge 2 + 2
    P y[6] = {R[1][2], R[1][3], R[1][4], R[3][0], R[3][1], R[3][2]};
    cswap(y[0], y[3]); cswap(y[1], y[4]); cswap(y[1], y[3]); cswap(y[2], y[5]); cswap(y[2], y[3]); cswap(y[3], y[4]);   // 3 + 3
    P w[7] = {xz[0], xz[1], xz[2], xz[3], R[2][1], R[2][2], R[2][3]};
    cswap(w[0], w[4]); cswap(w[1], w[4]); cswap(w[1], w[5]); cswap(w[2], w[5]); cswap(w[3], w[6]); cswap(w[3], w[4]);
    cswap(w[2], w[3]); cswap(w[4], w[5]);                                                 // merge 4 + 3
    P m = w[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) m = pmin(m, pmax(w[i], y[5 - i]));
    return m;
}

template <typename T>
__global__ void __launch_bounds__(256)
median5x5_packed_kernel(const T* __restrict__ src, T* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                        int64_t dsh, int64_t nplanes, int h, int w, int strips, int bands, int rows_per_band,
                        int border) {
    using P = typename PackedOf<T>::type;
    const int lane = threadIdx.x & 31;
    const int64_t wg = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int strip = (int)(wg % strips), band = (int)((wg / strips) % bands);
    const int64_t n = wg / ((int64_t)strips * bands);
    if (n >= nplanes) return;                      // warp-uniform
    const int x0 = strip * 256 + lane * 8;
    const bool active = x0 < w;
    const int y0 = band * rows_per_band, y1 = min(y0 + rows_per_band, h);
    const T* plane = src + n * ssn;
    T* oplane = dst + n * dsn;

    // issue_row / finish_row as in the 3x3 kernel (loads one row ahead of their use); finish_row gives six packed
    // words of image row y: [pixels x0-2, x0-1 | four own pairs | pixels x0+8, x0+9]
    struct Raw { uint4 q; uint32_t l, r; };
    auto issue_row = [&](int y, Raw& t) {
        const int sy = border_index(y, h, border);
        t.q = make_uint4(0u, 0u, 0u, 0u); t.l = 0u; t.r = 0u;
        if (sy >= 0 && active) {
            const T* row = plane + (int64_t)sy * ssh;
            if constexpr (sizeof(T) == 1) {
                const uint2 raw = __ldg(reinterpret_cast<const uint2*>(row + x0));
                t.q.x = raw.x; t.q.y = raw.y;
                if (lane == 0 && x0 != 0) t.l = (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(row + x0 - 2));
                if (lane == 31 && x0 + 8 != w) t.r = (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(row + x0 + 8));
            } else {
                t.q = __ldg(reinterpret_cast<const uint4*>(row + x0));
                if (lane == 0 && x0 != 0) t.l = __ldg(reinterpret_cast<const uint32_t*>(row + x0 - 2));
                if (lane == 31 && x0 + 8 != w) t.r = __ldg(reinterpret_cast<const uint32_t*>(row + x0 + 8));
            }
        }
    };
    auto finish_row = [&](int y, const Raw& t, P* r) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        uint32_t left = 0u, right = 0u;
        if (border_index(y, h, border) >= 0) {      // uniform
            if constexpr (sizeof(T) == 1) {
                v.x = __byte_perm(t.q.x, 0u, 0x4140); v.y = __byte_perm(t.q.x, 0u, 0x4342);
                v.z = __byte_perm(t.q.y, 0u, 0x4140); v.w = __byte_perm(t.q.y, 0u, 0x4342);
            } else {
                v = t.q;
            }
            left = __shfl_up_sync(0xffffffffu, v.w, 1);
            right = __shfl_down_sync(0xffffffffu, v.x, 1);
            if (active) {
                if (x0 == 0) {                      // pixels -2 (low half), -1 (high half)
                    left = border == MIE_BORDER_REFLECT ? __byte_perm(v.x, v.y, 0x3254)        // (px 2, px 1)
                         : border == MIE_BORDER_SYMMETRIC ? __byte_perm(v.x, 0u, 0x1032)       // (px 1, px 0)
                         : border == MIE_BORDER_REPLICATE ? __byte_perm(v.x, 0u, 0x1010) : 0u; // (px 0, px 0)
                } else if (lane == 0) {
                    if constexpr (sizeof(T) == 1) left = __byte_perm(t.l, 0u, 0x4140);
                    else left = t.l;
                }
                if (x0 + 8 == w) {                  // pixels w (low half), w + 1 (high half)
                    right = border == MIE_BORDER_REFLECT ? __byte_perm(v.w, v.z, 0x7610)       // (px w-2, px w-3)
                          : border == MIE_BORDER_SYMMETRIC ? __byte_perm(v.w, 0u, 0x1032)      // (px w-1, px w-2)
                          : border == MIE_BORDER_REPLICATE ? __byte_perm(v.w, 0u, 0x3232) : 0u;// (px w-1, px w-1)
                } else if (lane == 31) {
                    if constexpr (sizeof(T) == 1) right = __byte_perm(t.r, 0u, 0x4140);
                    else right = t.r;
                }
            }
        }
        r[0].v = left; r[1].v = v.x; r[2].v = v.y; r[3].v = v.z; r[4].v = v.w; r[5].v = right;
    };

    P ring[5][6];
    Raw nxt;
    {
        Raw t0, t1, t2, t3;
        issue_row(y0 - 2, t0); issue_row(y0 - 1, t1); issue_row(y0, t2); issue_row(y0 + 1, t3); issue_row(y0 + 2, nxt);
        finish_row(y0 - 2, t0, ring[0]); finish_row(y0 - 1, t1, ring[1]);
        finish_row(y0, t2, ring[2]); finish_row(y0 + 1, t3, ring[3]);
    }
    for (int yb = y0; yb < y1; yb += 5) {
#pragma unroll
        for (int u = 0; u < 5; ++u) {
            const int y = yb + u;
            if (y < y1) {                           // uniform
                const Raw cur = nxt;
                if (y + 1 < y1) issue_row(y + 3, nxt);   // uniform
                finish_row(y + 2, cur, ring[(u + 4) % 5]);
                P s[6][5];                          // vertically sorted samples of every word
#pragma unroll
                for (int c = 0; c < 6; ++c) {
#pragma unroll
                    for (int r = 0; r < 5; ++r) s[c][r] = ring[r][c];
                    sort5(s[c][0], s[c][1], s[c][2], s[c][3], s[c][4]);
                }
                P bt[5][5];                         // bt[j] = words j, j+1 shifted by one pixel: (hi of j, lo of j+1)
#pragma unroll
                for (int j = 0; j < 5; ++j)
#pragma unroll
                    for (int r = 0; r < 5; ++r) bt[j][r].v = __byte_perm(s[j][r].v, s[j + 1][r].v, 0x5432);
                uint32_t o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    o[k] = select25_sorted_columns(s[k], bt[k], s[k + 1], bt[k + 1], s[k + 2]).v;
                if (active) {
                    if constexpr (sizeof(T) == 1)
                        *reinterpret_cast<uint2*>(oplane + (int64_t)y * dsh + x0) =
                            make_uint2(__byte_perm(o[0], o[1], 0x6420), __byte_perm(o[2], o[3], 0x6420));
                    else
                        *reinterpret_cast<uint4*>(oplane + (int64_t)y * dsh + x0) = make_uint4(o[0], o[1], o[2], o[3]);
                }
            }
        }
    }
}

// ---------------------------------------------------------------- 2-D 3x3, float pixels (kornia's native dtype)
// The marching schedule of the packed kernels with one pixel per register: a lane owns 4 consecutive columns
// (one 128-bit load per row), the neighbours come from the adjacent lanes by shuffle, the three vertical
// samples of every column are sorted once per row, and the median of 9 is med3(max of minima, med3 of medians,
// min of maxima).  fminf / fmaxf semantics as in the generic kernel.
__global__ void __launch_bounds__(256)
median3x3_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                     int64_t dsh, int64_t nplanes, int h, int w, int strips, int bands, int rows_per_band, int border) {
    const int lane = threadIdx.x & 31;
    const int64_t wg = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int strip = (int)(wg % strips), band = (int)((wg / strips) % bands);
    const int64_t n = wg / ((int64_t)strips * bands);
    if (n >= nplanes) return;                      // warp-uniform
    const int x0 = strip * 128 + lane * 4;
    const bool active = x0 < w;
    const int y0 = band * rows_per_band, y1 = min(y0 + rows_per_band, h);
    const float* plane = src + n * ssn;
    float* oplane = dst + n * dsn;

    // issue_row / finish_row: loads one row ahead of their use, as in median3x3_packed_kernel
    struct Raw { float4 q; float l, r; };
    auto issue_row = [&](int y, Raw& t) {
        const int sy = border_index(y, h, border);
        t.q = make_float4(0.f, 0.f, 0.f, 0.f); t.l = 0.f; t.r = 0.f;
        if (sy >= 0 && active) {
            const float* row = plane + (int64_t)sy * ssh;
            t.q = __ldg(reinterpret_cast<const float4*>(row + x0));
            if (lane == 0 && x0 != 0) t.l = __ldg(row + x0 - 1);
            if (lane == 31 && x0 + 4 != w) t.r = __ldg(row + x0 + 4);
        }
    };
    auto finish_row = [&](int y, const Raw& t, float* r) {   // r[0] = pixel x0-1, r[1..4] = own pixels, r[5] = pixel x0+4
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        float left = 0.f, right = 0.f;
        if (border_index(y, h, border) >= 0) {      // uniform
            v = t.q;
            left = __shfl_up_sync(0xffffffffu, v.w, 1);
            right = __shfl_down_sync(0xffffffffu, v.x, 1);
            if (active) {
                if (x0 == 0)
                    left = border == MIE_BORDER_REFLECT ? v.y
                         : (border == MIE_BORDER_REPLICATE || border == MIE_BORDER_SYMMETRIC) ? v.x : 0.f;
                else if (lane == 0)
                    left = t.l;
                if (x0 + 4 == w)
                    right = border == MIE_BORDER_REFLECT ? v.z
                          : (border == MIE_BORDER_REPLICATE || border == MIE_BORDER_SYMMETRIC) ? v.w : 0.f;
                else if (lane == 31)
                    right = t.r;
            }
        }
        r[0] = left; r[1] = v.x; r[2] = v.y; r[3] = v.z; r[4] = v.w; r[5] = right;
    };

    float ring[3][6];
    Raw nxt;
    {
        Raw t0, t1;
        issue_row(y0 - 1, t0); issue_row(y0, t1); issue_row(y0 + 1, nxt);
        finish_row(y0 - 1, t0, ring[0]); finish_row(y0, t1, ring[1]);
    }
    for (int yb = y0; yb < y1; yb += 3) {
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            const int y = yb + u;
            if (y < y1) {                           // uniform
                const Raw cur = nxt;
                if (y + 1 < y1) issue_row(y + 2, nxt);   // uniform
                finish_row(y + 1, cur, ring[(u + 2) % 3]);
                float lo[6], mi[6], hi[6];
#pragma unroll
                for (int c = 0; c < 6; ++c) {
                    float a = ring[u % 3][c], b = ring[(u + 1) % 3][c], cc = ring[(u + 2) % 3][c];
                    cswap(a, b); cswap(b, cc); cswap(a, b);
                    lo[c] = a; mi[c] = b; hi[c] = cc;
                }
                float o[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float maxlo = fmaxf(fmaxf(lo[k], lo[k + 1]), lo[k + 2]);
                    const float minhi = fminf(fminf(hi[k], hi[k + 1]), hi[k + 2]);
                    const float a = fminf(mi[k], mi[k + 1]), b = fmaxf(mi[k], mi[k + 1]);
                    const float medmi = fmaxf(a, fminf(b, mi[k + 2]));
                    const float c = fminf(maxlo, medmi), d = fmaxf(maxlo, medmi);
                    o[k] = fmaxf(c, fminf(d, minhi));
                }
                if (active) *reinterpret_cast<float4*>(oplane + (int64_t)y * dsh + x0) = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
    }
}

static int try_median3x3_f32(const Image& s, const Image& d, int64_t n, int h, int w, int border, cudaStream_t st) {
    const bool off = kernel_policy(MIE_POLICY_GENERIC_MEDIAN);
    if (off || (w & 3) || h < 2) return -1;
    if (!s.aligned(16) || !d.aligned(16)) return -1;
    const int strips = ceil_div(w, 128);
    int rows = 32;
    while (rows > 8 && n * strips * ceil_div(h, rows) < 8 * 148 * 4) rows >>= 1;
    const int bands = ceil_div(h, rows);
    const int64_t blocks = (n * strips * bands + 7) / 8;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    median3x3_f32_kernel<<<(unsigned)blocks, 256, 0, st>>>((const float*)s.p, (float*)d.out(), s.sn, s.sh, d.sn, d.sh, n,
                                                          h, w, strips, bands, rows, border);
    return check_launch();
}

// 0 = launched, < 0 = not applicable (caller falls back to the generic kernel), > 0 = CUDA error
template <typename T>
static int try_median_packed(const Image& s, const Image& d, int64_t n, int h, int w, int border, int k,
                             cudaStream_t st) {
    const bool off = kernel_policy(MIE_POLICY_GENERIC_MEDIAN);
    if (off || (w & 7) || h < k - 1) return -1;
    if (!s.aligned(8 * sizeof(T)) || !d.aligned(8 * sizeof(T))) return -1;   // one 8-pixel vector per lane and row
    const int strips = ceil_div(w, 256);
    int rows = 32;                                 // 2 halo rows per band: 6 % extra loads
    while (rows > 8 && n * strips * ceil_div(h, rows) < 8 * 148 * 4) rows >>= 1;   // small jobs: more warps
    const int bands = ceil_div(h, rows);
    const int64_t warps = n * strips * bands;
    const int64_t blocks = (warps + 7) / 8;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    if (k == 5)
        median5x5_packed_kernel<T><<<(unsigned)blocks, 256, 0, st>>>((const T*)s.p, (T*)d.out(), s.sn, s.sh, d.sn, d.sh, n,
                                                                    h, w, strips, bands, rows, border);
    else
        median3x3_packed_kernel<T><<<(unsigned)blocks, 256, 0, st>>>((const T*)s.p, (T*)d.out(), s.sn, s.sh, d.sn, d.sh, n,
                                                                    h, w, strips, bands, rows, border);
    return check_launch();
}

template <typename T>
static int launch_median3d(const Image& s, const Image& o, int d, int h, int w, const void* lo, const void* hi,
                           int border, cudaStream_t st) {
    const void* src = s.p;
    void* dst = o.out();
    const int64_t ssd = s.sn, ssh = s.sh, dsd = o.sn, dsh = o.sh;
    const int zchunk = d >= 64 ? 32 : (d >= 16 ? 8 : d);
    if constexpr (sizeof(T) == 2) {
        const bool off = kernel_policy(MIE_POLICY_GENERIC_MEDIAN);
        const bool words_ok = !(w & 1) && s.aligned(4) && o.aligned(4) && !((uintptr_t)lo & 3) && !((uintptr_t)hi & 3);
        if (!off && words_ok) {
            const int tiles_x = ceil_div(w, 64), tiles_y = ceil_div(h, 8);
            dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)ceil_div(d, zchunk));
            median3d_direct_kernel<T><<<grid, 256, 0, st>>>((const T*)src, (T*)dst, ssd, ssh, dsd, dsh, d, h, w, tiles_x,
                                                           zchunk, (const T*)lo, (const T*)hi, border);
            return check_launch();
        }
        if (!off) {
            const int tiles_x = ceil_div(w, 64), tiles_y = ceil_div(h, 8);
            dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)ceil_div(d, zchunk));
            median3d_packed_kernel<T><<<grid, 256, 0, st>>>((const T*)src, (T*)dst, ssd, ssh, dsd, dsh, d, h, w, tiles_x,
                                                           tiles_y, zchunk, (const T*)lo, (const T*)hi, border);
            return check_launch();
        }
    }
    const int tiles_x = ceil_div(w, 32), tiles_y = ceil_div(h, 8);
    dim3 grid((unsigned)(tiles_x * tiles_y), (unsigned)ceil_div(d, zchunk));
    median3d_kernel<T><<<grid, 256, 0, st>>>((const T*)src, (T*)dst, ssd, ssh, dsd, dsh, d, h, w, tiles_x, tiles_y,
                                            zchunk, (const T*)lo, (const T*)hi, border);
    return check_launch();
}

}  // namespace mie

using namespace mie;

extern "C" {

int mie_median2d(const void* src, void* dst, int dtype, int64_t n, int h, int w, int64_t src_stride_n,
                 int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h, int ky, int kx, int border,
                 void* stream) {
    const Image s{src, dtype, src_stride_n, src_stride_h}, d{dst, dtype, dst_stride_n, dst_stride_h};
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    if (border != MIE_BORDER_CONSTANT && border != MIE_BORDER_REPLICATE && border != MIE_BORDER_REFLECT &&
        border != MIE_BORDER_SYMMETRIC)
        return MIE_E_BORDER;
    if (ky <= 0 || kx <= 0 || !(ky & 1) || !(kx & 1)) return MIE_E_KERNEL;
    if (n == 0) return MIE_OK;
    if (!valid_dtype(dtype)) return MIE_E_DTYPE;   // before the tuned paths, which pick their kernel by dtype
    cudaStream_t st = (cudaStream_t)stream;
    if (ky == 3 && kx == 3 && dtype == MIE_F32) {
        rc = try_median3x3_f32(s, d, n, h, w, border, st);
        if (rc >= 0) return rc;
    }
    if (ky == kx && (ky == 3 || ky == 5) && dtype != MIE_F32) {   // packed marching kernels (8 / 16-bit pixels)
        rc = dtype == MIE_U16   ? try_median_packed<uint16_t>(s, d, n, h, w, border, ky, st)
             : dtype == MIE_I16 ? try_median_packed<int16_t>(s, d, n, h, w, border, ky, st)
                                : try_median_packed<uint8_t>(s, d, n, h, w, border, ky, st);
        if (rc >= 0) return rc;
    }
    MIE_DISPATCH_SRC(dtype, return dispatch_median2d<SrcT>(ky, kx, src, dst, n, h, w, src_stride_n, src_stride_h,
                                                          dst_stride_n, dst_stride_h, border, st));
    return MIE_OK;
}

int mie_median3d(const void* src, void* dst, int dtype, int d, int h, int w, int64_t src_stride_d,
                 int64_t src_stride_h, int64_t dst_stride_d, int64_t dst_stride_h, const void* halo_lo,
                 const void* halo_hi, int border, void* stream) {
    const Image s{src, dtype, src_stride_d, src_stride_h}, o{dst, dtype, dst_stride_d, dst_stride_h};
    int rc = check_planes(s, o, d, h, w);
    if (rc) return rc;
    if (border != MIE_BORDER_CONSTANT && border != MIE_BORDER_REPLICATE) return MIE_E_BORDER;
    if (d == 0) return MIE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    MIE_DISPATCH_SRC(dtype, return launch_median3d<SrcT>(s, o, d, h, w, halo_lo, halo_hi, border, st));
    return MIE_OK;
}

}  // extern "C"
