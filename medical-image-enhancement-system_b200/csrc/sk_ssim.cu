// sk_ssim.cu — skimage.metrics.structural_similarity on planes (ndim 2) and whole volumes (ndim 3).
//
// RECALLED semantics (include/mie.h; the reference is the numpy transcription tests/sk_ssim_twin.py).  The five
// quantities a, b, a*a, b*b, a*b (products in the image's float type) go through scipy's 1-D filter along every axis
// in array order — z, y, x for volumes, y, x for planes — with scipy's line arithmetic in float64 and the values
// rounded to the image's float type between passes.  The box filter is scipy's running sum, so every output depends on
// the whole prefix of its line: one thread walks one line, in scipy's order.  The Gaussian is scipy's symmetric
// correlation.  Every step is one correctly rounded operation (rn_* / __d*_rn), so the map equals the twin bit for
// bit; only the mean's summation order differs from numpy's.
//
// The batch is cut into chunks of whole images, or of z ranges of one volume, whose two float buffers (z-pass and
// y-pass output) stay below kSsimChunkBytes whatever n and d: a long volume's z-pass carries its running sums from one
// chunk to the next.  Per chunk: the source pass (z for volumes, y for planes), the y pass (volumes), the x pass — which
// evaluates S, stores the map if asked and writes one float64 sum per row over the cropped interior — and a fold that
// adds each image's row sums, in a fixed order, to its entry of `mssim`.  A last launch divides by the interior's
// size.  No float atomics, so repeated runs give identical bits.
#include <algorithm>
#include <climits>
#include <type_traits>

#include "mie_common.cuh"

namespace mie {

constexpr int kQ = 5;                                     // a, b, a*a, b*b, a*b
constexpr size_t kSsimChunkBytes = (size_t)640 << 20;      // the float buffers of one chunk

// The filter of every axis: box of `size` taps (scipy uniform_filter1d) or, size == 0, Gaussian taps w[0 .. 2r].
struct SsimWin {
    int size, r;
    double w[MIE_MAX_TAPS];
};

// One chunk: images m0 .. m0 + nvol - 1, slices z0 .. z0 + nz - 1 of each (planes: d == nz == 1).  Buffers hold
// quantity q of chunk voxel v at q * cap + v, v = (k * h + y) * w + x with chunk slice k = image * nz + z - z0.
struct SsimGeom {
    int nd, d, h, w;
    int64_t m0, nvol;
    int z0, nz;
    int64_t cap;
    int64_t asn, asd, ash, bsn, bsd, bsh;
};

__device__ __forceinline__ int ss_mirror(int i, int n) { return border_index(i, n, MIE_BORDER_SYMMETRIC); }

// The five quantities at index i of a line through the two sources (bases and strides along the line given).
template <typename T>
struct SsimSrcLine {
    const T* a;
    const T* b;
    int64_t sa, sb;
    __device__ __forceinline__ void operator()(int i, double* q) const {
        using F = SkFloat<T>;
        const F va = (F)a[(int64_t)i * sa], vb = (F)b[(int64_t)i * sb];
        q[0] = va;
        q[1] = vb;
        q[2] = rn_mul(va, va);
        q[3] = rn_mul(vb, vb);
        q[4] = rn_mul(va, vb);
    }
};

// The same from a chunk buffer.
template <typename F>
struct SsimBufLine {
    const F* p;
    int64_t s, cap;
    __device__ __forceinline__ void operator()(int i, double* q) const {
#pragma unroll
        for (int k = 0; k < kQ; ++k) q[k] = (double)p[k * cap + (int64_t)i * s];
    }
};

// scipy's 1-D filter of a line of length len ('reflect' border, mirrored as often as needed), outputs i0 .. i1 - 1
// handed to emit(i, q) in order.  Box: tmp = sum of the first `size` extended samples, out[0] = tmp / size, then
// tmp += ext[i + r] - ext[i - r - 1] and out[i] = tmp / size.  `resume` takes tmp after output i0 - 1 from carry[k * cs],
// `save` stores tmp after output i1 - 1 there.  Gaussian: tmp = ext[i] w[r], then tmp += (ext[i + j] + ext[i - j]) w[j + r]
// for j = -r .. -1.
template <typename Ld, typename Emit>
__device__ __forceinline__ void ssim_line(const Ld& ld, int len, int i0, int i1, const SsimWin& win, double* carry,
                                          int64_t cs, bool resume, bool save, const Emit& emit) {
    double t[kQ], u[kQ], v[kQ];
    if (win.size) {
        const double size = (double)win.size;
        int i = i0;
        if (resume) {
#pragma unroll
            for (int k = 0; k < kQ; ++k) t[k] = carry[k * cs];
        } else {
#pragma unroll
            for (int k = 0; k < kQ; ++k) t[k] = 0.0;
#pragma unroll 1
            for (int j = 0; j < win.size; ++j) {
                ld(ss_mirror(j - win.r, len), u);
#pragma unroll
                for (int k = 0; k < kQ; ++k) t[k] = __dadd_rn(t[k], u[k]);
            }
#pragma unroll
            for (int k = 0; k < kQ; ++k) v[k] = __ddiv_rn(t[k], size);
            emit(i, v);
            ++i;
        }
#pragma unroll 1
        for (; i < i1; ++i) {
            ld(ss_mirror(i + win.r, len), u);
            ld(ss_mirror(i - win.r - 1, len), v);
#pragma unroll
            for (int k = 0; k < kQ; ++k) {
                t[k] = __dadd_rn(t[k], __dsub_rn(u[k], v[k]));
                v[k] = __ddiv_rn(t[k], size);
            }
            emit(i, v);
        }
        if (save) {
#pragma unroll
            for (int k = 0; k < kQ; ++k) carry[k * cs] = t[k];
        }
    } else {
#pragma unroll 1
        for (int i = i0; i < i1; ++i) {
            ld(i, u);
#pragma unroll
            for (int k = 0; k < kQ; ++k) t[k] = __dmul_rn(u[k], win.w[win.r]);
#pragma unroll 1
            for (int j = -win.r; j < 0; ++j) {
                ld(ss_mirror(i + j, len), u);
                ld(ss_mirror(i - j, len), v);
                const double wj = win.w[j + win.r];
#pragma unroll
                for (int k = 0; k < kQ; ++k) t[k] = __dadd_rn(t[k], __dmul_rn(__dadd_rn(u[k], v[k]), wj));
            }
            emit(i, t);
        }
    }
}

// First pass, over the sources: along z into the z buffer (volumes), along y into the y buffer (planes).  One thread
// per line, lanes along x.
template <typename T, int ND>
__global__ void __launch_bounds__(256)
sk_ssim_src_pass_kernel(const T* __restrict__ a, const T* __restrict__ b, SsimGeom g, SsimWin win,
                        SkFloat<T>* __restrict__ out, double* __restrict__ carry) {
    using F = SkFloat<T>;
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    const int64_t hw = (int64_t)g.h * g.w;
    const int x = (int)(t % g.w);
    if constexpr (ND == 3) {
        if (t >= g.nvol * hw) return;
        const int64_t v = t / hw;
        const int y = (int)(t % hw / g.w);
        const int64_t m = g.m0 + v;
        const SsimSrcLine<T> ld{a + m * g.asn + (int64_t)y * g.ash + x, b + m * g.bsn + (int64_t)y * g.bsh + x, g.asd,
                                g.bsd};
        F* o = out + (v * g.nz * g.h + y) * (int64_t)g.w + x;
        ssim_line(ld, g.d, g.z0, g.z0 + g.nz, win, carry + (int64_t)y * g.w + x, hw, g.z0 > 0, g.z0 + g.nz < g.d,
                  [&](int z, const double* q) {
#pragma unroll
                      for (int k = 0; k < kQ; ++k) o[k * g.cap + (int64_t)(z - g.z0) * hw] = (F)q[k];
                  });
    } else {
        if (t >= g.nvol * g.w) return;
        const int64_t p = t / g.w, m = g.m0 + p;
        const SsimSrcLine<T> ld{a + m * g.asn + x, b + m * g.bsn + x, g.ash, g.bsh};
        F* o = out + p * hw + x;
        ssim_line(ld, g.h, 0, g.h, win, nullptr, 0, false, false, [&](int y, const double* q) {
#pragma unroll
            for (int k = 0; k < kQ; ++k) o[k * g.cap + (int64_t)y * g.w] = (F)q[k];
        });
    }
}

// y pass of volumes: z buffer -> y buffer, one thread per (slice, x) line.
template <typename F>
__global__ void __launch_bounds__(256)
sk_ssim_y_pass_kernel(const F* __restrict__ in, F* __restrict__ out, SsimGeom g, SsimWin win) {
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    if (t >= g.nvol * g.nz * g.w) return;
    const int64_t base = t / g.w * g.h * g.w + t % g.w;
    const SsimBufLine<F> ld{in + base, g.w, g.cap};
    F* o = out + base;
    ssim_line(ld, g.h, 0, g.h, win, nullptr, 0, false, false, [&](int y, const double* q) {
#pragma unroll
        for (int k = 0; k < kQ; ++k) o[k * g.cap + (int64_t)y * g.w] = (F)q[k];
    });
}

// x pass: y buffer -> the filtered quantities of one row in the image's float type -> S in that type (upstream's
// element-wise order), stored in the map when one is given; rowsum[row] = float64 sum of S over the cropped interior
// (0 for a row outside it).
template <typename F>
__global__ void __launch_bounds__(256)
sk_ssim_x_pass_kernel(const F* __restrict__ in, SsimGeom g, SsimWin win, F cov_norm, F c1, F c2, int pad,
                      F* __restrict__ map, int64_t msn, int64_t msd, int64_t msh, double* __restrict__ rowsum) {
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    if (t >= g.nvol * g.nz * g.h) return;
    const int64_t k = t / g.h;
    const int y = (int)(t % g.h);
    const int64_t m = g.m0 + k / g.nz;
    const int z = g.z0 + (int)(k % g.nz);
    const bool row_in = y >= pad && y < g.h - pad && (g.nd == 2 || (z >= pad && z < g.d - pad));
    const SsimBufLine<F> ld{in + (k * g.h + y) * g.w, 1, g.cap};
    F* row = map ? map + m * msn + (int64_t)z * msd + (int64_t)y * msh : nullptr;
    const F two = F(2);
    double acc = 0.0;
    ssim_line(ld, g.w, 0, g.w, win, nullptr, 0, false, false, [&](int x, const double* q) {
        const F ux = (F)q[0], uy = (F)q[1], uxx = (F)q[2], uyy = (F)q[3], uxy = (F)q[4];
        const F vx = rn_mul(cov_norm, rn_sub(uxx, rn_mul(ux, ux)));
        const F vy = rn_mul(cov_norm, rn_sub(uyy, rn_mul(uy, uy)));
        const F vxy = rn_mul(cov_norm, rn_sub(uxy, rn_mul(ux, uy)));
        const F a1 = rn_add(rn_mul(rn_mul(two, ux), uy), c1);
        const F a2 = rn_add(rn_mul(two, vxy), c2);
        const F b1 = rn_add(rn_add(rn_mul(ux, ux), rn_mul(uy, uy)), c1);
        const F b2 = rn_add(rn_add(vx, vy), c2);
        const F s = rn_div(rn_mul(a1, a2), rn_mul(b1, b2));
        if (row) row[x] = s;
        if (row_in && x >= pad && x < g.w - pad) acc = __dadd_rn(acc, (double)s);
    });
    rowsum[t] = acc;
}

// One CTA per image of the chunk: mssim[image] += the fixed-order sum of its rows' sums.
__global__ void __launch_bounds__(256)
sk_ssim_fold_kernel(const double* __restrict__ rowsum, int64_t rows, int64_t m0, double* __restrict__ mssim) {
    __shared__ double s8[8];
    const int64_t v = blockIdx.x;
    double s = 0.0;
    for (int64_t j = threadIdx.x; j < rows; j += 256) s = __dadd_rn(s, rowsum[v * rows + j]);
    const double total = block_tree_256(s, s8);
    if (threadIdx.x == 0) mssim[m0 + v] = __dadd_rn(mssim[m0 + v], total);
}

// mode 0: mssim[m] = 0; mode 1: mssim[m] /= count (numpy's mean).
__global__ void sk_ssim_scale_kernel(double* mssim, int64_t n, double count, int mode) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) mssim[i] = mode ? __ddiv_rn(mssim[i], count) : 0.0;
}

// Images per chunk and slices of each, sized so that the chunk's float buffers stay within kSsimChunkBytes (at
// least one slice).
struct SsimPlan {
    int64_t vols;
    int nz;
    int64_t cap;   // voxels of a full chunk
};

static SsimPlan ssim_plan(int64_t n, int d, int h, int w, int nd, size_t fsz) {
    const int64_t hw = (int64_t)h * w;
    const int64_t slices = std::max<int64_t>(1, (int64_t)(kSsimChunkBytes / ((nd == 3 ? 2 : 1) * kQ * fsz)) / hw);
    SsimPlan p;
    if (d <= slices) {
        p.nz = d;
        p.vols = std::min<int64_t>(n, slices / d);
    } else {
        p.nz = (int)slices;
        p.vols = 1;
    }
    p.cap = p.vols * p.nz * hw;
    return p;
}

// carry (volumes), row sums, then the y buffer and (volumes) the z buffer.
static size_t ssim_workspace_bytes(int64_t n, int d, int h, int w, int nd, int src_dtype) {
    if (n <= 0 || d <= 0 || h <= 0 || w <= 0 || !valid_dtype(src_dtype)) return 0;
    const size_t fsz = src_dtype == MIE_F32 ? sizeof(float) : sizeof(double);
    const SsimPlan p = ssim_plan(n, d, h, w, nd, fsz);
    const size_t carry = nd == 3 ? align256((size_t)kQ * h * w * sizeof(double)) : 0;
    return carry + align256((size_t)p.vols * p.nz * h * sizeof(double)) + (nd == 3 ? 2 : 1) * align256(kQ * p.cap * fsz);
}

template <typename T, int ND>
static void ssim_launch(const T* a, const T* b, SsimGeom g, const SsimWin& win, int pad, double cov_norm, double c1,
                        double c2, void* map, int64_t msn, int64_t msd, int64_t msh, double* mssim, int64_t n,
                        uint8_t* ws, cudaStream_t st) {
    using F = SkFloat<T>;
    const SsimPlan p = ssim_plan(n, g.d, g.h, g.w, ND, sizeof(F));
    g.cap = p.cap;
    double* carry = (double*)ws;
    if (ND == 3) ws += align256((size_t)kQ * g.h * g.w * sizeof(double));
    double* rowsum = (double*)ws;
    ws += align256((size_t)p.vols * p.nz * g.h * sizeof(double));
    F* ybuf = (F*)ws;
    F* zbuf = (F*)(ws + align256(kQ * p.cap * sizeof(F)));
    const int64_t hw = (int64_t)g.h * g.w;
    auto blocks = [](int64_t threads) { return (unsigned)((threads + 255) / 256); };
    sk_ssim_scale_kernel<<<blocks(n), 256, 0, st>>>(mssim, n, 0.0, 0);
    for (int64_t m0 = 0; m0 < n; m0 += p.vols) {
        for (int z0 = 0; z0 < g.d; z0 += p.nz) {
            g.m0 = m0;
            g.nvol = std::min<int64_t>(p.vols, n - m0);
            g.z0 = z0;
            g.nz = std::min(p.nz, g.d - z0);
            const int64_t slices = g.nvol * g.nz;
            if (ND == 3) {
                sk_ssim_src_pass_kernel<T, 3><<<blocks(g.nvol * hw), 256, 0, st>>>(a, b, g, win, zbuf, carry);
                sk_ssim_y_pass_kernel<F><<<blocks(slices * g.w), 256, 0, st>>>(zbuf, ybuf, g, win);
            } else {
                sk_ssim_src_pass_kernel<T, 2><<<blocks(slices * g.w), 256, 0, st>>>(a, b, g, win, ybuf, carry);
            }
            sk_ssim_x_pass_kernel<F><<<blocks(slices * g.h), 256, 0, st>>>(ybuf, g, win, (F)cov_norm, (F)c1, (F)c2, pad,
                                                                          (F*)map, msn, msd, msh, rowsum);
            sk_ssim_fold_kernel<<<(unsigned)g.nvol, 256, 0, st>>>(rowsum, g.nz * (int64_t)g.h, m0, mssim);
        }
    }
    const double count = (double)(ND == 3 ? g.d - 2 * pad : 1) * (double)(g.h - 2 * pad) * (double)(g.w - 2 * pad);
    sk_ssim_scale_kernel<<<blocks(n), 256, 0, st>>>(mssim, n, count, 1);
}

// Checks after the layout checks of the entry points, then the launches.
static int ssim_run(const void* a, const void* b, void* map, int src_dtype, int map_dtype, int64_t n, int d, int h, int w,
                    int nd, int64_t asn, int64_t asd, int64_t ash, int64_t bsn, int64_t bsd, int64_t bsh, int64_t msn,
                    int64_t msd, int64_t msh, int win_size, const double* taps, int ntaps, double cov_norm, double c1,
                    double c2, double* mssim, void* workspace, size_t workspace_bytes, void* stream) {
    if (!valid_dtype(src_dtype)) return MIE_E_DTYPE;
    if (map && map_dtype != (src_dtype == MIE_F32 ? MIE_F32 : MIE_F64)) return MIE_E_DTYPE;
    if (win_size < 1 || win_size > MIE_MAX_TAPS || win_size % 2 == 0) return MIE_E_KERNEL;
    if (taps && (ntaps < 1 || ntaps > MIE_MAX_TAPS || ntaps % 2 == 0)) return MIE_E_KERNEL;
    if ((nd == 3 && d < win_size) || h < win_size || w < win_size) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    if (!mssim || !workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < ssim_workspace_bytes(n, d, h, w, nd, src_dtype)) return MIE_E_WORKSPACE;
    SsimWin win{};
    if (taps) {
        win.size = 0;
        win.r = ntaps / 2;
        for (int i = 0; i < ntaps; ++i) win.w[i] = taps[i];
    } else {
        win.size = win_size;
        win.r = win_size / 2;
    }
    SsimGeom g{};
    g.nd = nd; g.d = d; g.h = h; g.w = w;
    g.asn = asn; g.asd = asd; g.ash = ash; g.bsn = bsn; g.bsd = bsd; g.bsh = bsh;
    const int pad = (win_size - 1) / 2;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)workspace;
    MIE_DISPATCH_SRC(src_dtype, {
        if (nd == 3)
            ssim_launch<SrcT, 3>((const SrcT*)a, (const SrcT*)b, g, win, pad, cov_norm, c1, c2, map, msn, msd, msh, mssim,
                                 n, ws, st);
        else
            ssim_launch<SrcT, 2>((const SrcT*)a, (const SrcT*)b, g, win, pad, cov_norm, c1, c2, map, msn, msd, msh, mssim,
                                 n, ws, st);
    });
    return check_launch();
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_sk_structural_similarity_workspace_bytes(int64_t n, int h, int w, int src_dtype) {
    return ssim_workspace_bytes(n, 1, h, w, 2, src_dtype);
}

size_t mie_sk_structural_similarity3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype) {
    return ssim_workspace_bytes(n, d, h, w, 3, src_dtype);
}

int mie_sk_structural_similarity(const void* a, const void* b, void* map, int src_dtype, int map_dtype, int64_t n, int h,
                                 int w, int64_t a_stride_n, int64_t a_stride_h, int64_t b_stride_n, int64_t b_stride_h,
                                 int64_t map_stride_n, int64_t map_stride_h, int win_size, const double* taps, int ntaps,
                                 double cov_norm, double c1, double c2, double* mssim, void* workspace,
                                 size_t workspace_bytes, void* stream) {
    int rc = check_planes({a, src_dtype, a_stride_n, a_stride_h}, {b, src_dtype, b_stride_n, b_stride_h}, n, h, w);
    if (rc) return rc;
    if (map && !plane_strides_ok({map, map_dtype, map_stride_n, map_stride_h}, n, h, w)) return MIE_E_STRIDE;
    return ssim_run(a, b, map, src_dtype, map_dtype, n, 1, h, w, 2, a_stride_n, 0, a_stride_h, b_stride_n, 0, b_stride_h,
                    map_stride_n, 0, map_stride_h, win_size, taps, ntaps, cov_norm, c1, c2, mssim, workspace,
                    workspace_bytes, stream);
}

int mie_sk_structural_similarity3d(const void* a, const void* b, void* map, int src_dtype, int map_dtype, int64_t n,
                                   int d, int h, int w, int64_t a_stride_n, int64_t a_stride_d, int64_t a_stride_h,
                                   int64_t b_stride_n, int64_t b_stride_d, int64_t b_stride_h, int64_t map_stride_n,
                                   int64_t map_stride_d, int64_t map_stride_h, int win_size, const double* taps,
                                   int ntaps, double cov_norm, double c1, double c2, double* mssim, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    int rc = check_volumes({a, src_dtype, a_stride_n, a_stride_h}, a_stride_d, {b, src_dtype, b_stride_n, b_stride_h},
                           b_stride_d, n, d, h, w);
    if (rc) return rc;
    if (map && !volume_strides_ok({map, map_dtype, map_stride_n, map_stride_h}, map_stride_d, n, d, h, w))
        return MIE_E_STRIDE;
    return ssim_run(a, b, map, src_dtype, map_dtype, n, d, h, w, 3, a_stride_n, a_stride_d, a_stride_h, b_stride_n,
                    b_stride_d, b_stride_h, map_stride_n, map_stride_d, map_stride_h, win_size, taps, ntaps, cov_norm,
                    c1, c2, mssim, workspace, workspace_bytes, stream);
}

}  // extern "C"
