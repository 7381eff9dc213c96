// sk_tv.cu — skimage.restoration.denoise_tv_chambolle on planes (ndim 2) and whole volumes (ndim 3).
//
// RECALLED semantics (include/mie.h; the reference is the numpy transcription tests/sk_tv_chambolle_twin.py).  Every
// per-element step is one correctly rounded IEEE operation in upstream's order, written with explicit __d*_rn / __f*_rn
// so that nvcc cannot contract to fma: the result equals the twin bit for bit whenever the iteration counts agree.  Only
// the two energy sums differ from numpy's (fixed-order float64 sums here, pairwise there); they feed the stopping test
// alone.
//
// One launch per pass over the whole batch.  Pass i reads p from ping-pong buffer i % 2 (pass 0 reads none: p = 0),
// writes the updated p to buffer (i + 1) % 2 and one pair of partial energy sums per CTA.  The last CTA of an image to
// arrive reduces that image's partials in a fixed order and runs the stopping test, so the same input gives the same
// bits and counts on every run.  A stopped image's CTAs return at once in later passes.  The result of the stopping
// pass `last` is image + div(p entering it), which is buffer last % 2 — never overwritten after the image stops — so a
// finishing launch writes it.  Pass max_num_iter - 1 needs no launch of its own: its p update is discarded and its
// stopping test cannot change the result.
#include <climits>
#include <cmath>
#include <type_traits>

#include "mie_common.cuh"

namespace mie {

__device__ __forceinline__ float tv_add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double tv_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float tv_sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double tv_sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float tv_mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double tv_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float tv_div(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double tv_div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float tv_sqrt(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double tv_sqrt(double a) { return __dsqrt_rn(a); }

// The image's float type: float64 for integer images (img_as_float), float32 for float32 images.
template <typename T>
using TvF = typename std::conditional<std::is_same<T, float>::value, float, double>::type;

// Per-image state, re-initialised by every call.
struct TvState {
    double e_init, e_prev;   // energies, held exactly in double whatever the image's float type
    int done;                // stopping test met: later passes skip the image
    int last;                // index of the pass whose out is the result
    unsigned arrived;        // CTAs of the current pass that have written their partial sums
    int pad_;
};

// CTA tile: 32 columns x 8 rows x 16 slices for volumes (a thread walks z), 32 x 32 for planes (a thread takes every
// 8th row).  p component a of image m, voxel v sits at p + a * n * vox + m * vox + v (dense, whatever the layouts).
constexpr int kTvTx = 32, kTvRows = 8, kTvZ = 16, kTvPlaneSteps = 4;

struct TvGeom {
    int d, h, w;              // d == 1 for planes
    int ntx, nty;             // tiles along x and y
    int64_t tiles;            // tiles per image
    int64_t vox;              // d * h * w
    int64_t n;
    int64_t ssn, ssd, ssh;    // source strides (elements)
};

template <typename T>
__device__ __forceinline__ TvF<T> tv_src(const T* src, int64_t off) {
    if constexpr (std::is_same<T, float>::value) return src[off];
    else return skb_as_float<T>((int)src[off]);
}

// out = image + d at voxel (z, y, x) of image m, with d = -(p0 + p1 [+ p2]) and then, axis by axis, + p_a(x - e_a)
// where the coordinate along a is >= 1; on the first pass p = 0 and upstream takes out = image.  Axis order is the
// array's: (z, y, x) for volumes, (y, x) for planes.  *dval receives d.
template <typename T, int ND>
__device__ __forceinline__ TvF<T> tv_out(const T* src, const TvF<T>* p, const TvGeom& g, int64_t m, int z, int y, int x,
                                         bool first, TvF<T>* dval) {
    using F = TvF<T>;
    const F im = tv_src<T>(src, m * g.ssn + (int64_t)z * g.ssd + (int64_t)y * g.ssh + x);
    if (first) {
        *dval = F(0);
        return im;
    }
    const int64_t cs = g.n * g.vox;
    const int64_t v = m * g.vox + ((int64_t)z * g.h + y) * g.w + x;
    const int coord[3] = {ND == 3 ? z : y, ND == 3 ? y : x, x};
    const int64_t step[3] = {ND == 3 ? (int64_t)g.h * g.w : (int64_t)g.w, ND == 3 ? (int64_t)g.w : 1, 1};
    F s = p[v];
#pragma unroll
    for (int a = 1; a < ND; ++a) s = tv_add(s, p[a * cs + v]);
    F d = -s;
#pragma unroll
    for (int a = 0; a < ND; ++a)
        if (coord[a] >= 1) d = tv_add(d, p[a * cs + v - step[a]]);
    *dval = d;
    return tv_add(im, d);
}

// Fixed-order sum of (a, b) over the CTA (256 threads); the totals land in thread 0.
__device__ __forceinline__ void tv_block_sum2(double& a, double& b, double* s) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        a += __shfl_down_sync(0xffffffffu, a, o);
        b += __shfl_down_sync(0xffffffffu, b, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s[warp] = a; s[8 + warp] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = s[0]; b = s[8];
        for (int i = 1; i < 8; ++i) { a += s[i]; b += s[8 + i]; }
    }
}

// The voxels of one thread: (z0 + k, y, x) for volumes, (0, y + 8k, x) for planes.
template <int ND>
__device__ __forceinline__ void tv_voxel(const TvGeom& g, int64_t tile, int k, int& z, int& y, int& x) {
    const int64_t tx = tile % g.ntx, r = tile / g.ntx;
    x = (int)tx * kTvTx + (threadIdx.x & 31);
    const int row = threadIdx.x >> 5;
    if constexpr (ND == 3) {
        y = (int)(r % g.nty) * kTvRows + row;
        z = (int)(r / g.nty) * kTvZ + k;
    } else {
        y = (int)r * (kTvRows * kTvPlaneSteps) + row + kTvRows * k;
        z = 0;
    }
}

template <int ND>
__host__ __device__ constexpr int tv_steps() { return ND == 3 ? kTvZ : kTvPlaneSteps; }

// One pass of the loop (pass index `iter`, first == (iter == 0)) over every image of the batch that has not stopped.
template <typename T, int ND>
__global__ void __launch_bounds__(256)
sk_tv_pass_kernel(const T* __restrict__ src, const TvF<T>* __restrict__ p_in, TvF<T>* __restrict__ p_out, TvGeom g,
                  int iter, TvF<T> tau, TvF<T> tau_w, double weight, double eps, TvState* state, double2* partials) {
    using F = TvF<T>;
    __shared__ double s_red[16];
    __shared__ int s_last;
    const int64_t m = blockIdx.x / g.tiles, tile = blockIdx.x % g.tiles;
    if (state[m].done) return;
    const bool first = iter == 0;
    const int64_t cs = g.n * g.vox;
    const int lim[3] = {ND == 3 ? g.d : g.h, ND == 3 ? g.h : g.w, g.w};
    double sd = 0.0, sn = 0.0;
    F o_next = F(0), d_next = F(0);
    bool have_next = false;   // volumes: out at (z + 1, y, x) from the previous step
#pragma unroll 1
    for (int k = 0; k < tv_steps<ND>(); ++k) {
        int z, y, x;
        tv_voxel<ND>(g, tile, k, z, y, x);
        if (x >= g.w || y >= g.h || z >= g.d) break;
        F d0, o;
        if (have_next) { o = o_next; d0 = d_next; }
        else o = tv_out<T, ND>(src, p_in, g, m, z, y, x, first, &d0);
        sd += (double)tv_mul(d0, d0);
        const int coord[3] = {ND == 3 ? z : y, ND == 3 ? y : x, x};
        F gr[ND];
#pragma unroll
        for (int a = 0; a < ND; ++a) {
            gr[a] = F(0);
            if (coord[a] < lim[a] - 1) {
                const int nz = z + (ND == 3 && a == 0), ny = y + ((ND == 3 && a == 1) || (ND == 2 && a == 0)),
                          nx = x + (a == ND - 1);
                F dn;
                const F on = tv_out<T, ND>(src, p_in, g, m, nz, ny, nx, first, &dn);
                gr[a] = tv_sub(on, o);
                if (ND == 3 && a == 0) { o_next = on; d_next = dn; }
            }
        }
        have_next = ND == 3 && coord[0] < lim[0] - 1;
        F q = tv_mul(gr[0], gr[0]);
#pragma unroll
        for (int a = 1; a < ND; ++a) q = tv_add(q, tv_mul(gr[a], gr[a]));
        const F nrm = tv_sqrt(q);
        sn += (double)nrm;
        const F den = tv_add(tv_mul(nrm, tau_w), F(1));
        const int64_t v = m * g.vox + ((int64_t)z * g.h + y) * g.w + x;
#pragma unroll
        for (int a = 0; a < ND; ++a) {
            const F pv = first ? F(0) : p_in[a * cs + v];
            p_out[a * cs + v] = tv_div(tv_sub(pv, tv_mul(tau, gr[a])), den);
        }
    }
    tv_block_sum2(sd, sn, s_red);
    if (threadIdx.x == 0) {
        partials[m * g.tiles + tile] = make_double2(sd, sn);
        __threadfence();
        s_last = atomicAdd(&state[m].arrived, 1u) == (unsigned)(g.tiles - 1);
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // last CTA of image m: reduce its partials in index order, then the scalar steps in the image's float type
    double td = 0.0, tn = 0.0;
    for (int64_t j = threadIdx.x; j < g.tiles; j += 256) {
        const double2 pr = __ldcg(partials + m * g.tiles + j);
        td += pr.x;
        tn += pr.y;
    }
    __syncthreads();
    tv_block_sum2(td, tn, s_red);
    if (threadIdx.x == 0) {
        TvState& st = state[m];
        F e = tv_add((F)td, tv_mul((F)weight, (F)tn));
        e = tv_div(e, (F)(double)g.vox);
        if (first) {
            st.e_init = e;
            st.e_prev = e;
        } else if (fabs(tv_sub((F)st.e_prev, e)) < tv_mul((F)eps, (F)st.e_init)) {
            st.done = 1;
            st.last = iter;
        } else {
            st.e_prev = e;
        }
        st.arrived = 0;
    }
}

__global__ void sk_tv_init_kernel(TvState* state, int64_t n, int last) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) state[i] = TvState{0.0, 0.0, 0, last, 0u, 0};
}

// dst = image + div(p entering pass `last`) of every image; iters[m] = last + 1 when iters is given.
template <typename T, typename DstT, int ND>
__global__ void __launch_bounds__(256)
sk_tv_finish_kernel(const T* __restrict__ src, const TvF<T>* __restrict__ p0, const TvF<T>* __restrict__ p1, TvGeom g,
                    DstT* __restrict__ dst, int64_t dsn, int64_t dsd, int64_t dsh, const TvState* state, int* iters) {
    using F = TvF<T>;
    const int64_t m = blockIdx.x / g.tiles, tile = blockIdx.x % g.tiles;
    const int last = state[m].last;
    if (iters && tile == 0 && threadIdx.x == 0) iters[m] = last + 1;
    const F* p = (last & 1) ? p1 : p0;
#pragma unroll 1
    for (int k = 0; k < tv_steps<ND>(); ++k) {
        int z, y, x;
        tv_voxel<ND>(g, tile, k, z, y, x);
        if (x >= g.w || y >= g.h || z >= g.d) break;
        F d;
        const F o = tv_out<T, ND>(src, p, g, m, z, y, x, last == 0, &d);
        dst[m * dsn + (int64_t)z * dsd + (int64_t)y * dsh + x] = (DstT)o;
    }
}

static inline int64_t tv_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

static TvGeom tv_geom(int64_t n, int d, int h, int w, int nd) {
    TvGeom g{};
    g.d = d; g.h = h; g.w = w; g.n = n;
    const int64_t ntx = tv_cdiv(w, kTvTx);
    const int64_t nty = tv_cdiv(h, nd == 3 ? kTvRows : kTvRows * kTvPlaneSteps);
    const int64_t ntz = nd == 3 ? tv_cdiv(d, kTvZ) : 1;
    g.ntx = (int)ntx; g.nty = (int)nty;
    g.tiles = ntx * nty * ntz;
    g.vox = (int64_t)d * h * w;
    return g;
}

static size_t tv_workspace_bytes(int64_t n, int d, int h, int w, int nd, int src_dtype) {
    if (n <= 0 || d <= 0 || h <= 0 || w <= 0 || !valid_dtype(src_dtype)) return 0;
    const TvGeom g = tv_geom(n, d, h, w, nd);
    const size_t fsz = src_dtype == MIE_F32 ? sizeof(float) : sizeof(double);
    return align256((size_t)n * sizeof(TvState)) + align256((size_t)n * g.tiles * sizeof(double2)) +
           2 * (size_t)nd * (size_t)n * (size_t)g.vox * fsz;
}

template <typename T, int ND>
static void tv_launch(const T* src, void* dst, int dst_dtype, TvGeom g, int64_t dsn, int64_t dsd, int64_t dsh,
                      double weight, double eps, int max_num_iter, int* iters, uint8_t* ws, cudaStream_t st) {
    using F = TvF<T>;
    TvState* state = (TvState*)ws;
    ws += align256((size_t)g.n * sizeof(TvState));
    double2* partials = (double2*)ws;
    ws += align256((size_t)g.n * g.tiles * sizeof(double2));
    F* p[2] = {(F*)ws, (F*)ws + ND * g.n * g.vox};
    const double tau = 1.0 / (2.0 * ND);
    const unsigned blocks = (unsigned)(g.n * g.tiles);
    sk_tv_init_kernel<<<(unsigned)((g.n + 255) / 256), 256, 0, st>>>(state, g.n, max_num_iter - 1);
    for (int i = 0; i + 1 < max_num_iter; ++i)
        sk_tv_pass_kernel<T, ND><<<blocks, 256, 0, st>>>(src, p[i & 1], p[(i + 1) & 1], g, i, (F)tau, (F)(tau / weight),
                                                          weight, eps, state, partials);
    if (dst_dtype == MIE_F32)
        sk_tv_finish_kernel<T, float, ND><<<blocks, 256, 0, st>>>(src, p[0], p[1], g, (float*)dst, dsn, dsd, dsh, state, iters);
    else
        sk_tv_finish_kernel<T, double, ND><<<blocks, 256, 0, st>>>(src, p[0], p[1], g, (double*)dst, dsn, dsd, dsh, state, iters);
}

// Checks after the layout checks of the entry points, then the launches.
static int tv_run(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w, int nd,
                  int64_t ssn, int64_t ssd, int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, double weight, double eps,
                  int max_num_iter, int* iters, void* workspace, size_t workspace_bytes, void* stream) {
    if (!valid_dtype(src_dtype) || (dst_dtype != MIE_F32 && dst_dtype != MIE_F64)) return MIE_E_DTYPE;
    if (!(weight > 0.0) || !std::isfinite(weight)) return MIE_E_RANGE;
    if (max_num_iter < 1) return MIE_E_SHAPE;
    TvGeom g = tv_geom(n, d, h, w, nd);
    if (n * g.tiles > INT_MAX) return MIE_E_SHAPE;   // one CTA per tile on a flat grid
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < tv_workspace_bytes(n, d, h, w, nd, src_dtype)) return MIE_E_WORKSPACE;
    g.ssn = ssn; g.ssd = ssd; g.ssh = ssh;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)workspace;
    MIE_DISPATCH_SRC(src_dtype, {
        if (nd == 3) tv_launch<SrcT, 3>((const SrcT*)src, dst, dst_dtype, g, dsn, dsd, dsh, weight, eps, max_num_iter, iters, ws, st);
        else tv_launch<SrcT, 2>((const SrcT*)src, dst, dst_dtype, g, dsn, dsd, dsh, weight, eps, max_num_iter, iters, ws, st);
    });
    return check_launch();
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_sk_tv_chambolle_workspace_bytes(int64_t n, int h, int w, int src_dtype) {
    return tv_workspace_bytes(n, 1, h, w, 2, src_dtype);
}

size_t mie_sk_tv_chambolle3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype) {
    return tv_workspace_bytes(n, d, h, w, 3, src_dtype);
}

int mie_sk_denoise_tv_chambolle(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                                int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                                double weight, double eps, int max_num_iter, int* iters, void* workspace,
                                size_t workspace_bytes, void* stream) {
    const int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h},
                                n, h, w);
    if (rc) return rc;
    return tv_run(src, dst, src_dtype, dst_dtype, n, 1, h, w, 2, src_stride_n, 0, src_stride_h, dst_stride_n, 0,
                  dst_stride_h, weight, eps, max_num_iter, iters, workspace, workspace_bytes, stream);
}

int mie_sk_denoise_tv_chambolle3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                                  int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                                  int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                                  double weight, double eps, int max_num_iter, int* iters, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    const int rc = check_volumes({src, src_dtype, src_stride_n, src_stride_h}, src_stride_d,
                                 {dst, dst_dtype, dst_stride_n, dst_stride_h}, dst_stride_d, n, d, h, w);
    if (rc) return rc;
    return tv_run(src, dst, src_dtype, dst_dtype, n, d, h, w, 3, src_stride_n, src_stride_d, src_stride_h, dst_stride_n,
                  dst_stride_d, dst_stride_h, weight, eps, max_num_iter, iters, workspace, workspace_bytes, stream);
}

}  // extern "C"
