// sk_ridges.cu — skimage.filters.frangi / hessian / sato / meijering and skimage.feature.hessian_matrix /
// hessian_matrix_eigvals on planes (ndim 2) and whole volumes (ndim 3).
//
// RECALLED semantics (include/mie.h; the reference is the numpy transcription tests/sk_ridges_twin.py).  Per scale the
// Hessian elements are Gaussian-derivative filters composed as upstream composes them: G_a = gaussian_filter(image,
// order e_a), H_ab = gaussian_filter(G_a, order e_b), each N-D filter a 1-D pass along z, then y, then x with scipy's
// line arithmetic in float64 and the values rounded to the image's float type F between passes.  Every step is one
// correctly rounded operation, so the elements equal scipy's bit for bit.  Passes that share a prefix run once: a
// volume's scale takes 24 passes instead of 27, a plane's 10.
//
// A pass is one thread per output: the taps of its line in scipy's pairing (symmetric for order 0, antisymmetric for
// order 1), the line extended by the border mode.  After the passes an epilogue launch per scale computes the
// eigenvalues (the closed form of 2x2, a cyclic Jacobi in float64 for 3x3), the filter's formula and the running
// maximum over scales; another launch before it takes a per-image maximum when the scale needs one.  frangi's
// implicit gamma (the first scale's max of s) and meijering's per-scale maximum are per-image maxima of non-negative
// values, taken as integer atomicMax on their bit patterns: order-independent, so repeated runs give the same bits.
//
// The batch runs in chunks of whole images of at most kRidgeChunkVoxels voxels (one image if it is larger), all scales
// of a chunk before the next, so the workspace depends on one image's size and not on n.
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "mie_common.cuh"

namespace mie {

constexpr int kRidgeMaxTaps = 2 * MIE_SK_RIDGE_MAX_RADIUS + 1;
constexpr int64_t kRidgeChunkVoxels = (int64_t)1 << 24;
constexpr int64_t kRidgeMaxChunkImages = 65535;           // grid.y of the epilogue

// One pass's correlation weights w[0 .. 2r] (scipy's order: out[i] = sum_j w[j + r] ext[i + j]).
struct RidgeTaps {
    int r, anti;
    double w[kRidgeMaxTaps];
};

// Image m, voxel (z, y, x) at p + m sn + z sd + y sh + x.
template <typename T>
struct RVol {
    T* p;
    int64_t sn, sd, sh;
};

// Source value as the image's float type F: raw (the ridge filters' image.astype(F)) or img_as_float (hessian_matrix),
// negated for black_ridges=False.
template <typename T, typename F>
__device__ __forceinline__ double ridge_load(T v, int as_float, int neg) {
    F f;
    if constexpr (std::is_floating_point<T>::value) {
        f = (F)v;
    } else {
        f = as_float ? (F)skb_as_float<T>((int)v) : (F)v;
    }
    return (double)(neg ? -f : f);
}

// One 1-D Gaussian-derivative pass along AX (0 z, 1 y, 2 x) of images 0 .. nimg - 1: scipy's correlate1d with
// tmp = ext[c] w[r], then tmp += (ext[c + j] +/- ext[c - j]) w[j + r] for j = -r .. -1, rounded to F.
template <typename T, typename F, int AX>
__global__ void __launch_bounds__(256)
sk_ridge_pass_kernel(RVol<const T> in, RVol<F> out, int64_t nimg, int d, int h, int w, RidgeTaps k, int mode,
                     double cval, int as_float, int neg) {
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    const int64_t hw = (int64_t)h * w;
    if (t >= nimg * d * hw) return;
    const int x = (int)(t % w);
    const int y = (int)(t / w % h);
    const int z = (int)(t / hw % d);
    const int64_t m = t / (hw * d);
    const T* base = in.p + m * in.sn + (int64_t)z * in.sd + (int64_t)y * in.sh + x;
    const int i = AX == 0 ? z : (AX == 1 ? y : x);
    const int n = AX == 0 ? d : (AX == 1 ? h : w);
    const int64_t s = AX == 0 ? in.sd : (AX == 1 ? in.sh : 1);
    auto ld = [&](int j) -> double {
        int q = i + j;
        if (q < 0 || q >= n) {
            q = border_index(q, n, mode);
            if (q < 0) return cval;
        }
        return ridge_load<T, F>(base[(int64_t)(q - i) * s], as_float, neg);
    };
    double tmp = __dmul_rn(ld(0), k.w[k.r]);
    if (k.anti) {
#pragma unroll 1
        for (int j = -k.r; j < 0; ++j) tmp = __dadd_rn(tmp, __dmul_rn(__dsub_rn(ld(j), ld(-j)), k.w[j + k.r]));
    } else {
#pragma unroll 1
        for (int j = -k.r; j < 0; ++j) tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(ld(j), ld(-j)), k.w[j + k.r]));
    }
    out.p[m * out.sn + (int64_t)z * out.sd + (int64_t)y * out.sh + x] = (F)tmp;
}

// ---------------------------------------------------------------- eigenvalues
// np.maximum: NaN if either is NaN, else the larger (the first on equality).
template <typename F>
__device__ __forceinline__ F np_max(F a, F b) { return (b != b || b > a) ? b : a; }

// 2x2: upstream's closed form in F, (m + hs, m - hs) with m = (M00 + M11) / 2, hs = sqrt(M01^2 + ((M00 - M11) / 2)^2).
template <typename F>
__device__ __forceinline__ void eig2(F a, F b, F c, F* e) {
    const F m = rn_div(rn_add(a, c), F(2));
    const F q = rn_div(rn_sub(a, c), F(2));
    const F hs = rn_sqrt(rn_add(rn_mul(b, b), rn_mul(q, q)));
    e[0] = rn_add(m, hs);
    e[1] = rn_sub(m, hs);
}

// One Jacobi rotation annihilating a[P][Q] (Rutishauser's formulas); a negligible a[P][Q] is set to zero.
template <int P, int Q>
__device__ __forceinline__ void jacobi_rot(double (&a)[3][3]) {
    constexpr int R = 3 - P - Q;
    const double apq = a[P][Q];
    if (apq == 0.0) return;
    const double app = a[P][P], aqq = a[Q][Q];
    const double g = 100.0 * fabs(apq);
    if (fabs(app) + g == fabs(app) && fabs(aqq) + g == fabs(aqq)) {
        a[P][Q] = a[Q][P] = 0.0;
        return;
    }
    const double theta = 0.5 * (aqq - app) / apq;
    double t;
    if (fabs(theta) > 1e150) t = 0.5 / theta;
    else t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
    const double c = 1.0 / sqrt(t * t + 1.0), s = t * c, tau = s / (1.0 + c);
    a[P][P] = app - t * apq;
    a[Q][Q] = aqq + t * apq;
    a[P][Q] = a[Q][P] = 0.0;
    const double arp = a[R][P], arq = a[R][Q];
    a[R][P] = a[P][R] = arp - s * (arq + tau * arp);
    a[R][Q] = a[Q][R] = arq + s * (arp - tau * arq);
}

// 3x3 symmetric: cyclic Jacobi in float64 (absolute error a few ulp of the largest |eigenvalue|), decreasing order.
__device__ __forceinline__ void eig3(double a00, double a01, double a02, double a11, double a12, double a22,
                                     double* e) {
    double a[3][3] = {{a00, a01, a02}, {a01, a11, a12}, {a02, a12, a22}};
#pragma unroll 1
    for (int sweep = 0; sweep < 32; ++sweep) {
        if (a[0][1] == 0.0 && a[0][2] == 0.0 && a[1][2] == 0.0) break;
        jacobi_rot<0, 1>(a);
        jacobi_rot<0, 2>(a);
        jacobi_rot<1, 2>(a);
    }
    double x = a[0][0], y = a[1][1], z = a[2][2], u;
    if (x < y) { u = x; x = y; y = u; }
    if (y < z) { u = y; y = z; z = u; }
    if (x < y) { u = x; x = y; y = u; }
    e[0] = x; e[1] = y; e[2] = z;
}

// Eigenvalues in decreasing order of the Hessian at chunk offset v (elements in upstream's order).
template <typename F, int ND>
__device__ __forceinline__ void hessian_eig(const F* const* H, int64_t v, F* e) {
    if constexpr (ND == 2) {
        eig2<F>(H[0][v], H[1][v], H[2][v], e);
    } else {
        double d[3];
        eig3(H[0][v], H[1][v], H[2][v], H[3][v], H[4][v], H[5][v], d);
        e[0] = (F)d[0]; e[1] = (F)d[1]; e[2] = (F)d[2];
    }
}

// ---------------------------------------------------------------- filters
template <typename F> struct RBits;
template <> struct RBits<double> {
    using type = unsigned long long;
    static __device__ __forceinline__ type of(double v) { return (unsigned long long)__double_as_longlong(v); }
    static __device__ __forceinline__ double value(type b) { return __longlong_as_double((long long)b); }
};
template <> struct RBits<float> {
    using type = unsigned int;
    static __device__ __forceinline__ type of(float v) { return __float_as_uint(v); }
    static __device__ __forceinline__ float value(type b) { return __uint_as_float(b); }
};

enum RidgePhase { kPhaseGamma = 0, kPhaseMeijering = 1, kPhaseFinal = 2 };

template <typename F>
struct RidgeEpi {
    const F* H[6];                 // dense chunk buffers, upstream's element order
    void* M;                       // running maximum over scales (chunk buffer of RidgeMax<F, ND>)
    F* V;                          // meijering: this scale's values (chunk buffer)
    typename RBits<F>::type* gmax; // per chunk image: frangi's first-scale max of s
    typename RBits<F>::type* vmax; // per chunk image: meijering's max of this scale
    int64_t vox;                   // voxels per image
    int d, h, w;
    int filter, phase, first, last, implicit_gamma;
    double ca, cb, cg;             // 2 alpha^2, 2 beta^2, 2 gamma^2 (explicit gamma)
    double sig2, malpha;           // sato: sigma^2; meijering: alpha
};

// frangi's (or hessian's) vals and s of one voxel; e in decreasing order.
// exp of an F value: float through double, so that results in float's subnormal range are not flushed to zero (numpy
// keeps them, and hessian's out[out <= 0] = 1 tells 0 from a subnormal).
__device__ __forceinline__ double rexp(double x) { return exp(x); }
__device__ __forceinline__ float rexp(float x) { return (float)exp((double)x); }

// The type upstream's running maximum ends up in: for planes, frangi's first factor is the float64 scalar
// 1 - exp(-inf), so from there on its values are float64 whatever F is (NumPy 2 promotion); volumes stay in F.
template <typename F, int ND>
using RidgeMax = typename std::conditional<ND == 2, double, F>::type;

// s_only: the first scale's s, for the implicit gamma.
template <typename F, int ND>
__device__ __forceinline__ RidgeMax<F, ND> frangi_vals(const F* e, F ca, F cb, F cg, bool s_only) {
    // take_along_axis(e, abs(e).argsort(0), 0): a stable sort by |e|, ascending
    F l[3] = {e[0], e[1], ND == 3 ? e[2] : F(0)};
#pragma unroll
    for (int i = 1; i < ND; ++i) {
#pragma unroll
        for (int j = i; j > 0; --j) {
            if (fabs(l[j - 1]) > fabs(l[j])) { const F u = l[j]; l[j] = l[j - 1]; l[j - 1] = u; }
        }
    }
    const F tiny = F(1e-10);
    F s2 = rn_add(rn_mul(l[0], l[0]), rn_mul(l[1], l[1]));
    if (ND == 3) s2 = rn_add(s2, rn_mul(l[2], l[2]));
    const F s = rn_sqrt(s2);
    if (s_only) return s;
    const F l2 = np_max(l[1], tiny);
    using R = RidgeMax<F, ND>;
    R vals;
    F rb;
    if constexpr (ND == 2) {
        rb = rn_div(fabs(l[0]), l2);
        vals = R(1);   // 1 - exp(-inf)
    } else {
        const F l3 = np_max(l[2], tiny);
        const F ra = rn_div(l2, l3);
        rb = rn_div(fabs(l[0]), rn_sqrt(rn_mul(l2, l3)));
        vals = rn_sub(F(1), rexp(rn_div(-rn_mul(ra, ra), ca)));
    }
    vals = rn_mul(vals, (R)rexp(rn_div(-rn_mul(rb, rb), cb)));
    vals = rn_mul(vals, (R)rn_sub(F(1), rexp(rn_div(-rn_mul(s, s), cg))));
    return vals;
}

template <typename F, int ND>
__device__ __forceinline__ F meijering_vals(const F* e, F a) {
    F best = F(0), babs = F(-1);
#pragma unroll
    for (int i = 0; i < ND; ++i) {
        F v = F(0);
#pragma unroll
        for (int j = 0; j < ND; ++j) v = rn_add(v, rn_mul(i == j ? F(1) : a, e[j]));
        if (fabs(v) > babs || (babs < F(0))) { best = v; babs = fabs(v); }
    }
    return np_max(best, F(0));
}

// One launch per scale (and phase): grid (x over the voxels of an image, y over the chunk's images).
template <typename F, typename D, int ND>
__global__ void __launch_bounds__(256)
sk_ridge_epilogue_kernel(RidgeEpi<F> p, RVol<D> dst) {
    using B = RBits<F>;
    using R = RidgeMax<F, ND>;
    R* M = (R*)p.M;
    __shared__ typename B::type smax[8];
    const int64_t m = blockIdx.y;
    const int64_t hw = (int64_t)p.h * p.w;
    F ca = (F)p.ca, cb = (F)p.cb, cg = (F)p.cg;
    if (p.implicit_gamma && p.phase == kPhaseFinal) {
        F g = rn_div(B::value(p.gmax[m]), F(2));
        if (g == F(0)) g = F(1);
        cg = rn_mul(F(2), rn_mul(g, g));
    }
    F vmax = F(0);
    if (p.filter == MIE_SK_MEIJERING && p.phase == kPhaseFinal) vmax = B::value(p.vmax[m]);
    typename B::type red = 0;
    for (int64_t i = blockIdx.x * 256LL + threadIdx.x; i < p.vox; i += (int64_t)gridDim.x * 256) {
        const int64_t v = m * p.vox + i;
        R vals;
        if (p.filter == MIE_SK_MEIJERING && p.phase == kPhaseFinal) {
            vals = vmax > F(0) ? rn_div(p.V[v], vmax) : p.V[v];
        } else {
            F e[3];
            hessian_eig<F, ND>(p.H, v, e);
            if (p.filter == MIE_SK_SATO) {
                const F r = ND == 2 ? np_max(e[0], F(0)) : rn_sqrt(rn_mul(np_max(e[0], F(0)), np_max(e[1], F(0))));
                vals = rn_mul((F)p.sig2, r);
            } else if (p.filter == MIE_SK_MEIJERING) {
                vals = meijering_vals<F, ND>(e, (F)p.malpha);
            } else if (p.phase == kPhaseGamma) {
                vals = frangi_vals<F, ND>(e, ca, cb, cg, true);
            } else {
                vals = frangi_vals<F, ND>(e, ca, cb, cg, false);
            }
        }
        if (p.phase != kPhaseFinal) {
            const F fv = (F)vals;   // exact: these phases compute in F
            if (p.phase == kPhaseMeijering) p.V[v] = fv;
            if (fv > F(0) || fv != fv) red = max(red, B::of(fv));
            continue;
        }
        R f = np_max(p.first ? R(0) : M[v], vals);
        if (!p.last) {
            M[v] = f;
            continue;
        }
        if (p.filter == MIE_SK_HESSIAN && f <= R(0)) f = R(1);
        const int x = (int)(i % p.w), y = (int)(i / p.w % p.h), z = (int)(i / hw);
        dst.p[m * dst.sn + (int64_t)z * dst.sd + (int64_t)y * dst.sh + x] = (D)f;
    }
    if (p.phase == kPhaseFinal) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) red = max(red, __shfl_xor_sync(0xffffffffu, red, o));
    if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = red;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 1; k < 8; ++k) red = max(red, smax[k]);
        atomicMax(p.phase == kPhaseGamma ? &p.gmax[m] : &p.vmax[m], red);
    }
}

// Empty sigmas: zeros (hessian: ones, after its out[out <= 0] = 1).
template <typename D>
__global__ void sk_ridge_fill_kernel(RVol<D> dst, int64_t n, int d, int h, int w, D value) {
    const int64_t t = blockIdx.x * 256LL + threadIdx.x;
    const int64_t hw = (int64_t)h * w;
    if (t >= n * d * hw) return;
    const int64_t m = t / (hw * d);
    dst.p[m * dst.sn + t / hw % d * dst.sd + t / w % h * dst.sh + t % w] = value;
}

template <typename F>
__global__ void __launch_bounds__(256)
sk_hessian_eigvals_kernel(const F* __restrict__ h, F* __restrict__ eig, int nd, int64_t count, int64_t hs, int64_t es) {
    const int64_t v = blockIdx.x * 256LL + threadIdx.x;
    if (v >= count) return;
    const F* H[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) H[k] = h + k * hs;
    F e[3];
    if (nd == 2) {
        hessian_eig<F, 2>(H, v, e);
    } else {
        hessian_eig<F, 3>(H, v, e);
        eig[2 * es + v] = e[2];
    }
    eig[v] = e[0];
    eig[es + v] = e[1];
}

// ---------------------------------------------------------------- host side
struct RidgePlan {
    int64_t imgs;   // images per chunk
    int64_t cap;    // voxels per chunk buffer
};

static RidgePlan ridge_plan(int64_t n, int64_t vox) {
    RidgePlan p;
    p.imgs = std::max<int64_t>(1, std::min<int64_t>({n, kRidgeChunkVoxels / vox, kRidgeMaxChunkImages}));
    p.cap = p.imgs * vox;
    return p;
}

// Float buffers per chunk: the passes' two temporaries (one for planes), G_0 .. G_{nd-1}, and for the ridge filters
// the Hessian elements that cannot reuse a G buffer plus the running maximum.
static int ridge_buffers(int nd, bool filter) {
    if (nd == 3) return filter ? 9 : 5;
    return filter ? 5 : 3;
}

// Bytes of the running maximum's buffer: float64 for planes (RidgeMax), F for volumes.
static size_t ridge_max_bytes(const RidgePlan& p, int nd, size_t fsz) {
    return align256((size_t)p.cap * (nd == 2 ? sizeof(double) : fsz));
}

static size_t ridge_workspace_bytes(int64_t n, int d, int h, int w, int nd, int src_dtype, bool filter) {
    if (n <= 0 || d <= 0 || h <= 0 || w <= 0 || !valid_dtype(src_dtype)) return 0;
    const size_t fsz = src_dtype == MIE_F32 ? sizeof(float) : sizeof(double);
    const RidgePlan p = ridge_plan(n, (int64_t)d * h * w);
    const size_t bufs = (ridge_buffers(nd, filter) - (filter ? 1 : 0)) * align256((size_t)p.cap * fsz);
    return bufs + (filter ? ridge_max_bytes(p, nd, fsz) + 2 * align256((size_t)p.imgs * sizeof(double)) : 0);
}

template <typename T, typename F>
struct RidgeRun {
    int nd, d, h, w, mode, as_float, neg;
    double cval;
    cudaStream_t st;

    template <typename X>
    void pass(RVol<const X> in, RVol<F> out, int64_t nimg, int ax, const RidgeTaps& k, bool src) const {
        const unsigned blocks = (unsigned)((nimg * d * h * w + 255) / 256);
        const int af = src ? as_float : 0, ng = src ? neg : 0;
        if (ax == 0)
            sk_ridge_pass_kernel<X, F, 0><<<blocks, 256, 0, st>>>(in, out, nimg, d, h, w, k, mode, cval, af, ng);
        else if (ax == 1)
            sk_ridge_pass_kernel<X, F, 1><<<blocks, 256, 0, st>>>(in, out, nimg, d, h, w, k, mode, cval, af, ng);
        else
            sk_ridge_pass_kernel<X, F, 2><<<blocks, 256, 0, st>>>(in, out, nimg, d, h, w, k, mode, cval, af, ng);
    }

    // gaussian_filter of `in` with derivative order 1 along axis `da` (and order 0 along the others), in array axis
    // order; returns after writing `out`.  Axes of a plane are 1 (y) and 2 (x).
    template <typename X>
    void filter(RVol<const X> in, RVol<F> out, int64_t nimg, int da, const RidgeTaps* k, F* A, F* B, bool src) const {
        const int64_t vox = (int64_t)d * h * w;
        const RVol<F> a{A, vox, (int64_t)h * w, w}, b{B, vox, (int64_t)h * w, w};
        if (nd == 3) {
            pass<X>(in, a, nimg, 0, k[da == 0], src);
            pass<F>(RVol<const F>{a.p, a.sn, a.sd, a.sh}, b, nimg, 1, k[da == 1], false);
            pass<F>(RVol<const F>{b.p, b.sn, b.sd, b.sh}, out, nimg, 2, k[da == 2], false);
        } else {
            pass<X>(in, a, nimg, 1, k[da == 1], src);
            pass<F>(RVol<const F>{a.p, a.sn, a.sd, a.sh}, out, nimg, 2, k[da == 2], false);
        }
    }

    // The Hessian of images 0 .. nimg - 1 of `src`: H[k] in upstream's order.  For volumes, H_01 / H_02 share their z
    // pass (order 0) over G_0, H_11 / H_12 theirs over G_1, and G_1 / G_2 theirs over the image.  An H[k] may alias
    // G[a] when no later pass reads G[a] (the ridge filters put H_01, H_11, H_22 over G_0, G_1, G_2).
    void hessian(RVol<const T> src, int64_t nimg, const RidgeTaps* k, F* A, F* B, F* const* G, const RVol<F>* H) const {
        const int64_t vox = (int64_t)d * h * w;
        auto gv = [&](int a) { return RVol<F>{G[a], vox, (int64_t)h * w, w}; };
        auto cg = [&](int a) { return RVol<const F>{G[a], vox, (int64_t)h * w, w}; };
        if (nd == 2) {
            for (int a = 0; a < 2; ++a) filter<T>(src, gv(a), nimg, a + 1, k, A, B, true);
            filter<F>(cg(0), H[0], nimg, 1, k, A, B, false);
            filter<F>(cg(0), H[1], nimg, 2, k, A, B, false);
            filter<F>(cg(1), H[2], nimg, 2, k, A, B, false);
            return;
        }
        const RVol<F> a{A, vox, (int64_t)h * w, w}, b{B, vox, (int64_t)h * w, w};
        const RVol<const F> ac{A, vox, (int64_t)h * w, w}, bc{B, vox, (int64_t)h * w, w};
        // one z pass of order 0 over `in`, then y / x passes giving d/dy -> o1 and d/dx -> o2 (either may be null)
        auto fork = [&](auto in, bool src_in, const RVol<F>* o1, const RVol<F>* o2) {
            using X = typename std::remove_const<typename std::remove_pointer<decltype(in.p)>::type>::type;
            pass<X>(in, a, nimg, 0, k[0], src_in);
            if (o1) {
                pass<F>(ac, b, nimg, 1, k[1], false);
                pass<F>(bc, *o1, nimg, 2, k[0], false);
            }
            pass<F>(ac, b, nimg, 1, k[0], false);
            pass<F>(bc, *o2, nimg, 2, k[1], false);
        };
        filter<T>(src, gv(0), nimg, 0, k, A, B, true);
        const RVol<F> g1 = gv(1), g2 = gv(2);
        fork(src, true, &g1, &g2);
        filter<F>(cg(0), H[0], nimg, 0, k, A, B, false);
        fork(cg(0), false, &H[1], &H[2]);
        fork(cg(1), false, &H[3], &H[4]);
        fork(cg(2), false, nullptr, &H[5]);
    }
};

static bool taps_ok(const double* w, int r, bool anti) {
    for (int j = 0; j < r; ++j)
        if (!(w[j] == (anti ? -w[2 * r - j] : w[2 * r - j]))) return false;
    return true;
}

static int ridge_check_taps(int nscales, const double* sigmas, const int* radii, const double* taps0,
                            const double* taps1) {
    if (nscales < 0) return MIE_E_SHAPE;
    if (nscales > 0 && (!sigmas || !radii || !taps0 || !taps1)) return MIE_E_NULL;
    int64_t off = 0;
    for (int s = 0; s < nscales; ++s) {
        const int r = radii[s];
        if (r < 0 || r > MIE_SK_RIDGE_MAX_RADIUS) return MIE_E_KERNEL;
        if (!(sigmas[s] >= 0.0) || !std::isfinite(sigmas[s])) return MIE_E_RANGE;
        if (!taps_ok(taps0 + off, r, false) || !taps_ok(taps1 + off, r, true)) return MIE_E_KERNEL;
        off += 2 * r + 1;
    }
    return MIE_OK;
}

static void fill_taps(RidgeTaps* k, const double* t0, const double* t1, int r) {
    k[0].r = k[1].r = r;
    k[0].anti = 0;
    k[1].anti = 1;
    for (int i = 0; i <= 2 * r; ++i) {
        k[0].w[i] = t0[i];
        k[1].w[i] = t1[i];
    }
}

struct RidgeArgs {
    int filter, nscales, mode, black_ridges;
    const double *sigmas, *taps0, *taps1;
    const int* radii;
    double cval, alpha, beta, gamma;
};

template <typename T, typename F, typename D>
static void ridge_launch(const T* src, D* dst, int64_t n, int nd, int d, int h, int w, int64_t ssn, int64_t ssd,
                         int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, const RidgeArgs& a, uint8_t* ws,
                         cudaStream_t st) {
    const int64_t vox = (int64_t)d * h * w;
    const RidgePlan plan = ridge_plan(n, vox);
    const size_t bb = align256((size_t)plan.cap * sizeof(F));
    // planes: A G0 G1 H00 M (H01 over G0, H11 over G1); volumes: A B G0 G1 G2 H00 H02 H12 M; then the per-image maxima
    const int nf = ridge_buffers(nd, true) - 1;
    F* buf[8];
    for (int i = 0; i < nf; ++i) buf[i] = (F*)(ws + i * bb);
    void* M = ws + nf * bb;
    auto* gmax = (typename RBits<F>::type*)(ws + nf * bb + ridge_max_bytes(plan, nd, sizeof(F)));
    auto* vmax = (typename RBits<F>::type*)((uint8_t*)gmax + align256((size_t)plan.imgs * sizeof(double)));
    F *A = buf[0], *B = nd == 3 ? buf[1] : nullptr;
    F* G[3] = {buf[nd == 3 ? 2 : 1], buf[nd == 3 ? 3 : 2], nd == 3 ? buf[4] : nullptr};
    const int64_t hw = (int64_t)h * w;
    auto dense = [&](F* p) { return RVol<F>{p, vox, hw, w}; };
    RVol<F> H[6];
    if (nd == 2) {
        H[0] = dense(buf[3]); H[1] = dense(G[0]); H[2] = dense(G[1]);
    } else {
        H[0] = dense(buf[5]); H[1] = dense(G[0]); H[2] = dense(buf[6]);
        H[3] = dense(G[1]); H[4] = dense(buf[7]); H[5] = dense(G[2]);
    }
    const RidgeRun<T, F> run{nd, d, h, w, a.mode, 0, a.black_ridges ? 0 : 1, a.cval, st};
    RidgeTaps k[2];
    const bool implicit_gamma = a.gamma < 0.0 && (a.filter == MIE_SK_FRANGI || a.filter == MIE_SK_HESSIAN);
    for (int64_t m0 = 0; m0 < n; m0 += plan.imgs) {
        const int64_t nimg = std::min<int64_t>(plan.imgs, n - m0);
        const RVol<const T> s{src + m0 * ssn, ssn, ssd, ssh};
        const RVol<D> o{dst + m0 * dsn, dsn, dsd, dsh};
        const unsigned gx = (unsigned)std::min<int64_t>((vox + 255) / 256, std::max<int64_t>(1, 4096 / nimg));
        const dim3 grid(gx, (unsigned)nimg);
        int64_t off = 0;
        for (int sc = 0; sc < a.nscales; ++sc) {
            const int r = a.radii[sc];
            fill_taps(k, a.taps0 + off, a.taps1 + off, r);
            off += 2 * r + 1;
            run.hessian(s, nimg, k, A, B, G, H);
            RidgeEpi<F> p{};
            for (int i = 0; i < 6; ++i) p.H[i] = i < 3 * (nd - 1) ? H[i].p : nullptr;
            p.M = M; p.V = A; p.gmax = gmax; p.vmax = vmax;
            p.vox = vox; p.d = d; p.h = h; p.w = w;
            p.filter = a.filter; p.first = sc == 0; p.last = sc == a.nscales - 1;
            p.implicit_gamma = implicit_gamma;
            p.ca = 2.0 * a.alpha * a.alpha; p.cb = 2.0 * a.beta * a.beta;
            p.cg = implicit_gamma ? 1.0 : 2.0 * a.gamma * a.gamma;
            p.sig2 = a.sigmas[sc] * a.sigmas[sc];
            p.malpha = a.alpha;
            auto epi = [&](int phase) {
                p.phase = phase;
                if (nd == 2) sk_ridge_epilogue_kernel<F, D, 2><<<grid, 256, 0, st>>>(p, o);
                else sk_ridge_epilogue_kernel<F, D, 3><<<grid, 256, 0, st>>>(p, o);
            };
            if (implicit_gamma && sc == 0) {
                cudaMemsetAsync(gmax, 0, (size_t)nimg * sizeof(*gmax), st);
                epi(kPhaseGamma);
            }
            if (a.filter == MIE_SK_MEIJERING) {
                cudaMemsetAsync(vmax, 0, (size_t)nimg * sizeof(*vmax), st);
                epi(kPhaseMeijering);
            }
            epi(kPhaseFinal);
        }
    }
    if (a.nscales == 0) {
        const D value = a.filter == MIE_SK_HESSIAN ? D(1) : D(0);
        sk_ridge_fill_kernel<D><<<(unsigned)((n * vox + 255) / 256), 256, 0, st>>>(RVol<D>{dst, dsn, dsd, dsh}, n, d, h,
                                                                                   w, value);
    }
}

static int ridge_common_checks(int src_dtype, int dst_dtype, int mode, int64_t n, void* workspace,
                               size_t workspace_bytes, size_t need) {
    if (!valid_dtype(src_dtype)) return MIE_E_DTYPE;
    if (dst_dtype != MIE_F64 && dst_dtype != MIE_F32) return MIE_E_DTYPE;
    if (mode < MIE_BORDER_CONSTANT || mode > MIE_BORDER_SYMMETRIC) return MIE_E_BORDER;
    if (n == 0) return 1;
    if (!workspace) return MIE_E_NULL;
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < need) return MIE_E_WORKSPACE;
    return MIE_OK;
}

static int ridge_run(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int nd, int d, int h, int w,
                     int64_t ssn, int64_t ssd, int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, const RidgeArgs& a,
                     void* workspace, size_t workspace_bytes, void* stream) {
    if (a.filter < MIE_SK_FRANGI || a.filter > MIE_SK_MEIJERING) return MIE_E_UNSUPPORTED;
    int rc = ridge_check_taps(a.nscales, a.sigmas, a.radii, a.taps0, a.taps1);
    if (rc) return rc;
    rc = ridge_common_checks(src_dtype, dst_dtype, a.mode, n, workspace, workspace_bytes,
                             ridge_workspace_bytes(n, d, h, w, nd, src_dtype, true));
    if (rc) return rc > 0 ? MIE_OK : rc;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)workspace;
    MIE_DISPATCH_SRC(src_dtype, {
        using F = SkFloat<SrcT>;
        if (dst_dtype == MIE_F64)
            ridge_launch<SrcT, F, double>((const SrcT*)src, (double*)dst, n, nd, d, h, w, ssn, ssd, ssh, dsn, dsd, dsh,
                                          a, ws, st);
        else
            ridge_launch<SrcT, F, float>((const SrcT*)src, (float*)dst, n, nd, d, h, w, ssn, ssd, ssh, dsn, dsd, dsh, a,
                                         ws, st);
    });
    return check_launch();
}

static int hessian_run(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int nd, int d, int h,
                       int w, int64_t ssn, int64_t ssd, int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, int64_t dse,
                       int radius, const double* taps0, const double* taps1, int mode, double cval, void* workspace,
                       size_t workspace_bytes, void* stream) {
    if (!valid_dtype(src_dtype)) return MIE_E_DTYPE;
    if (dst_dtype != (src_dtype == MIE_F32 ? MIE_F32 : MIE_F64)) return MIE_E_DTYPE;
    const double sigma = 1.0;   // the taps carry sigma; only the checks of ridge_check_taps read it
    int rc = ridge_check_taps(1, &sigma, &radius, taps0, taps1);
    if (rc) return rc;
    const int64_t extent = n == 0 ? 0 : (n - 1) * dsn + (int64_t)(d - 1) * dsd + (int64_t)(h - 1) * dsh + w;
    if (n > 0 && dse < extent) return MIE_E_STRIDE;
    rc = ridge_common_checks(src_dtype, dst_dtype, mode, n, workspace, workspace_bytes,
                             ridge_workspace_bytes(n, d, h, w, nd, src_dtype, false));
    if (rc) return rc > 0 ? MIE_OK : rc;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)workspace;
    MIE_DISPATCH_SRC(src_dtype, {
        using F = SkFloat<SrcT>;
        const int64_t vox = (int64_t)d * h * w;
        const RidgePlan plan = ridge_plan(n, vox);
        const size_t bb = align256((size_t)plan.cap * sizeof(F));
        F* buf[5];
        for (int i = 0; i < ridge_buffers(nd, false); ++i) buf[i] = (F*)(ws + i * bb);
        F* A = buf[0];
        F* B = nd == 3 ? buf[1] : nullptr;
        F* G[3] = {buf[nd == 3 ? 2 : 1], buf[nd == 3 ? 3 : 2], nd == 3 ? buf[4] : nullptr};
        RidgeTaps k[2];
        fill_taps(k, taps0, taps1, radius);
        const RidgeRun<SrcT, F> run{nd, d, h, w, mode, 1, 0, cval, st};
        for (int64_t m0 = 0; m0 < n; m0 += plan.imgs) {
            const int64_t nimg = std::min<int64_t>(plan.imgs, n - m0);
            RVol<F> H[6];
            for (int e = 0; e < nd * (nd + 1) / 2; ++e) H[e] = RVol<F>{(F*)dst + e * dse + m0 * dsn, dsn, dsd, dsh};
            run.hessian(RVol<const SrcT>{(const SrcT*)src + m0 * ssn, ssn, ssd, ssh}, nimg, k, A, B, G, H);
        }
    });
    return check_launch();
}

}  // namespace mie

using namespace mie;

extern "C" {

size_t mie_sk_ridge_filter_workspace_bytes(int64_t n, int h, int w, int src_dtype) {
    return ridge_workspace_bytes(n, 1, h, w, 2, src_dtype, true);
}

size_t mie_sk_ridge_filter3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype) {
    return ridge_workspace_bytes(n, d, h, w, 3, src_dtype, true);
}

size_t mie_sk_hessian_matrix_workspace_bytes(int64_t n, int h, int w, int src_dtype) {
    return ridge_workspace_bytes(n, 1, h, w, 2, src_dtype, false);
}

size_t mie_sk_hessian_matrix3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype) {
    return ridge_workspace_bytes(n, d, h, w, 3, src_dtype, false);
}

int mie_sk_ridge_filter(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                        int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                        int filter, int nscales, const double* sigmas, const int* radii, const double* taps0,
                        const double* taps1, int mode, double cval, int black_ridges, double alpha, double beta,
                        double gamma, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h}, n,
                          h, w);
    if (rc) return rc;
    const RidgeArgs a{filter, nscales, mode, black_ridges, sigmas, taps0, taps1, radii, cval, alpha, beta, gamma};
    return ridge_run(src, dst, src_dtype, dst_dtype, n, 2, 1, h, w, src_stride_n, 0, src_stride_h, dst_stride_n, 0,
                     dst_stride_h, a, workspace, workspace_bytes, stream);
}

int mie_sk_ridge_filter3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                          int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h, int64_t dst_stride_n,
                          int64_t dst_stride_d, int64_t dst_stride_h, int filter, int nscales, const double* sigmas,
                          const int* radii, const double* taps0, const double* taps1, int mode, double cval,
                          int black_ridges, double alpha, double beta, double gamma, void* workspace,
                          size_t workspace_bytes, void* stream) {
    int rc = check_volumes({src, src_dtype, src_stride_n, src_stride_h}, src_stride_d,
                           {dst, dst_dtype, dst_stride_n, dst_stride_h}, dst_stride_d, n, d, h, w);
    if (rc) return rc;
    const RidgeArgs a{filter, nscales, mode, black_ridges, sigmas, taps0, taps1, radii, cval, alpha, beta, gamma};
    return ridge_run(src, dst, src_dtype, dst_dtype, n, 3, d, h, w, src_stride_n, src_stride_d, src_stride_h,
                     dst_stride_n, dst_stride_d, dst_stride_h, a, workspace, workspace_bytes, stream);
}

int mie_sk_hessian_matrix(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                          int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                          int64_t dst_stride_e, int radius, const double* taps0, const double* taps1, int mode,
                          double cval, void* workspace, size_t workspace_bytes, void* stream) {
    int rc = check_planes({src, src_dtype, src_stride_n, src_stride_h}, {dst, dst_dtype, dst_stride_n, dst_stride_h}, n,
                          h, w);
    if (rc) return rc;
    return hessian_run(src, dst, src_dtype, dst_dtype, n, 2, 1, h, w, src_stride_n, 0, src_stride_h, dst_stride_n, 0,
                       dst_stride_h, dst_stride_e, radius, taps0, taps1, mode, cval, workspace, workspace_bytes, stream);
}

int mie_sk_hessian_matrix3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                            int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h, int64_t dst_stride_n,
                            int64_t dst_stride_d, int64_t dst_stride_h, int64_t dst_stride_e, int radius,
                            const double* taps0, const double* taps1, int mode, double cval, void* workspace,
                            size_t workspace_bytes, void* stream) {
    int rc = check_volumes({src, src_dtype, src_stride_n, src_stride_h}, src_stride_d,
                           {dst, dst_dtype, dst_stride_n, dst_stride_h}, dst_stride_d, n, d, h, w);
    if (rc) return rc;
    return hessian_run(src, dst, src_dtype, dst_dtype, n, 3, d, h, w, src_stride_n, src_stride_d, src_stride_h,
                       dst_stride_n, dst_stride_d, dst_stride_h, dst_stride_e, radius, taps0, taps1, mode, cval,
                       workspace, workspace_bytes, stream);
}

int mie_sk_hessian_eigvals(const void* h, void* eig, int dtype, int ndim, int64_t count, int64_t h_stride_e,
                           int64_t eig_stride_e, void* stream) {
    if (dtype != MIE_F32 && dtype != MIE_F64) return MIE_E_DTYPE;
    if ((ndim != 2 && ndim != 3) || count < 0) return MIE_E_SHAPE;
    if (count == 0) return MIE_OK;
    if (!h || !eig) return MIE_E_NULL;
    if (h_stride_e < count || eig_stride_e < count) return MIE_E_STRIDE;
    const unsigned blocks = (unsigned)((count + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == MIE_F64)
        sk_hessian_eigvals_kernel<double><<<blocks, 256, 0, st>>>((const double*)h, (double*)eig, ndim, count,
                                                                   h_stride_e, eig_stride_e);
    else
        sk_hessian_eigvals_kernel<float><<<blocks, 256, 0, st>>>((const float*)h, (float*)eig, ndim, count, h_stride_e,
                                                                 eig_stride_e);
    return check_launch();
}

}  // extern "C"
