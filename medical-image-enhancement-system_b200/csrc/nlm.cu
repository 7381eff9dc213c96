// nlm.cu — non-local means denoising, skimage.restoration.denoise_nl_means(fast_mode=True) semantics
// (scikit-image 0.26.0, reference pyproject.toml:12 / uv.lock:619-650; SURVEY.md §8(a) A8, BASELINE.json
// config 5's "else" branch: 7x7 patches on 256x256 slices).  The upstream source is not on disk; the
// algorithm below restates its published fast mode (Darbon et al., ISBI 2008, integral images) [RECALLED]:
//
//   s = patch_size (+1 if even), o = s / 2, d = patch_distance, I = image reflect-padded by o + d + 1
//   out(p) = sum_t c_t w_t(p) I(p + t) / sum_t c_t w_t(p),      t in [-d, d]^2,  c_0 = 2, c_t = 1 otherwise
//   w_t(p) = exp(-dist) if dist <= 5 else 0,   dist = max(D, 0) / (h^2 s^2)
//   D      = sum_{q in (-o, o]^2} ((I(p + q) - I(p + q + t))^2 - 2 sigma^2)
// (the box of the upstream integral-image difference spans rows/columns p - o + 1 .. p + o, i.e.
// (s - 1)^2 pixels, and the centre pixel is accumulated twice — both quirks are kept).
//
// This op is compute bound outright (SURVEY.md §8(d)): (2d+1)^2 = 529 shifts per pixel.  One block owns
// a 32x32 output tile with its (32 + 2(o + d))^2 neighbourhood in shared memory; per shift it forms the
// squared differences once, sums them separably (horizontal sliding sums into shared memory, vertical
// sums in registers) and accumulates the weighted shifted pixel — ~35 instructions per pixel and shift
// instead of ~110 for the direct 36-term patch distance.  exp() is ex2.approx (MUFU): the result is
// within the north star's fp32 tolerance (rel 1e-5) of the float64 oracle, not bit-exact.

#include <cmath>

#include "mie_common.cuh"

namespace mie {

constexpr int kNlmTile = 32;
constexpr int kNlmMaxO = 4;    // patch size <= 9
constexpr int kNlmMaxD = 16;   // patch distance <= 16

struct NlmArgs {
    int h, w, tiles_x, tiles_y;
    int o, d;
    float inv_h2s2;   // 1 / (h^2 s^2)
    float var_term;   // (s-1)^2 * 2 sigma^2
    float lo, rg;
};

template <typename SrcT, typename DstT, int O>
__global__ void __launch_bounds__(256)
nlm_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
           NlmArgs a) {
    extern __shared__ __align__(16) float smem[];
    constexpr int T = kNlmTile;
    constexpr int o = O;
    const int d = a.d, R = o + d;
    const int E = T + 2 * R, pitch = E | 1;      // neighbourhood edge, odd pitch
    const int HR = T + 2 * o - 1;                // rows of horizontal sums: tile rows -o+1 .. T-1+o
    float* S = smem;                             // E x pitch
    float* H = smem + E * pitch;                 // HR x (T + 1)
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * T, ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * T;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const SrcT* plane = src + n * ssn;
    for (int i = threadIdx.x; i < E * E; i += 256) {
        const int r = i / E, c = i - r * E;
        const int sy = border_index(ty0 - R + r, a.h, MIE_BORDER_REFLECT);
        const int sx = border_index(tx0 - R + c, a.w, MIE_BORDER_REFLECT);
        S[r * pitch + c] = Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], a.lo, a.rg);
    }
    __syncthreads();

    // stage-2 ownership: column lx, rows ly0 + 8k (k = 0..3)
    const int lx = threadIdx.x & 31, ly0 = threadIdx.x >> 5;
    float num[4] = {0.f, 0.f, 0.f, 0.f}, den[4] = {0.f, 0.f, 0.f, 0.f};
    // stage-1 ownership: (row hy of H, 8-column segment hs); HR * 4 items over 256 threads
    constexpr int box = 2 * O;                   // pixels per box side
    const float neg_log2e = -1.4426950408889634f;

    for (int ty = -d; ty <= d; ++ty) {
        for (int tx = -d; tx <= d; ++tx) {
            // ---- horizontal sums of squared differences
            for (int it = threadIdx.x; it < HR * 4; it += 256) {
                const int hy = it >> 2, hs = it & 3;
                const float* p = S + (hy + 1 + d) * pitch + (8 * hs + 1 + d);   // tile row hy - o + 1, column 8hs - o + 1
                const float* q = p + ty * pitch + tx;
                float d2[8 + box - 1];
#pragma unroll
                for (int k = 0; k < 8 + box - 1; ++k) {
                    const float df = p[k] - q[k];
                    d2[k] = df * df;
                }
                float* hrow = H + hy * (T + 1) + 8 * hs;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float sacc = d2[j];
#pragma unroll
                    for (int k = 1; k < box; ++k) sacc += d2[j + k];
                    hrow[j] = sacc;
                }
            }
            __syncthreads();
            // ---- vertical sums, weights, accumulation
            const float cmul = (ty == 0 && tx == 0) ? 2.0f : 1.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int oy = ly0 + 8 * k;
                float D = H[oy * (T + 1) + lx];
#pragma unroll
                for (int j = 1; j < box; ++j) D += H[(oy + j) * (T + 1) + lx];
                const float dist = fmaxf(D - a.var_term, 0.0f) * a.inv_h2s2;
                if (dist <= 5.0f) {
                    const float wgt = cmul * exp2f(dist * neg_log2e);
                    num[k] = fmaf(wgt, S[(oy + R + ty) * pitch + lx + R + tx], num[k]);
                    den[k] += wgt;
                }
            }
            __syncthreads();
        }
    }
    const int x = tx0 + lx;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int y = ty0 + ly0 + 8 * k;
        if (y < a.h && x < a.w) dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(num[k] / den[k], a.lo, a.rg);
    }
}

// ---------------------------------------------------------------- marching variant (no barriers per shift)
// The tile kernel above synchronises the block twice per shift (1 058 barriers per tile for d = 11) and keeps
// only 148 of its 256 threads busy while the horizontal sums are formed: ~59 issue slots per pixel and shift.
// Here a warp works alone on a band of BH output rows x VL = 33 - 2o output columns: lane l owns the column
// of squared differences c = x0 - o + 1 + l, the horizontal box sum over columns c .. c + 2o - 1 is three
// shuffle-adds (s2 = d + d[+1]; s4 = s2 + s2[+2]; s6 = s4 + s2[+4] for o = 3), the vertical box sum is the sum
// of a register ring of the last 2o row sums, and the BH accumulator pairs (num, den) of the lane's output
// column stay in registers across all (2d+1)^2 shifts.  After the neighbourhood is staged in shared memory
// (read-only from then on) there is not a single barrier; ~23 instructions per lane and row step, 84 % of the
// lanes and BH / (BH + 2o - 1) of the row steps produce an output.
// Box sum over lanes l - O + 1 .. l + O, landing on lane l itself (valid for lanes O - 1 .. 31 - O): the lane
// that owns a column of squared differences also owns the output of that column, so the shifted centre pixel
// I(p + t) it needs is the q value it loaded O row steps earlier — a register, not another shared-memory load.
template <int O>
__device__ __forceinline__ float nlm_hsum(float d2) {
    if (O == 1) return d2 + __shfl_down_sync(0xffffffffu, d2, 1);                        // l, l+1
    if (O == 2) {
        const float t = d2 + __shfl_up_sync(0xffffffffu, d2, 1);                          // l-1, l
        return t + __shfl_down_sync(0xffffffffu, t, 2);                                   // l-1 .. l+2
    }
    const float s2 = d2 + __shfl_down_sync(0xffffffffu, d2, 1);                           // l, l+1
    if (O == 3) return s2 + __shfl_up_sync(0xffffffffu, s2, 2) + __shfl_down_sync(0xffffffffu, s2, 2);   // l-2 .. l+3
    const float s4 = s2 + __shfl_down_sync(0xffffffffu, s2, 2);                           // l .. l+3
    return __shfl_up_sync(0xffffffffu, s4, 3) + __shfl_down_sync(0xffffffffu, s4, 1);     // l-3 .. l, l+1 .. l+4
}
__device__ __forceinline__ float nlm_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

template <int O> struct NlmMarch {
    static constexpr int box = 2 * O, VL = 33 - box, BH = 32, TWB = 2 * VL, THB = 4 * BH;
    static constexpr int RMAX = O + kNlmMaxD, PITCH = (TWB + 2 * RMAX) | 1;
};

template <typename SrcT, typename DstT, int O>
__global__ void __launch_bounds__(256, 2)
nlm_march_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                 int64_t dsh, NlmArgs a) {
    using G = NlmMarch<O>;
    constexpr int box = G::box, VL = G::VL, BH = G::BH, PITCH = G::PITCH;
    extern __shared__ __align__(16) float S[];
    const int d = a.d, R = O + d;
    const int EW = G::TWB + 2 * R, EH = G::THB + 2 * R;
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * G::TWB, ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * G::THB;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const SrcT* plane = src + n * ssn;
    for (int i = threadIdx.x; i < EH * EW; i += 256) {
        const int r = i / EW, c = i - r * EW;
        const int sy = border_index(ty0 - R + r, a.h, MIE_BORDER_REFLECT);
        const int sx = border_index(tx0 - R + c, a.w, MIE_BORDER_REFLECT);
        S[r * PITCH + c] = Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], a.lo, a.rg);
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = (warp & 1) * VL, y0 = (warp >> 1) * BH;                 // the warp's outputs, tile coordinates
    // lane l owns tile column x0 - (O - 1) + l: differences AND output (valid outputs: lanes O-1 .. O-2+VL)
    const float* pbase = S + (R + y0 - O + 1) * PITCH + (R + x0 - O + 1 + lane);   // difference row 0, own column
    const float* cbase = pbase + (O - 1) * PITCH;                                  // output row 0, own column
    const float k2 = -1.4426950408889634f * a.inv_h2s2;                    // weight = 2^(k2 * max(D - var, 0))
    const float cut = -5.0f * 1.4426950408889634f;                         // distance 5 on that scale
    float num[BH], den[BH];
#pragma unroll
    for (int j = 0; j < BH; ++j) {                                         // zero shift: D = 0, weight 2 (upstream quirk)
        const float c = cbase[j * PITCH];
        num[j] = c + c; den[j] = 2.0f;
    }
    for (int ty = -d; ty <= d; ++ty) {
        for (int tx = -d; tx <= d; ++tx) {
            if (ty == 0 && tx == 0) continue;
            const int toff = ty * PITCH + tx;
            const float* q = pbase + toff;
            float hs[box], qr[O + 1];           // rings: row sums of the last 2O rows, q of the last O + 1 rows
#pragma unroll
            for (int s = 0; s < BH + box - 1; ++s) {
                const float qv = q[s * PITCH];
                qr[s % (O + 1)] = qv;
                const float df = pbase[s * PITCH] - qv;
                hs[s % box] = nlm_hsum<O>(df * df);
                if (s >= box - 1) {
                    const int j = s - (box - 1);              // output row j: centre = difference row j + O - 1 = s - O
                    float V = hs[0];
#pragma unroll
                    for (int k = 1; k < box; ++k) V += hs[k];
                    const float e = fmaxf(V - a.var_term, 0.0f) * k2;
                    const float wgt = e >= cut ? nlm_ex2(e) : 0.0f;     // branch-free: select, not a divergent region
                    num[j] = fmaf(wgt, qr[(s - O) % (O + 1)], num[j]);
                    den[j] += wgt;
                }
            }
        }
    }
    const int x = tx0 + x0 - (O - 1) + lane;
    if (lane >= O - 1 && lane < O - 1 + VL && x < a.w) {
#pragma unroll
        for (int j = 0; j < BH; ++j) {
            const int y = ty0 + y0 + j;
            if (y < a.h) dst[n * dsn + (int64_t)y * dsh + x] = Px<DstT>::from01(num[j] / den[j], a.lo, a.rg);
        }
    }
}

int nlm_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
             int64_t dsn, int64_t dsh, int patch_size, int patch_distance, float hpar, float sigma, float lo, float hi,
             cudaStream_t st) {
    int rc = check_planes({src, sd, ssn, ssh}, {dst, dd, dsn, dsh}, n, h, w);
    if (rc) return rc;
    rc = check_dtypes(sd, dd, lo, hi);
    if (rc) return rc;
    if (patch_size <= 0 || patch_distance < 0) return MIE_E_KERNEL;
    const int s = patch_size + (patch_size % 2 == 0 ? 1 : 0);
    const int o = s / 2;
    if (o < 1 || o > kNlmMaxO || patch_distance > kNlmMaxD) return MIE_E_KERNEL;
    if (!(hpar > 0.0f) || sigma < 0.0f) return MIE_E_RANGE;
    // numpy 'reflect' padding by o + d + 1 must be a single reflection
    if (o + patch_distance + 1 >= h || o + patch_distance + 1 >= w) return MIE_E_BORDER;
    if (n == 0) return MIE_OK;
    NlmArgs a;
    a.h = h; a.w = w; a.tiles_x = ceil_div(w, kNlmTile); a.tiles_y = ceil_div(h, kNlmTile);
    a.o = o; a.d = patch_distance;
    a.inv_h2s2 = (float)(1.0 / ((double)hpar * hpar * s * s));
    a.var_term = (float)((double)(2 * o) * (2 * o) * 2.0 * (double)sigma * sigma);
    a.lo = lo; a.rg = hi - lo;
    const bool no_march = kernel_policy(MIE_POLICY_GENERIC_NLM);
    if (!no_march) {
#define MIE_NLM_MARCH(O_)                                                                                      \
    {                                                                                                          \
        using G = NlmMarch<O_>;                                                                                \
        a.tiles_x = ceil_div(w, G::TWB); a.tiles_y = ceil_div(h, G::THB);                                      \
        const int64_t mblocks = n * a.tiles_x * a.tiles_y;                                                     \
        if (mblocks > 2147483647LL) return MIE_E_SHAPE;                                                        \
        const size_t msmem = (size_t)(G::THB + 2 * (O_ + patch_distance)) * G::PITCH * 4;                      \
        MIE_ENSURE_SMEM((nlm_march_kernel<SrcT, DstT, O_>), (G::THB + 2 * G::RMAX) * G::PITCH * 4);            \
        nlm_march_kernel<SrcT, DstT, O_><<<(unsigned)mblocks, 256, msmem, st>>>((const SrcT*)src, (DstT*)dst, ssn, ssh, \
                                                                              dsn, dsh, a);                    \
    }
        switch (o) {
            case 1: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_MARCH(1)); break;
            case 2: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_MARCH(2)); break;
            case 3: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_MARCH(3)); break;
            default: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_MARCH(4)); break;
        }
#undef MIE_NLM_MARCH
        return check_launch();
    }
    const int64_t blocks = n * a.tiles_x * a.tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    const int E = kNlmTile + 2 * (o + patch_distance);
    const size_t smem = (size_t)(E * (E | 1) + (kNlmTile + 2 * o - 1) * (kNlmTile + 1)) * 4;
#define MIE_NLM_LAUNCH(O_)                                                                               \
    MIE_ENSURE_SMEM((nlm_kernel<SrcT, DstT, O_>), 64 * 1024);                                            \
    nlm_kernel<SrcT, DstT, O_><<<(unsigned)blocks, 256, smem, st>>>((const SrcT*)src, (DstT*)dst, ssn, ssh, dsn, dsh, a)
    switch (o) {
        case 1: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_LAUNCH(1)); break;
        case 2: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_LAUNCH(2)); break;
        case 3: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_LAUNCH(3)); break;
        default: MIE_DISPATCH_SRC_DST(sd, dd, MIE_NLM_LAUNCH(4)); break;
    }
#undef MIE_NLM_LAUNCH
    return check_launch();
}


// ================================================================ slow mode (fast_mode=False)
// skimage's _nl_means_denoising_2d / patch_distance_2d [RECALLED; SURVEY.md Appendix B4, oracle/mie_oracle.c
// orc_nlm_slow]: Gaussian patch weights, the image reflect-padded by the patch radius only, the search window
// clipped at the image, and the running distance tested against the cut-off 5 before every patch ROW — which is why
// this mode cannot use the separable sliding sums above: the test makes the result depend on the order of the sum.
// The arithmetic is float64 in upstream's order (B200 runs DFMA at half the FFMA rate), so the kernel agrees with the
// float64 oracle to the last bits of exp(); one thread per pixel, the block's neighbourhood as doubles in shared memory.
constexpr int kNlmSlowTile = 16;
constexpr int kNlmSlowMaxS = 15;   // patch size <= 15: the weights travel as a kernel parameter
constexpr int kNlmSlowMaxD = 32;

struct NlmSlowArgs {
    int h, w, tiles_x, tiles_y;
    int s, d;
    double var2;    // 2 sigma^2
    float lo, rg;
    double wgt[kNlmSlowMaxS * kNlmSlowMaxS];   // w[i][j] / (sum(w) h^2), row-major s x s
};

template <typename DstT> struct SlowOut {
    static __device__ __forceinline__ DstT put(double y, float lo, float rg) { return Px<DstT>::from01((float)y, lo, rg); }
};
template <> struct SlowOut<double> {
    static __device__ __forceinline__ double put(double y, float, float) { return y; }
};

template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256)
nlm_slow_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                const __grid_constant__ NlmSlowArgs a) {
    extern __shared__ __align__(16) double dsm[];
    constexpr int T = kNlmSlowTile;
    const int s = a.s, o = s / 2, d = a.d, R = o + d;
    const int E = T + 2 * R, pitch = E | 1;
    double* S = dsm;                 // E x pitch
    double* W = dsm + E * pitch;     // s x s
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * T, ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * T;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const SrcT* plane = src + n * ssn;
    for (int i = threadIdx.x; i < E * E; i += 256) {
        const int r = i / E, c = i - r * E;
        const int sy = border_index(ty0 - R + r, a.h, MIE_BORDER_REFLECT);
        const int sx = border_index(tx0 - R + c, a.w, MIE_BORDER_REFLECT);
        S[r * pitch + c] = (double)Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], a.lo, a.rg);
    }
    for (int i = threadIdx.x; i < s * s; i += 256) W[i] = a.wgt[i];
    __syncthreads();
    const int lx = threadIdx.x & (T - 1), ly = threadIdx.x / T;
    const int col = tx0 + lx, row = ty0 + ly;
    if (col >= a.w || row >= a.h) return;
    const int i0 = row - min(d, row), i1 = row + min(d + 1, a.h - row);
    const int j0 = col - min(d, col), j1 = col + min(d + 1, a.w - col);
    // top-left corner of the central patch in tile coordinates
    const double* P1 = S + (ly + R - o) * pitch + (lx + R - o);
    double num = 0.0, den = 0.0;
    for (int ci = i0; ci < i1; ++ci) {
        for (int cj = j0; cj < j1; ++cj) {
            const double* P2 = S + (ci - ty0 + R - o) * pitch + (cj - tx0 + R - o);
            double dist = 0.0;
            bool cut = false;
            for (int pi = 0; pi < s; ++pi) {
                if (dist > 5.0) { cut = true; break; }
                const double* r1 = P1 + pi * pitch;
                const double* r2 = P2 + pi * pitch;
                const double* wr = W + pi * s;
                for (int pj = 0; pj < s; ++pj) {
                    const double df = __dsub_rn(r1[pj], r2[pj]);
                    dist = __dadd_rn(dist, __dmul_rn(wr[pj], __dsub_rn(__dmul_rn(df, df), a.var2)));
                }
            }
            if (!cut) {
                const double weight = exp(-fmax(0.0, dist));
                den = __dadd_rn(den, weight);
                num = __dadd_rn(num, __dmul_rn(weight, P2[o * pitch + o]));
            }
        }
    }
    dst[n * dsn + (int64_t)row * dsh + col] = SlowOut<DstT>::put(num / den, a.lo, a.rg);
}

static int nlm_slow_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
                         int64_t dsn, int64_t dsh, int patch_size, int patch_distance, double hpar, double sigma, float lo,
                         float hi, cudaStream_t st) {
    int rc = check_planes({src, sd, ssn, ssh}, {dst, dd, dsn, dsh}, n, h, w);
    if (rc) return rc;
    if (!valid_dtype(sd) || !(dd == sd || dd == MIE_F32 || dd == MIE_F64)) return MIE_E_DTYPE;
    if (sd != MIE_F32 && !(hi > lo)) return MIE_E_RANGE;
    if (patch_size <= 0 || patch_distance < 0) return MIE_E_KERNEL;
    const int s = patch_size + (patch_size % 2 == 0 ? 1 : 0);
    const int o = s / 2;
    if (o < 1 || s > kNlmSlowMaxS || patch_distance > kNlmSlowMaxD) return MIE_E_KERNEL;
    if (!(hpar > 0.0) || sigma < 0.0) return MIE_E_RANGE;
    if (o >= h || o >= w) return MIE_E_BORDER;   // np.pad(mode='reflect') by o needs o < size
    if (n == 0) return MIE_OK;
    NlmSlowArgs a;
    a.h = h; a.w = w; a.tiles_x = ceil_div(w, kNlmSlowTile); a.tiles_y = ceil_div(h, kNlmSlowTile);
    a.s = s; a.d = patch_distance; a.var2 = 2.0 * sigma * sigma; a.lo = lo; a.rg = hi - lo;
    {   // the patch weights exactly as upstream forms them (and as orc_nlm_patch_weights does): host libm, float64
        const double A = ((double)s - 1.0) / 4.0;
        double sum = 0.0;
        for (int i = 0; i < s; ++i)
            for (int j = 0; j < s; ++j) {
                const double di = (double)(i - o), dj = (double)(j - o);
                a.wgt[i * s + j] = std::exp(-(di * di + dj * dj) / (2.0 * A * A));
                sum += a.wgt[i * s + j];
            }
        const double scale = 1.0 / (sum * hpar * hpar);
        for (int i = 0; i < s * s; ++i) a.wgt[i] *= scale;
    }
    const int64_t blocks = n * a.tiles_x * a.tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    const int E = kNlmSlowTile + 2 * (o + patch_distance);
    const size_t smem = (size_t)(E * (E | 1) + s * s) * 8;
    constexpr int kMaxE = kNlmSlowTile + 2 * (kNlmSlowMaxS / 2 + kNlmSlowMaxD);
    constexpr size_t kMaxSmem = (size_t)(kMaxE * (kMaxE | 1) + kNlmSlowMaxS * kNlmSlowMaxS) * 8;
#define MIE_NLM_SLOW(D_)                                                                                               \
    MIE_ENSURE_SMEM((nlm_slow_kernel<SrcT, D_>), kMaxSmem);                                                            \
    nlm_slow_kernel<SrcT, D_><<<(unsigned)blocks, 256, smem, st>>>((const SrcT*)src, (D_*)dst, ssn, ssh, dsn, dsh, a)
    if (dd == MIE_F64) { MIE_DISPATCH_SRC(sd, MIE_NLM_SLOW(double)); }
    else if (dd == MIE_F32) { MIE_DISPATCH_SRC(sd, MIE_NLM_SLOW(float)); }
    else { MIE_DISPATCH_SRC(sd, MIE_NLM_SLOW(SrcT)); }
#undef MIE_NLM_SLOW
    return check_launch();
}

}  // namespace mie

using namespace mie;

extern "C" int mie_nlm(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                       int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                       int patch_size, int patch_distance, float h_param, float sigma, float lo, float hi,
                       void* stream) {
    return nlm_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n, dst_stride_h,
                    patch_size, patch_distance, h_param, sigma, lo, hi, (cudaStream_t)stream);
}

extern "C" int mie_nlm_slow(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                            int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                            int patch_size, int patch_distance, double h_param, double sigma, float lo, float hi,
                            void* stream) {
    return nlm_slow_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n, dst_stride_h,
                         patch_size, patch_distance, h_param, sigma, lo, hi, (cudaStream_t)stream);
}
