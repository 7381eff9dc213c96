// clahe.cu — standalone CLAHE: per-tile histogram -> clip/redistribute -> LUT kernel
// and the bilinear LUT-interpolation kernel.  Replaces
// kornia.enhance.equalize_clahe (SURVEY.md §8(a) A1) and cv::CLAHE on uint8
// (§8(a) A1').  One block per CLAHE tile builds the histogram in shared memory
// (per-warp sub-histograms, warp-uniform fast path for constant regions such as
// CT air), then clips, redistributes and scans in-block.
#include "clahe.cuh"
#include "window.cuh"

namespace mie {

// clahe_fast.cu
int clahe_lut_fast_mode(const ClaheGeom& g, const Image& s, float lo, float hi, WinCvt* cv);
int launch_clahe_lut_fast(const Image& s, int64_t n, const ClaheGeom& g, const LutParams& lp, uint32_t* hist,
                          uint8_t* luts, int mode, const WinCvt& cv, cudaStream_t st);
size_t clahe_cells_bytes(int64_t n, int gh, int gw);
int clahe_apply_fast_mode(const ClaheGeom& g, const Image& s, const Image& d, float lo, float hi, WinCvt* cv);
int launch_clahe_apply_fast(const Image& s, const Image& d, int64_t n, const ClaheGeom& g, const uint8_t* luts,
                            void* cells, int mode, const WinCvt& cv, cudaStream_t st);

// ---------------------------------------------------------------- LUT kernel
template <typename SrcT, int SEM>
__global__ void __launch_bounds__(256)
clahe_lut_kernel(const SrcT* __restrict__ src, int64_t ssn, int64_t ssh, ClaheGeom g, float lo, float rg,
                 LutParams lp, uint32_t* __restrict__ hist_out, uint8_t* __restrict__ lut_out) {
    __shared__ int s_hist[8][kBins];
    __shared__ int s_red[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int i = 0; i < 8; ++i) s_hist[i][tid] = 0;
    __syncthreads();

    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % g.gw);
    const int ty = (int)((tile / g.gw) % g.gh);
    const int64_t n = tile / ((int64_t)g.gw * g.gh);
    const SrcT* plane = src + n * ssn;

    for (int yy = warp; yy < g.th; yy += 8) {
        const int sy = border_index(ty * g.th + yy, g.h, MIE_BORDER_REFLECT);
        const SrcT* row = plane + (int64_t)sy * ssh;
        for (int x0 = 0; x0 < g.tw; x0 += 32) {
            const int xx = x0 + lane;
            int bin = -1;
            if (xx < g.tw) {
                const int sx = border_index(tx * g.tw + xx, g.w, MIE_BORDER_REFLECT);
                SrcT raw = row[sx];
                if (SEM == MIE_CLAHE_KORNIA) bin = kornia_bin(Px<SrcT>::to01(raw, lo, rg));
                else bin = (int)raw;  // uint8 only (checked on the host)
            }
            // Warp-aggregated update: a warp whose valid lanes all hit one bin
            // (constant background) issues a single add.
            const unsigned act = __ballot_sync(0xffffffffu, bin >= 0);
            if (act == 0) continue;
            const int leader = __ffs(act) - 1;
            const int b0 = __shfl_sync(0xffffffffu, bin, leader);
            if (__all_sync(0xffffffffu, bin < 0 || bin == b0)) {
                if (lane == leader) s_hist[warp][b0] += __popc(act);
            } else if (bin >= 0) {
                atomicAdd(&s_hist[warp][bin], 1);
            }
            __syncwarp();
        }
    }
    __syncthreads();
    int hv = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) hv += s_hist[i][tid];
    if (hist_out) hist_out[tile * kBins + tid] = (uint32_t)hv;
    if (lut_out) lut_out[tile * kBins + tid] = lut_entry_from_count<SEM>(hv, lp, s_red);
}

// ---------------------------------------------------------------- apply kernel
// One thread per 4 horizontally adjacent pixels.
template <typename SrcT, typename DstT, int SEM>
__global__ void __launch_bounds__(256)
clahe_apply_kernel(const SrcT* __restrict__ src, DstT* __restrict__ dst, int64_t ssn, int64_t ssh, int64_t dsn,
                   int64_t dsh, ClaheGeom g, float lo, float rg, const uint8_t* __restrict__ luts) {
    const int x0 = (blockIdx.x * 64 + (threadIdx.x & 63)) * 4;
    const int y = blockIdx.y * 4 + (threadIdx.x >> 6);
    const int64_t n = blockIdx.z;
    if (y >= g.h || x0 >= g.w) return;
    const SrcT* srow = src + n * ssn + (int64_t)y * ssh;
    DstT* drow = dst + n * dsn + (int64_t)y * dsh;
    const uint8_t* nl = luts + n * (int64_t)g.gh * g.gw * kBins;

    int j0, j1;
    float wy = 0.f, ya = 0.f, ya1 = 0.f;
    if (SEM == MIE_CLAHE_KORNIA) kornia_axis(y, g.th, g.gh, j0, j1, wy);
    else opencv_axis(y, __fdiv_rn(1.0f, (float)g.th), g.gh, j0, j1, ya, ya1);
    const uint8_t* r0 = nl + (int64_t)j0 * g.gw * kBins;
    const uint8_t* r1 = nl + (int64_t)j1 * g.gw * kBins;
    const float inv_tw = __fdiv_rn(1.0f, (float)g.tw);

#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int x = x0 + k;
        if (x >= g.w) break;
        const SrcT raw = srow[x];
        int i0, i1;
        if (SEM == MIE_CLAHE_KORNIA) {
            float wx;
            kornia_axis(x, g.tw, g.gw, i0, i1, wx);
            const int idx = kornia_idx(Px<SrcT>::to01(raw, lo, rg));
            const float tl = (float)__ldg(r0 + i0 * kBins + idx), tr = (float)__ldg(r0 + i1 * kBins + idx);
            const float bl = (float)__ldg(r1 + i0 * kBins + idx), br = (float)__ldg(r1 + i1 * kBins + idx);
            const float o = __fdiv_rn(kornia_blend(tl, tr, bl, br, wx, wy), 255.0f);
            drow[x] = Px<DstT>::from01(o, lo, rg);
        } else {
            float xa, xa1;
            opencv_axis(x, inv_tw, g.gw, i0, i1, xa, xa1);
            const int idx = (int)raw;
            const float l11 = (float)__ldg(r0 + i0 * kBins + idx), l12 = (float)__ldg(r0 + i1 * kBins + idx);
            const float l21 = (float)__ldg(r1 + i0 * kBins + idx), l22 = (float)__ldg(r1 + i1 * kBins + idx);
            float res = rintf(opencv_blend(l11, l12, l21, l22, xa, xa1, ya, ya1));
            res = fminf(fmaxf(res, 0.0f), 255.0f);
            drow[x] = (DstT)res;
        }
    }
}

// ---------------------------------------------------------------- host side
static int clahe_common_checks(const Image& s, int64_t n, int h, int w, int gh, int gw, int semantics, float lo, float hi,
                               ClaheGeom* g) {
    const int sd = s.dtype;
    if (n < 0 || h <= 0 || w <= 0) return MIE_E_SHAPE;
    if (n > 0 && !s.p) return MIE_E_NULL;
    if (!valid_dtype(sd)) return MIE_E_DTYPE;
    if (!plane_strides_ok(s, n, h, w)) return MIE_E_STRIDE;
    if (semantics != MIE_CLAHE_KORNIA && semantics != MIE_CLAHE_OPENCV) return MIE_E_UNSUPPORTED;
    if (semantics == MIE_CLAHE_OPENCV && sd != MIE_U8) return MIE_E_UNSUPPORTED;  // uint16: mie_clahe / mie_clahe16_luts
    if (semantics == MIE_CLAHE_KORNIA && sd != MIE_F32 && !(hi > lo)) return MIE_E_RANGE;
    return make_clahe_geom(h, w, gh, gw, semantics, g);
}

template <typename SrcT>
static int launch_lut(const void* src, int64_t n, int64_t ssn, int64_t ssh, const ClaheGeom& g, float lo, float rg,
                      const LutParams& lp, int semantics, uint32_t* hist, uint8_t* luts, cudaStream_t st) {
    const int64_t tiles = n * g.gh * g.gw;
    if (tiles == 0) return MIE_OK;
    if (tiles > 2147483647LL) return MIE_E_SHAPE;
    if (semantics == MIE_CLAHE_KORNIA)
        clahe_lut_kernel<SrcT, MIE_CLAHE_KORNIA><<<(unsigned)tiles, 256, 0, st>>>((const SrcT*)src, ssn, ssh, g, lo, rg,
                                                                               lp, hist, luts);
    else
        clahe_lut_kernel<SrcT, MIE_CLAHE_OPENCV><<<(unsigned)tiles, 256, 0, st>>>((const SrcT*)src, ssn, ssh, g, lo, rg,
                                                                               lp, hist, luts);
    return check_launch();
}

int clahe_luts_impl(const void* src, int sd, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int gh, int gw,
                    double clip_limit, int semantics, float lo, float hi, uint32_t* hist, uint8_t* luts,
                    cudaStream_t st) {
    const Image s{src, sd, ssn, ssh};
    ClaheGeom g;
    int rc = clahe_common_checks(s, n, h, w, gh, gw, semantics, lo, hi, &g);
    if (rc) return rc;
    if ((int64_t)g.th * g.tw >= (1 << 24)) return MIE_E_SHAPE;  // counts are carried in fp32-exact range
    const LutParams lp = make_lut_params(g, clip_limit, semantics);
    const float rg = hi - lo;
    if (semantics == MIE_CLAHE_KORNIA) {
        WinCvt cv = {};
        const int mode = clahe_lut_fast_mode(g, s, lo, hi, &cv);
        if (mode >= 0) return launch_clahe_lut_fast(s, n, g, lp, hist, luts, mode, cv, st);
    }
    MIE_DISPATCH_SRC(sd, return launch_lut<SrcT>(src, n, ssn, ssh, g, lo, rg, lp, semantics, hist, luts, st));
    return MIE_OK;
}

int clahe_apply_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
                     int64_t dsn, int64_t dsh, int gh, int gw, int semantics, float lo, float hi, const uint8_t* luts,
                     cudaStream_t st) {
    ClaheGeom g;
    int rc = clahe_common_checks({src, sd, ssn, ssh}, n, h, w, gh, gw, semantics, lo, hi, &g);
    if (rc) return rc;
    if (!dst || !luts) return MIE_E_NULL;
    rc = check_dtypes(sd, dd, 0.f, 1.f);
    if (rc) return rc;
    if (semantics == MIE_CLAHE_OPENCV && dd != sd) return MIE_E_DTYPE;
    if (!plane_strides_ok({dst, dd, dsn, dsh}, n, h, w)) return MIE_E_STRIDE;
    if (n == 0) return MIE_OK;
    if (n > 65535) return MIE_E_SHAPE;
    const float rg = hi - lo;
    dim3 grid(ceil_div(w, 256), ceil_div(h, 4), (unsigned)n);
    if (semantics == MIE_CLAHE_KORNIA) {
        MIE_DISPATCH_SRC_DST(sd, dd, (clahe_apply_kernel<SrcT, DstT, MIE_CLAHE_KORNIA><<<grid, 256, 0, st>>>(
                                         (const SrcT*)src, (DstT*)dst, ssn, ssh, dsn, dsh, g, lo, rg, luts)));
    } else {
        clahe_apply_kernel<uint8_t, uint8_t, MIE_CLAHE_OPENCV><<<grid, 256, 0, st>>>(
            (const uint8_t*)src, (uint8_t*)dst, ssn, ssh, dsn, dsh, g, lo, rg, luts);
    }
    return check_launch();
}

}  // namespace mie

namespace mie {
int clahe16_impl(const void* src, void* dst, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int64_t dsn, int64_t dsh,
                 int gh, int gw, double clip_limit, void* workspace, size_t workspace_bytes, cudaStream_t st);
}

using namespace mie;

extern "C" {

// LUTs (256 B per tile, rounded up to 256 B) followed by the packed cell tables of the tuned
// interpolation kernel (2 KB per interpolation cell)
static size_t clahe_lut_region(int64_t n, int gh, int gw) { return ((size_t)n * gh * gw * kBins + 255) & ~(size_t)255; }

size_t mie_clahe_workspace_bytes(int64_t n, int h, int w, int gh, int gw) {
    (void)h; (void)w;
    if (n <= 0 || gh <= 0 || gw <= 0) return 0;
    return clahe_lut_region(n, gh, gw) + clahe_cells_bytes(n, gh, gw);
}

int mie_clahe_hist(const void* src, int src_dtype, int64_t n, int h, int w, int64_t src_stride_n,
                   int64_t src_stride_h, int gh, int gw, int semantics, float lo, float hi, uint32_t* hist,
                   void* stream) {
    if (!hist) return MIE_E_NULL;
    return clahe_luts_impl(src, src_dtype, n, h, w, src_stride_n, src_stride_h, gh, gw, 0.0, semantics, lo, hi, hist,
                           nullptr, (cudaStream_t)stream);
}

int mie_clahe_luts(const void* src, int src_dtype, int64_t n, int h, int w, int64_t src_stride_n,
                   int64_t src_stride_h, int gh, int gw, double clip_limit, int semantics, float lo, float hi,
                   uint8_t* luts, void* stream) {
    if (!luts) return MIE_E_NULL;
    return clahe_luts_impl(src, src_dtype, n, h, w, src_stride_n, src_stride_h, gh, gw, clip_limit, semantics, lo, hi,
                           nullptr, luts, (cudaStream_t)stream);
}

int mie_clahe_apply(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                    int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h, int gh,
                    int gw, int semantics, float lo, float hi, const uint8_t* luts, void* stream) {
    return clahe_apply_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                            dst_stride_h, gh, gw, semantics, lo, hi, luts, (cudaStream_t)stream);
}

int mie_clahe(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
              int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h, int gh, int gw,
              double clip_limit, int semantics, float lo, float hi, void* workspace, size_t workspace_bytes,
              void* stream) {
    const Image s{src, src_dtype, src_stride_n, src_stride_h}, d{dst, dst_dtype, dst_stride_n, dst_stride_h};
    if (semantics == MIE_CLAHE_OPENCV && src_dtype == MIE_U16) {  // 65 536-bin mode (clahe16.cu)
        if (dst_dtype != MIE_U16) return MIE_E_DTYPE;
        int rc16 = check_planes(s, d, n, h, w);
        if (rc16) return rc16;
        return clahe16_impl(src, dst, n, h, w, src_stride_n, src_stride_h, dst_stride_n, dst_stride_h, gh, gw,
                            clip_limit, workspace, workspace_bytes, (cudaStream_t)stream);
    }
    // the destination is validated with the source, before the LUT pass is launched
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    if (!workspace) return MIE_E_NULL;
    if (workspace_bytes < mie_clahe_workspace_bytes(n, h, w, gh, gw)) return MIE_E_WORKSPACE;
    rc = clahe_luts_impl(src, src_dtype, n, h, w, src_stride_n, src_stride_h, gh, gw, clip_limit, semantics, lo,
                             hi, nullptr, (uint8_t*)workspace, (cudaStream_t)stream);
    if (rc) return rc;
    // clahe_luts_impl has validated the source, the range and the geometry; clahe_apply_fast_mode accepts only a
    // destination dtype of the source's or float32
    if (semantics == MIE_CLAHE_KORNIA && n > 0 && n <= 65535) {
        ClaheGeom g;
        make_clahe_geom(h, w, gh, gw, semantics, &g);
        WinCvt cv = {};
        const int mode = clahe_apply_fast_mode(g, s, d, lo, hi, &cv);
        if (mode >= 0)
            return launch_clahe_apply_fast(s, d, n, g, (const uint8_t*)workspace,
                                           (uint8_t*)workspace + clahe_lut_region(n, gh, gw), mode, cv,
                                           (cudaStream_t)stream);
    }
    return clahe_apply_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                            dst_stride_h, gh, gw, semantics, lo, hi, (const uint8_t*)workspace, (cudaStream_t)stream);
}

}  // extern "C"
