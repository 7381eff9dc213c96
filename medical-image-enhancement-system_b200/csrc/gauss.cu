// gauss.cu — separable Gaussian blur and unsharp mask.
// Replaces kornia.filters.gaussian_blur2d / kornia.filters.unsharp_mask
// (reference pyproject.toml:8; SURVEY.md §8(a) A3, A4).
#include "stencil.cuh"
#include "window.cuh"

namespace mie {

// gauss_march.cu
int gauss_march_mode(const Image& s, const Image& d, int h, int w, int kx, int ky, int border, float lo, float hi,
                     WinCvt* cv);
int launch_gauss_march(const Image& s, const Image& d, int64_t n, int h, int w, const Taps& wx, const Taps& wy,
                       int border, int unsharp, int mode, const WinCvt& cv, cudaStream_t st);

struct GaussArgs {
    const void* src;
    void* dst;
    int64_t ssn, ssh, dsn, dsh;
    int h, w;
    int tiles_x, tiles_y;
    int border;
    int unsharp;
    float amount;   // out = fma(amount, x - blur, x); amount == 1 is kornia's x + (x - blur), bit for bit
    int clip;       // clamp the result to [0, 1] (skimage.filters.unsharp_mask without preserve_range)
    float lo, rg;
};

template <typename SrcT>
__device__ __forceinline__ float load01(const SrcT* plane, int64_t ssh, int gy, int gx, int h, int w, int border,
                                        float lo, float rg) {
    const int sy = border_index(gy, h, border), sx = border_index(gx, w, border);
    if (sy < 0 || sx < 0) return 0.0f;
    return Px<SrcT>::to01(plane[(int64_t)sy * ssh + sx], lo, rg);
}

// Fast path: square kernel of radius R in {1..4}, 64x64 output tiles.
template <typename SrcT, typename DstT, int R>
__global__ void __launch_bounds__(256)
gauss_tile_kernel(GaussArgs a, Taps wx, Taps wy) {
    extern __shared__ __align__(16) float smem[];
    float* s_in = smem;
    float* s_mid = smem + TileSmem<R>::in_words;

    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * kTile;
    const int ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * kTile;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const SrcT* plane = (const SrcT*)a.src + n * a.ssn;
    DstT* oplane = (DstT*)a.dst + n * a.dsn;

    // Coordinates further than the halo from the image only feed masked outputs;
    // clamp them so that border_index stays in its domain.
    const int ymax = a.h + R - 1, xmax = a.w + R - 1;
    tile_load<R>(s_in, ty0, tx0, [&](int gy, int gx) {
        return load01<SrcT>(plane, a.ssh, min(gy, ymax), min(gx, xmax), a.h, a.w, a.border, a.lo, a.rg);
    });
    __syncthreads();
    tile_row_pass<R>(s_in, s_mid, wx);
    __syncthreads();
    tile_col_pass<R>(s_mid, wy, [&](int r, int c, float4 v) {
        const int y = ty0 + r, x = tx0 + c;
        if (y >= a.h) return;
        float o[4] = {v.x, v.y, v.z, v.w};
        if (a.unsharp) {
            const float* ctr = s_in + (r + R) * TileSmem<R>::pin + c + R;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                o[k] = __fmaf_rn(a.amount, __fsub_rn(ctr[k], o[k]), ctr[k]);
                if (a.clip) o[k] = fminf(fmaxf(o[k], 0.0f), 1.0f);
            }
        }
        DstT* drow = oplane + (int64_t)y * a.dsh;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x + k < a.w) drow[x + k] = Px<DstT>::from01(o[k], a.lo, a.rg);
    });
}

// Generic path: any odd kx, ky <= MIE_MAX_TAPS; 32x32 output tiles, runtime tap loops.
template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256)
gauss_generic_kernel(GaussArgs a, Taps wx, int rx, Taps wy, int ry) {
    extern __shared__ __align__(16) float smem[];
    constexpr int T = 32;
    const int ew = T + 2 * rx, eh = T + 2 * ry;
    float* s_in = smem;            // eh x ew
    float* s_mid = smem + eh * ew;  // eh x T

    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * T;
    const int ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * T;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const SrcT* plane = (const SrcT*)a.src + n * a.ssn;
    DstT* oplane = (DstT*)a.dst + n * a.dsn;
    const int ymax = a.h + ry - 1, xmax = a.w + rx - 1;

    for (int i = threadIdx.x; i < eh * ew; i += 256) {
        const int r = i / ew, c = i - r * ew;
        s_in[i] = load01<SrcT>(plane, a.ssh, min(ty0 - ry + r, ymax), min(tx0 - rx + c, xmax), a.h, a.w, a.border,
                               a.lo, a.rg);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < eh * T; i += 256) {
        const int r = i / T, c = i - r * T;
        const float* p = s_in + r * ew + c;
        float acc = __fmul_rn(wx.w[0], p[0]);
        for (int t = 1; t <= 2 * rx; ++t) acc = __fmaf_rn(wx.w[t], p[t], acc);
        s_mid[i] = acc;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < T * T; i += 256) {
        const int r = i / T, c = i - r * T;
        const int y = ty0 + r, x = tx0 + c;
        if (y >= a.h || x >= a.w) continue;
        const float* p = s_mid + r * T + c;
        float acc = __fmul_rn(wy.w[0], p[0]);
        for (int t = 1; t <= 2 * ry; ++t) acc = __fmaf_rn(wy.w[t], p[t * T], acc);
        if (a.unsharp) {
            const float ctr = s_in[(r + ry) * ew + c + rx];
            acc = __fmaf_rn(a.amount, __fsub_rn(ctr, acc), ctr);
            if (a.clip) acc = fminf(fmaxf(acc, 0.0f), 1.0f);
        }
        oplane[(int64_t)y * a.dsh + x] = Px<DstT>::from01(acc, a.lo, a.rg);
    }
}

template <typename SrcT, typename DstT, int R>
static int launch_tile(const GaussArgs& a, const Taps& wx, const Taps& wy, int64_t n, cudaStream_t st) {
    MIE_ENSURE_SMEM((gauss_tile_kernel<SrcT, DstT, R>), TileSmem<R>::bytes);
    GaussArgs b = a;
    b.tiles_x = ceil_div(a.w, kTile);
    b.tiles_y = ceil_div(a.h, kTile);
    const int64_t blocks = n * b.tiles_x * b.tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    gauss_tile_kernel<SrcT, DstT, R><<<(unsigned)blocks, 256, TileSmem<R>::bytes, st>>>(b, wx, wy);
    return check_launch();
}

template <typename SrcT, typename DstT>
static int launch_any(const GaussArgs& a, const Taps& wx, int kx, const Taps& wy, int ky, int64_t n,
                      cudaStream_t st) {
    if (kx == ky) {
        switch (kx / 2) {
            case 1: return launch_tile<SrcT, DstT, 1>(a, wx, wy, n, st);
            case 2: return launch_tile<SrcT, DstT, 2>(a, wx, wy, n, st);
            case 3: return launch_tile<SrcT, DstT, 3>(a, wx, wy, n, st);
            case 4: return launch_tile<SrcT, DstT, 4>(a, wx, wy, n, st);
            default: break;
        }
    }
    const int rx = kx / 2, ry = ky / 2;
    const size_t smem = (size_t)((32 + 2 * ry) * (32 + 2 * rx) + (32 + 2 * ry) * 32) * 4;
    MIE_ENSURE_SMEM((gauss_generic_kernel<SrcT, DstT>), 64 * 1024);
    GaussArgs b = a;
    b.tiles_x = ceil_div(a.w, 32);
    b.tiles_y = ceil_div(a.h, 32);
    const int64_t blocks = n * b.tiles_x * b.tiles_y;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    gauss_generic_kernel<SrcT, DstT><<<(unsigned)blocks, 256, smem, st>>>(b, wx, rx, wy, ry);
    return check_launch();
}

int check_taps(const float* wx, int kx, const float* wy, int ky, int border, int h, int w) {
    if (!wx || !wy) return MIE_E_NULL;
    if (kx <= 0 || ky <= 0 || !(kx & 1) || !(ky & 1) || kx > MIE_MAX_TAPS || ky > MIE_MAX_TAPS) return MIE_E_KERNEL;
    if (border < MIE_BORDER_CONSTANT || border > MIE_BORDER_SYMMETRIC) return MIE_E_BORDER;
    // torch F.pad: reflect needs pad < dim, circular pad <= dim.
    if (border == MIE_BORDER_REFLECT && (kx / 2 >= w || ky / 2 >= h)) return MIE_E_BORDER;
    if (border == MIE_BORDER_CIRCULAR && (kx / 2 > w || ky / 2 > h)) return MIE_E_BORDER;
    return MIE_OK;
}

// F32 sources may also be written to any integer dtype (internal use by the
// unfused chain fallback); the public ABI restricts dst to {src, F32}.
int gauss_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
               int64_t dsn, int64_t dsh, const float* wxp, int kx, const float* wyp, int ky, int border, float lo,
               float hi, int unsharp, bool internal, cudaStream_t st, float amount, int clip) {
    const Image s{src, sd, ssn, ssh}, d{dst, dd, dsn, dsh};
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    if (!valid_dtype(sd) || !valid_dtype(dd)) return MIE_E_DTYPE;
    if (!(internal && sd == MIE_F32) && dd != sd && dd != MIE_F32) return MIE_E_DTYPE;
    if ((sd != MIE_F32 || dd != MIE_F32) && !(hi > lo)) return MIE_E_RANGE;
    rc = check_taps(wxp, kx, wyp, ky, border, h, w);
    if (rc) return rc;
    if (n == 0) return MIE_OK;
    Taps wx, wy;
    for (int i = 0; i < MIE_MAX_TAPS; ++i) {
        wx.w[i] = i < kx ? wxp[i] : 0.f;
        wy.w[i] = i < ky ? wyp[i] : 0.f;
    }
    // common geometry (square 9-tap kernel, W % 128 == 0, H % 64 == 0): marching kernel (gauss_march.cu)
    if (!unsharp || (amount == 1.0f && !clip)) {
        WinCvt cv = {};
        const int mode = gauss_march_mode(s, d, h, w, kx, ky, border, lo, hi, &cv);
        if (mode >= 0) return launch_gauss_march(s, d, n, h, w, wx, wy, border, unsharp, mode, cv, st);
    }
    GaussArgs a;
    a.src = src; a.dst = dst; a.ssn = ssn; a.ssh = ssh; a.dsn = dsn; a.dsh = dsh;
    a.h = h; a.w = w; a.tiles_x = a.tiles_y = 0; a.border = border; a.unsharp = unsharp;
    a.amount = amount; a.clip = clip;
    a.lo = lo; a.rg = hi - lo;
    if (sd == MIE_F32 && dd != MIE_F32) {
        switch (dd) {
            case MIE_U8: return launch_any<float, uint8_t>(a, wx, kx, wy, ky, n, st);
            case MIE_U16: return launch_any<float, uint16_t>(a, wx, kx, wy, ky, n, st);
            default: return launch_any<float, int16_t>(a, wx, kx, wy, ky, n, st);
        }
    }
    MIE_DISPATCH_SRC_DST(sd, dd, return (launch_any<SrcT, DstT>(a, wx, kx, wy, ky, n, st)));
    return MIE_OK;
}

}  // namespace mie

using namespace mie;

extern "C" {

int mie_gaussian2d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                   const float* wx, int kx, const float* wy, int ky, int border, float lo, float hi, void* stream) {
    return gauss_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                      dst_stride_h, wx, kx, wy, ky, border, lo, hi, 0, false, (cudaStream_t)stream, 1.0f, 0);
}

int mie_unsharp(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                const float* wx, int kx, const float* wy, int ky, int border, float lo, float hi, void* stream) {
    return gauss_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                      dst_stride_h, wx, kx, wy, ky, border, lo, hi, 1, false, (cudaStream_t)stream, 1.0f, 0);
}

int mie_unsharp_amount(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                       int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n, int64_t dst_stride_h,
                       const float* wx, int kx, const float* wy, int ky, int border, float amount, int clip, float lo,
                       float hi, void* stream) {
    return gauss_impl(src, dst, src_dtype, dst_dtype, n, h, w, src_stride_n, src_stride_h, dst_stride_n,
                      dst_stride_h, wx, kx, wy, ky, border, lo, hi, 1, false, (cudaStream_t)stream, amount,
                      clip ? 1 : 0);
}

}  // extern "C"
