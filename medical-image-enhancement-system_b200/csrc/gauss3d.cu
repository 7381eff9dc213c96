// gauss3d.cu — separable 3-D Gaussian blur and unsharp mask over whole (d, h, w) volumes:
// skimage.filters.gaussian / skimage.filters.unsharp_mask on a 3-D array (scipy.ndimage.gaussian_filter over all
// three axes).  Restated per voxel by orc_gaussian3d_ex in tests/gaussian3d_oracle.c
// (built on oracle/mie_oracle.c).
//
// Operation order: x pass, then y pass, then z pass; each pass acc = w[0]*v[0]; acc = fma(w[t], v[t], acc) in tap
// order, the rule of the 2-D kernels (stencil.cuh).  With kz == 1 (weight 1.0) the z pass is exact, so a volume blurred
// with sigma (0, s, s) equals the per-plane 2-D result bit for bit.  Every source index goes through border_index, so
// any radius is legal on any axis length (thin volumes included).
//
// Schedule (one launch, no fp32 intermediate in global memory): a CTA owns a 32-column x TY-row tile of the volume and
// a z-range [z0, z1).  It walks the source planes z0 - rz .. z1 - 1 + rz in order; for each plane it stages the tile
// with its (ry, rx) halo in shared memory, runs the x pass (shared -> shared) and the y pass (shared -> registers), and
// feeds the result to the z pass.  The z pass is a register ring of partial accumulators: the arriving plane applies
// fma(w[t], v, acc) to every live output plane, the plane that received its last tap is written out and the ring
// shifts by one.  Planes arrive in tap order, so this is the gather-form fma chain, bit for bit.  The next plane's
// source values are loaded into registers before the y / z work of the current one, so their latency is covered.
#include "mie_common.cuh"

namespace mie {

constexpr int kG3Cols = 32;      // tile columns (one per lane)
constexpr int kG3Threads = 256;  // 8 warps; warp g owns tile rows g*P .. g*P + P - 1

// R: radius bucket, >= every axis radius of the launch.  Loops run to the bucket with per-tap guards against the
// actual tap counts, so register windows are indexed by constants only.
template <int R>
struct G3Shape {
    static constexpr int P = R <= 4 ? 4 : 2;           // output rows per thread
    static constexpr int TY = 8 * P;                   // tile rows
    static constexpr int KZ = 2 * R + 1;               // z ring slots
    static constexpr int ROWS = TY + 2 * R;            // haloed rows (bucket)
    static constexpr int NV = (4 + 2 * R + 3) / 4;     // float4 loads per x-pass window (4 outputs)
    static constexpr int PITCH = 28 + 4 * NV;          // >= 32 + 2R; covers segment 7's window
    static constexpr int FR = (ROWS + 7) / 8;          // staged rows per warp
};

struct Gauss3Args {
    const void* src;
    void* dst;
    int64_t ssn, ssd, ssh, dsn, dsd, dsh;
    int d, h, w;
    int kx, ky, kz;
    int tiles_x, tiles_y, zsplit, zlen;
    int border, unsharp, clip;
    float amount, lo, rg;
};

// wzr: the z weights in reverse order (wzr[u] = wz[kz - 1 - u]): ring slot u is the output plane that takes tap
// kz - 1 - u from the arriving plane, so the slot index stays a constant.
template <typename SrcT, typename DstT, int R>
__global__ void __launch_bounds__(kG3Threads)
gauss3d_kernel(Gauss3Args a, Taps wx, Taps wy, Taps wzr) {
    using S = G3Shape<R>;
    __shared__ __align__(16) float s_in[S::ROWS * S::PITCH];
    __shared__ __align__(16) float s_mid[S::ROWS * kG3Cols];
    __shared__ int s_col[2 * kG3Cols];
    __shared__ int s_row[S::ROWS];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t b = blockIdx.x;
    const int tx = (int)(b % a.tiles_x); b /= a.tiles_x;
    const int ty = (int)(b % a.tiles_y); b /= a.tiles_y;
    const int zs = (int)(b % a.zsplit);
    const int64_t n = b / a.zsplit;
    const int x0 = tx * kG3Cols, y0 = ty * S::TY;
    const int z0 = zs * a.zlen, z1 = min(z0 + a.zlen, a.d);
    const int rx = a.kx >> 1, ry = a.ky >> 1, rz = a.kz >> 1;
    const int ew = kG3Cols + 2 * rx, eh = S::TY + 2 * ry;
    const SrcT* src = (const SrcT*)a.src + n * a.ssn;
    DstT* dst = (DstT*)a.dst + n * a.dsn;

    for (int c = tid; c < ew; c += kG3Threads) s_col[c] = border_index(x0 - rx + c, a.w, a.border);
    for (int r = tid; r < eh; r += kG3Threads) s_row[r] = border_index(y0 - ry + r, a.h, a.border);
    __syncthreads();

    // Staging: thread (lane, warp) holds haloed columns lane, lane + 32 of rows warp + 8 i.  Raw values are held
    // across the y / z work and converted when they are stored.
    SrcT raw[S::FR][2];
    unsigned live = 0;
    auto fetch = [&](int zv) {
        const int sz = border_index(zv, a.d, a.border);
        const SrcT* plane = src + (int64_t)(sz < 0 ? 0 : sz) * a.ssd;
        live = 0;
#pragma unroll
        for (int i = 0; i < S::FR; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int r = warp + 8 * i, c = lane + 32 * j;
                raw[i][j] = SrcT(0);
                if (r < eh && c < ew && sz >= 0) {
                    const int sy = s_row[r], sx = s_col[c];
                    if (sy >= 0 && sx >= 0) {
                        raw[i][j] = plane[(int64_t)sy * a.ssh + sx];
                        live |= 1u << (2 * i + j);
                    }
                }
            }
    };
    auto stash = [&]() {
#pragma unroll
        for (int i = 0; i < S::FR; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int r = warp + 8 * i, c = lane + 32 * j;
                if (r < eh && c < ew)
                    s_in[r * S::PITCH + c] = (live >> (2 * i + j)) & 1u ? Px<SrcT>::to01(raw[i][j], a.lo, a.rg) : 0.0f;
            }
    };
    // x pass: eh rows x 32 outputs, four consecutive outputs per work item.
    auto xpass = [&]() {
        for (int i = tid; i < eh * 8; i += kG3Threads) {
            const int r = i >> 3, seg = i & 7;
            const float4* p = reinterpret_cast<const float4*>(s_in + r * S::PITCH + seg * 4);
            float win[4 * S::NV];
#pragma unroll
            for (int v = 0; v < S::NV; ++v) {
                const float4 t = p[v];
                win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
            }
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float acc = __fmul_rn(wx.w[0], win[j]);
#pragma unroll
                for (int t = 1; t <= 2 * R; ++t)
                    if (t < a.kx) acc = __fmaf_rn(wx.w[t], win[j + t], acc);
                o[j] = acc;
            }
            *reinterpret_cast<float4*>(s_mid + r * kG3Cols + seg * 4) = make_float4(o[0], o[1], o[2], o[3]);
        }
    };

    const int zb = z0 - rz, ze = z1 + rz;   // source planes [zb, ze)
    fetch(zb);
    stash();
    __syncthreads();
    xpass();
    __syncthreads();

    const int x = x0 + lane;
    float acc[S::P][S::KZ];
#pragma unroll
    for (int p = 0; p < S::P; ++p)
#pragma unroll
        for (int u = 0; u < S::KZ; ++u) acc[p][u] = 0.0f;

    for (int zv = zb; zv < ze; ++zv) {
        const bool more = zv + 1 < ze;
        if (more) fetch(zv + 1);
        // y pass: rows warp*P + p of the tile, column lane.
        float win[S::P + 2 * R];
#pragma unroll
        for (int i = 0; i < S::P + 2 * R; ++i) win[i] = s_mid[(warp * S::P + i) * kG3Cols + lane];
        const bool emit = zv - zb >= a.kz - 1;
        const int o = zv - rz;   // output plane that receives its last tap from this plane
#pragma unroll
        for (int p = 0; p < S::P; ++p) {
            float v = __fmul_rn(wy.w[0], win[p]);
#pragma unroll
            for (int t = 1; t <= 2 * R; ++t)
                if (t < a.ky) v = __fmaf_rn(wy.w[t], win[p + t], v);
#pragma unroll
            for (int u = 0; u < S::KZ; ++u) {
                if (u < a.kz - 1) acc[p][u] = __fmaf_rn(wzr.w[u], v, acc[p][u]);
                else if (u == a.kz - 1) acc[p][u] = __fmul_rn(wzr.w[u], v);
            }
            const int y = y0 + warp * S::P + p;
            if (emit && y < a.h && x < a.w) {
                float r = acc[p][0];
                if (a.unsharp) {
                    const float c = Px<SrcT>::to01(src[(int64_t)o * a.ssd + (int64_t)y * a.ssh + x], a.lo, a.rg);
                    r = __fmaf_rn(a.amount, __fsub_rn(c, r), c);
                    if (a.clip) r = fminf(fmaxf(r, 0.0f), 1.0f);
                }
                dst[(int64_t)o * a.dsd + (int64_t)y * a.dsh + x] = Px<DstT>::from01(r, a.lo, a.rg);
            }
#pragma unroll
            for (int u = 0; u + 1 < S::KZ; ++u) acc[p][u] = acc[p][u + 1];
        }
        if (more) stash();
        __syncthreads();   // s_in complete; every y-pass read of s_mid done
        if (more) xpass();
        __syncthreads();
    }
}

template <typename SrcT, typename DstT, int R>
static int launch3(Gauss3Args a, const Taps& wx, const Taps& wy, const Taps& wzr, int64_t n, cudaStream_t st) {
    using S = G3Shape<R>;
    a.tiles_x = ceil_div(a.w, kG3Cols);
    a.tiles_y = ceil_div(a.h, S::TY);
    // z split from geometry alone: about eight CTAs per SM in all, but z-ranges of at least max(8, 4 rz) planes so
    // that the 2 rz planes of z halo each range reads stay a small share of its work.
    const int64_t cols = n * a.tiles_x * a.tiles_y;
    const int64_t want = (148 * 8 + cols - 1) / cols;
    const int min_len = max(8, 4 * (a.kz >> 1));
    const int64_t most = a.d / min_len > 1 ? a.d / min_len : 1;
    a.zsplit = (int)(want < most ? want : most);
    a.zlen = ceil_div(a.d, a.zsplit);
    a.zsplit = ceil_div(a.d, a.zlen);
    const int64_t blocks = cols * a.zsplit;
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    gauss3d_kernel<SrcT, DstT, R><<<(unsigned)blocks, kG3Threads, 0, st>>>(a, wx, wy, wzr);
    return check_launch();
}

template <typename SrcT, typename DstT>
static int launch3_any(const Gauss3Args& a, const Taps& wx, const Taps& wy, const Taps& wzr, int64_t n,
                       cudaStream_t st) {
    const int r = max(a.kx, max(a.ky, a.kz)) >> 1;
    if (r <= 2) return launch3<SrcT, DstT, 2>(a, wx, wy, wzr, n, st);
    if (r <= 4) return launch3<SrcT, DstT, 4>(a, wx, wy, wzr, n, st);
    if (r <= 8) return launch3<SrcT, DstT, 8>(a, wx, wy, wzr, n, st);
    return launch3<SrcT, DstT, 16>(a, wx, wy, wzr, n, st);
}

static bool bad_taps(int k) { return k <= 0 || !(k & 1) || k > MIE_MAX_TAPS; }

static int gauss3d_impl(const void* src, void* dst, int sd, int dd, int64_t n, int d, int h, int w, int64_t ssn,
                        int64_t ssd, int64_t ssh, int64_t dsn, int64_t dsd, int64_t dsh, const float* wxp, int kx,
                        const float* wyp, int ky, const float* wzp, int kz, int border, int unsharp, float amount,
                        int clip, float lo, float hi, cudaStream_t st) {
    int rc = check_volumes({src, sd, ssn, ssh}, ssd, {dst, dd, dsn, dsh}, dsd, n, d, h, w);
    if (rc) return rc;
    rc = check_dtypes(sd, dd, lo, hi);
    if (rc) return rc;
    if (!wxp || !wyp || !wzp) return MIE_E_NULL;
    if (bad_taps(kx) || bad_taps(ky) || bad_taps(kz)) return MIE_E_KERNEL;
    if (border < MIE_BORDER_CONSTANT || border > MIE_BORDER_SYMMETRIC) return MIE_E_BORDER;
    // tile coordinates (index + radius) stay in int
    if (d > 2147483647 - 64 || h > 2147483647 - 64 || w > 2147483647 - 64) return MIE_E_SHAPE;
    if (n == 0) return MIE_OK;
    Taps wx, wy, wzr;
    for (int i = 0; i < MIE_MAX_TAPS; ++i) {
        wx.w[i] = i < kx ? wxp[i] : 0.f;
        wy.w[i] = i < ky ? wyp[i] : 0.f;
        wzr.w[i] = i < kz ? wzp[kz - 1 - i] : 0.f;
    }
    Gauss3Args a;
    a.src = src; a.dst = dst;
    a.ssn = ssn; a.ssd = ssd; a.ssh = ssh; a.dsn = dsn; a.dsd = dsd; a.dsh = dsh;
    a.d = d; a.h = h; a.w = w; a.kx = kx; a.ky = ky; a.kz = kz;
    a.tiles_x = a.tiles_y = a.zsplit = a.zlen = 0;
    a.border = border; a.unsharp = unsharp; a.clip = clip ? 1 : 0;
    a.amount = amount; a.lo = lo; a.rg = hi - lo;
    MIE_DISPATCH_SRC_DST(sd, dd, return (launch3_any<SrcT, DstT>(a, wx, wy, wzr, n, st)));
    return MIE_OK;
}

}  // namespace mie

using namespace mie;

extern "C" {

int mie_gaussian3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h, int64_t dst_stride_n,
                   int64_t dst_stride_d, int64_t dst_stride_h, const float* wx, int kx, const float* wy, int ky,
                   const float* wz, int kz, int border, float lo, float hi, void* stream) {
    return gauss3d_impl(src, dst, src_dtype, dst_dtype, n, d, h, w, src_stride_n, src_stride_d, src_stride_h,
                        dst_stride_n, dst_stride_d, dst_stride_h, wx, kx, wy, ky, wz, kz, border, 0, 1.0f, 0, lo, hi,
                        (cudaStream_t)stream);
}

int mie_unsharp3d(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int d, int h, int w,
                  int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h, int64_t dst_stride_n,
                  int64_t dst_stride_d, int64_t dst_stride_h, const float* wx, int kx, const float* wy, int ky,
                  const float* wz, int kz, int border, float amount, int clip, float lo, float hi, void* stream) {
    return gauss3d_impl(src, dst, src_dtype, dst_dtype, n, d, h, w, src_stride_n, src_stride_d, src_stride_h,
                        dst_stride_n, dst_stride_d, dst_stride_h, wx, kx, wy, ky, wz, kz, border, 1, amount, clip, lo,
                        hi, (cudaStream_t)stream);
}

}  // extern "C"
