// chain.cu — fused Gaussian denoise -> CLAHE -> unsharp mask (BASELINE.json config 2).
//
// Two launches:
//   chain_a : one block per CLAHE tile.  Gaussian of the haloed tile in shared
//             memory; the blurred value G never leaves the SM — only its lookup
//             index trunc(G*255) (1 byte/pixel) is written, while floor(G*256)
//             feeds the shared-memory histogram; clip / redistribute / scan -> LUT
//             in the same block.
//   chain_b : one block per 64x64 output tile.  Reads the index plane with a
//             halo, rebuilds the CLAHE output C = blend(LUTs[idx]) / 255 for every
//             haloed pixel (C depends on idx and position only), blurs C, forms
//             C + (C - blur(C)) and quantises.
// The result equals mie_gaussian2d -> mie_clahe -> mie_unsharp with F32
// intermediates bit for bit (same operation order; tests/test_chain_gpu.py).
// Shapes the fused kernels do not cover (CLAHE padding needed, tiles > 64 px,
// non-square or > 9-tap kernels) run those three stages unfused.

#include "window.cuh"

namespace mie {

int gauss_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
               int64_t dsn, int64_t dsh, const float* wxp, int kx, const float* wyp, int ky, int border, float lo,
               float hi, int unsharp, bool internal, cudaStream_t st, float amount = 1.0f, int clip = 0);
int check_taps(const float* wx, int kx, const float* wy, int ky, int border, int h, int w);
int clahe_luts_impl(const void* src, int sd, int64_t n, int h, int w, int64_t ssn, int64_t ssh, int gh, int gw,
                    double clip_limit, int semantics, float lo, float hi, uint32_t* hist, uint8_t* luts,
                    cudaStream_t st);
int clahe_apply_impl(const void* src, void* dst, int sd, int dd, int64_t n, int h, int w, int64_t ssn, int64_t ssh,
                     int64_t dsn, int64_t dsh, int gh, int gw, int semantics, float lo, float hi, const uint8_t* luts,
                     cudaStream_t st);

template <typename SrcT, int R>
__global__ void __launch_bounds__(256)
chain_a_kernel(ChainAArgs a, Taps wx, Taps wy) {
    extern __shared__ __align__(16) float smem[];
    float* s_in = smem;
    float* s_mid = smem + TileSmem<R>::in_words;
    int* s_hist = reinterpret_cast<int*>(smem + TileSmem<R>::in_words + TileSmem<R>::mid_words);  // [8][256]
    __shared__ int s_red[8];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int i = 0; i < 8; ++i) s_hist[i * kBins + tid] = 0;

    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % a.g.gw), ty = (int)((tile / a.g.gw) % a.g.gh);
    const int64_t n = tile / ((int64_t)a.g.gw * a.g.gh);
    const int tx0 = tx * a.g.tw, ty0 = ty * a.g.th;
    const SrcT* plane = (const SrcT*)a.src + n * a.ssn;
    uint8_t* iplane = a.idx + n * (int64_t)a.g.h * a.g.w;
    const int h = a.g.h, w = a.g.w;

    tile_load<R>(s_in, ty0, tx0, [&](int gy, int gx) {
        const int sy = border_index(gy, h, a.border), sx = border_index(gx, w, a.border);
        if (sy < 0 || sx < 0) return 0.0f;
        return Px<SrcT>::to01(plane[(int64_t)sy * a.ssh + sx], a.lo, a.rg);
    });
    __syncthreads();
    tile_row_pass<R>(s_in, s_mid, wx);
    __syncthreads();
    const bool packed = ((w | a.g.tw) & 3) == 0;
    tile_col_pass<R>(s_mid, wy, [&](int r, int c, float4 v) {
        const float gv[4] = {v.x, v.y, v.z, v.w};
        const bool row_ok = r < a.g.th;
        uint32_t pack = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool ok = row_ok && (c + k) < a.g.tw;
            const int bin = ok ? kornia_bin(gv[k]) : -1;
            pack |= (uint32_t)kornia_idx(gv[k]) << (8 * k);
            const unsigned act = __ballot_sync(0xffffffffu, bin >= 0);
            if (act) {
                const int leader = __ffs(act) - 1;
                const int b0 = __shfl_sync(0xffffffffu, bin, leader);
                if (__all_sync(0xffffffffu, bin < 0 || bin == b0)) {
                    if (lane == leader) s_hist[warp * kBins + b0] += __popc(act);
                } else if (bin >= 0) {
                    atomicAdd(&s_hist[warp * kBins + bin], 1);
                }
                __syncwarp();
            }
        }
        if (!row_ok) return;
        uint8_t* irow = iplane + (int64_t)(ty0 + r) * w + tx0 + c;
        if (packed && c + 3 < a.g.tw) {
            *reinterpret_cast<uint32_t*>(irow) = pack;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (c + k < a.g.tw) irow[k] = (uint8_t)(pack >> (8 * k));
        }
    });
    __syncthreads();
    int hv = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) hv += s_hist[i * kBins + tid];
    a.luts[tile * kBins + tid] = lut_entry_from_count<MIE_CLAHE_KORNIA>(hv, a.lp, s_red);
}

struct AxisEntry {
    int o0, o1;  // LUT offsets (bytes) of the two neighbouring tiles along this axis
    float wgt;   // weight of o0
    int src;     // mapped source coordinate, -1 = constant border
};

template <typename DstT, int R>
__global__ void __launch_bounds__(256)
chain_b_kernel(ChainBArgs a, Taps wx, Taps wy) {
    extern __shared__ __align__(16) float smem[];
    constexpr int E = kTile + 2 * R;
    float* s_in = smem;
    float* s_mid = smem + TileSmem<R>::in_words;
    uint8_t* s_lut = reinterpret_cast<uint8_t*>(smem + TileSmem<R>::in_words + TileSmem<R>::mid_words);
    __shared__ AxisEntry s_row[E], s_col[E];
    __shared__ int s_lim[4];  // jlo, jhi, ilo, ihi

    const int tid = threadIdx.x;
    const int64_t tile = blockIdx.x;
    const int tx0 = (int)(tile % a.tiles_x) * kTile;
    const int ty0 = (int)((tile / a.tiles_x) % a.tiles_y) * kTile;
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const int h = a.g.h, w = a.g.w;

    if (tid == 0) { s_lim[0] = a.g.gh; s_lim[1] = -1; s_lim[2] = a.g.gw; s_lim[3] = -1; }
    __syncthreads();
    if (tid < 2 * E) {
        const bool is_row = tid < E;
        const int k = is_row ? tid : tid - E;
        const int len = is_row ? h : w;
        // coordinates beyond image+halo only feed masked outputs: clamp
        const int raw = min((is_row ? ty0 : tx0) - R + k, len + R - 1);
        AxisEntry e;
        e.src = border_index(raw, len, a.border);
        e.o0 = e.o1 = 0; e.wgt = 0.f;
        if (e.src >= 0) {
            kornia_axis(e.src, is_row ? a.g.th : a.g.tw, is_row ? a.g.gh : a.g.gw, e.o0, e.o1, e.wgt);
            atomicMin(&s_lim[is_row ? 0 : 2], e.o0);
            atomicMax(&s_lim[is_row ? 1 : 3], e.o1);
        }
        (is_row ? s_row : s_col)[k] = e;
    }
    __syncthreads();
    const int jlo = s_lim[0], ilo = s_lim[2];
    const int nlr = s_lim[1] - jlo + 1, nlc = s_lim[3] - ilo + 1;
    if (nlr * nlc > a.max_lut_tiles) __trap();   // host-side capacity rule (fused_ok) violated: never write past s_lut
    // stage the nlr x nlc neighbourhood of LUTs (256 B each) with 16-byte copies
    {
        const uint4* gl = reinterpret_cast<const uint4*>(a.luts + n * (int64_t)a.g.gh * a.g.gw * kBins);
        uint4* sl = reinterpret_cast<uint4*>(s_lut);
        const int total = nlr * nlc * 16;
        for (int i = tid; i < total; i += 256) {
            const int t = i >> 4, part = i & 15;
            const int jr = t / nlc, ic = t - jr * nlc;
            sl[i] = gl[((int64_t)(jlo + jr) * a.g.gw + (ilo + ic)) * 16 + part];
        }
    }
    if (tid < 2 * E) {
        const bool is_row = tid < E;
        AxisEntry& e = (is_row ? s_row : s_col)[is_row ? tid : tid - E];
        if (is_row) { e.o0 = (e.o0 - jlo) * nlc * kBins; e.o1 = (e.o1 - jlo) * nlc * kBins; }
        else { e.o0 = (e.o0 - ilo) * kBins; e.o1 = (e.o1 - ilo) * kBins; }
    }
    __syncthreads();

    const uint8_t* iplane = a.idx + n * (int64_t)h * w;
    for (int i = tid; i < E * E; i += 256) {
        const int r = i / E, c = i - r * E;
        const AxisEntry er = s_row[r], ec = s_col[c];
        float val = 0.0f;
        if (er.src >= 0 && ec.src >= 0) {
            const int idx = iplane[(int64_t)er.src * w + ec.src];
            const float tl = (float)s_lut[er.o0 + ec.o0 + idx], tr = (float)s_lut[er.o0 + ec.o1 + idx];
            const float bl = (float)s_lut[er.o1 + ec.o0 + idx], br = (float)s_lut[er.o1 + ec.o1 + idx];
            val = __fdiv_rn(kornia_blend(tl, tr, bl, br, ec.wgt, er.wgt), 255.0f);
        }
        s_in[r * TileSmem<R>::pin + c] = val;
    }
    __syncthreads();
    tile_row_pass<R>(s_in, s_mid, wx);
    __syncthreads();
    DstT* oplane = (DstT*)a.dst + n * a.dsn;
    tile_col_pass<R>(s_mid, wy, [&](int r, int c, float4 v) {
        const int y = ty0 + r, x = tx0 + c;
        if (y >= h) return;
        const float o[4] = {v.x, v.y, v.z, v.w};
        const float* ctr = s_in + (r + R) * TileSmem<R>::pin + c + R;
        DstT* drow = oplane + (int64_t)y * a.dsh;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (x + k < w) drow[x + k] = Px<DstT>::from01(__fadd_rn(ctr[k], __fsub_rn(ctr[k], o[k])), a.lo, a.rg);
    });
}

// ---------------------------------------------------------------- host side
static bool fused_ok(const ClaheGeom& g, int kgx, int kgy, int kux, int kuy, int border, int* lut_cap) {
    if (kgx != kgy || kux != kuy) return false;
    if (kgx < 3 || kgx > 9 || kux < 3 || kux > 9) return false;
    if (g.hp != g.h || g.wp != g.w) return false;
    if (g.th > kTile || g.tw > kTile) return false;
    const int R = kux / 2;
    // A block's haloed rows / columns touch a contiguous run of tiles — except with a circular border, where
    // the halo of the first / last blocks wraps to the opposite edge: the run then spans the whole grid.
    const bool wrap = border == MIE_BORDER_CIRCULAR;
    const int capr = wrap ? g.gh : (kTile + 2 * R) / g.th + 3, capc = wrap ? g.gw : (kTile + 2 * R) / g.tw + 3;
    const int cr = capr < g.gh ? capr : g.gh, cc = capc < g.gw ? capc : g.gw;
    if ((size_t)cr * cc * kBins > 96 * 1024) return false;
    *lut_cap = cr * cc;
    return true;
}

template <typename SrcT, int R>
static int launch_a(const ChainAArgs& a, const Taps& wx, const Taps& wy, int64_t n, cudaStream_t st) {
    const size_t smem = TileSmem<R>::bytes + 8 * kBins * 4;
    MIE_ENSURE_SMEM((chain_a_kernel<SrcT, R>), smem);
    chain_a_kernel<SrcT, R><<<(unsigned)(n * a.g.gh * a.g.gw), 256, smem, st>>>(a, wx, wy);
    return check_launch();
}

template <typename DstT, int R>
static int launch_b(const ChainBArgs& a, const Taps& wx, const Taps& wy, int64_t n, int lut_cap, cudaStream_t st) {
    const size_t smem = TileSmem<R>::bytes + (size_t)lut_cap * kBins;
    MIE_ENSURE_SMEM((chain_b_kernel<DstT, R>), 200 * 1024);
    chain_b_kernel<DstT, R><<<(unsigned)(n * a.tiles_x * a.tiles_y), 256, smem, st>>>(a, wx, wy);
    return check_launch();
}

static void fill_taps(Taps& t, const float* w, int k) {
    for (int i = 0; i < MIE_MAX_TAPS; ++i) t.w[i] = i < k ? w[i] : 0.f;
}

}  // namespace mie

using namespace mie;

extern "C" {

int mie_chain_is_fused(int h, int w, int gh, int gw, int kgx, int kgy, int kux, int kuy) {
    ClaheGeom g;
    int cap = 0;
    if (make_clahe_geom(h, w, gh, gw, MIE_CLAHE_KORNIA, &g)) return 0;
    if (!fused_ok(g, kgx, kgy, kux, kuy, MIE_BORDER_REFLECT, &cap)) return 0;
    // 2: tuned kernels (chain_a, cell packing, chain_b = 3 launches) when the buffers are 16-byte
    // aligned and the integer range is the dtype default; 1: generic fused kernels (2 launches)
    return (g.th == kTile && g.tw == kTile && kux == 9) ? 2 : 1;
}

size_t mie_chain_workspace_bytes(int64_t n, int h, int w, int gh, int gw) {
    if (n <= 0 || h <= 0 || w <= 0 || gh <= 0 || gw <= 0) return 0;
    // LUTs (256 B per tile, rounded to 256 B) + one fp32 plane per image: enough
    // for the unfused fallback; the fused path uses 1 byte per pixel of it.
    size_t luts = (size_t)n * gh * gw * kBins;
    return luts + (size_t)n * h * w * 4;
}

int mie_chain_gauss_clahe_unsharp(const void* src, void* dst, int src_dtype, int dst_dtype, int64_t n, int h, int w,
                                  int64_t src_stride_n, int64_t src_stride_h, int64_t dst_stride_n,
                                  int64_t dst_stride_h, const float* wgx, int kgx, const float* wgy, int kgy, int gh,
                                  int gw, double clip_limit, const float* wux, int kux, const float* wuy, int kuy,
                                  int border, float lo, float hi, int stages, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    const Image s{src, src_dtype, src_stride_n, src_stride_h}, d{dst, dst_dtype, dst_stride_n, dst_stride_h};
    int rc = check_planes(s, d, n, h, w);
    if (rc) return rc;
    rc = check_dtypes(src_dtype, dst_dtype, lo, hi);
    if (rc) return rc;
    rc = check_taps(wgx, kgx, wgy, kgy, border, h, w);
    if (rc) return rc;
    rc = check_taps(wux, kux, wuy, kuy, border, h, w);
    if (rc) return rc;
    ClaheGeom g;
    rc = make_clahe_geom(h, w, gh, gw, MIE_CLAHE_KORNIA, &g);
    if (rc) return rc;
    if (stages & ~(MIE_CHAIN_ALL | MIE_CHAIN_PREFER_MARCH | MIE_CHAIN_PREFER_TILES)) return MIE_E_UNSUPPORTED;
    const int hints = stages & (MIE_CHAIN_PREFER_MARCH | MIE_CHAIN_PREFER_TILES);
    stages &= MIE_CHAIN_ALL;
    if (stages < MIE_CHAIN_STAGE_A) return MIE_E_UNSUPPORTED;
    if (n == 0) return MIE_OK;
    if (!workspace) return MIE_E_NULL;
    // chain_a stores 32-bit index words, chain_b loads LUTs as uint4 and cell tables as uint2: the carve-up below
    // keeps every piece 256-byte aligned only if the workspace itself is
    if ((uintptr_t)workspace % 256) return MIE_E_ALIGN;
    if (workspace_bytes < mie_chain_workspace_bytes(n, h, w, gh, gw)) return MIE_E_WORKSPACE;
    if (n * (int64_t)gh * gw > 2147483647LL) return MIE_E_SHAPE;

    uint8_t* luts = (uint8_t*)workspace;
    uint8_t* plane = luts + (size_t)n * gh * gw * kBins;  // 256-byte aligned when workspace is

    int lut_cap = 0;
    if (!fused_ok(g, kgx, kgy, kux, kuy, border, &lut_cap)) {
        if (stages != MIE_CHAIN_ALL) return MIE_E_UNSUPPORTED;
        float* f = (float*)plane;
        const int64_t fsn = (int64_t)h * w, fsh = w;
        rc = gauss_impl(src, f, src_dtype, MIE_F32, n, h, w, src_stride_n, src_stride_h, fsn, fsh, wgx, kgx, wgy, kgy,
                        border, lo, hi, 0, false, st);
        if (rc) return rc;
        rc = clahe_luts_impl(f, MIE_F32, n, h, w, fsn, fsh, gh, gw, clip_limit, MIE_CLAHE_KORNIA, 0.f, 1.f, nullptr,
                             luts, st);
        if (rc) return rc;
        rc = clahe_apply_impl(f, f, MIE_F32, MIE_F32, n, h, w, fsn, fsh, fsn, fsh, gh, gw, MIE_CLAHE_KORNIA, 0.f, 1.f,
                              luts, st);
        if (rc) return rc;
        return gauss_impl(f, dst, MIE_F32, dst_dtype, n, h, w, fsn, fsh, dst_stride_n, dst_stride_h, wux, kux, wuy,
                          kuy, border, lo, hi, 1, true, st);
    }

    Taps tgx, tgy, tux, tuy;
    fill_taps(tgx, wgx, kgx); fill_taps(tgy, wgy, kgy); fill_taps(tux, wux, kux); fill_taps(tuy, wuy, kuy);

    ChainAArgs a;
    a.src = src; a.ssn = src_stride_n; a.ssh = src_stride_h; a.idx = plane; a.luts = luts; a.g = g;
    a.lp = make_lut_params(g, clip_limit, MIE_CLAHE_KORNIA);
    a.border = border; a.lo = lo; a.rg = hi - lo;
    WinCvt cv = {};
    const int mode = fast_chain_mode(g, s, d, kgx, kux, border, lo, hi, &cv);
    const bool fast = mode >= 0;
    const WinCvt* win = mode == 1 ? &cv : nullptr;   // integer value_range window (window.cuh)
    ChainBArgs b;
    b.idx = plane; b.luts = luts; b.dst = dst; b.dsn = dst_stride_n; b.dsh = dst_stride_h; b.g = g;
    b.tiles_x = ceil_div(w, kTile); b.tiles_y = ceil_div(h, kTile); b.border = border; b.max_lut_tiles = lut_cap;
    b.lo = lo; b.rg = hi - lo;
    if (n * (int64_t)b.tiles_x * b.tiles_y > 2147483647LL) return MIE_E_SHAPE;
    // The marching kernels run one block per 64-row band: unbeatable once the bands fill the machine, but a
    // single 512x512 slice is 8 blocks walking 72 rows each (30.8 us for the step against 12.3 us with one
    // block per 64x64 tile).  Measured crossover on B200: ~24 slices of 512x512 (benchmarks/
    // chain_latency_probe.py), i.e. about 1.5 band-blocks per SM.
    const bool enough_bands = n * (int64_t)g.gh >= 222;
    const bool march = fast && march_chain_ok(g, kgx, kux) &&
                       !(hints & MIE_CHAIN_PREFER_TILES) && (enough_bands || (hints & MIE_CHAIN_PREFER_MARCH)) &&
                       (int64_t)h * src_stride_h * 4 < (1LL << 31);  // 32-bit source-row offsets
    if (fast) {
        if (stages & MIE_CHAIN_STAGE_A) {
            rc = march ? launch_chain_a_march(a, src_dtype, tgx, tgy, n, st, win)
                       : launch_chain_a_fast(a, src_dtype, tgx, tgy, kgx / 2, n, st, win);
            if (rc) return rc;
        }
        if (!(stages & MIE_CHAIN_STAGE_B)) return MIE_OK;
        if (kux == 9) {
            // cell tables live behind the index plane (always inside the workspace bound:
            // 2 (gh+1)(gw+1) KB <= 3 bytes per pixel for 64x64-pixel tiles)
            size_t off = ((size_t)n * gh * gw * kBins + (size_t)n * h * w + 255) & ~(size_t)255;
            if (off + chain_cells_bytes(n, gh, gw) > workspace_bytes) return MIE_E_WORKSPACE;
            return march ? launch_chain_b_march(b, dst_dtype, (uint8_t*)workspace + off, tux, tuy, n, st, win)
                         : launch_chain_b_fast(b, dst_dtype, (uint8_t*)workspace + off, tux, tuy, n, st, win);
        }
        stages = MIE_CHAIN_STAGE_B;  // other unsharp sizes: generic chain_b on the same index plane / LUTs
    }
#define MIE_CHAIN_A(R_)                                                                          \
    MIE_DISPATCH_SRC(src_dtype, rc = (launch_a<SrcT, R_>(a, tgx, tgy, n, st)))
    if (stages & MIE_CHAIN_STAGE_A) {
        switch (kgx / 2) {
            case 1: MIE_CHAIN_A(1); break;
            case 2: MIE_CHAIN_A(2); break;
            case 3: MIE_CHAIN_A(3); break;
            default: MIE_CHAIN_A(4); break;
        }
    }
#undef MIE_CHAIN_A
    if (rc || !(stages & MIE_CHAIN_STAGE_B)) return rc;
#define MIE_CHAIN_B(R_)                                                                          \
    switch (dst_dtype) {                                                                         \
        case MIE_U8: rc = launch_b<uint8_t, R_>(b, tux, tuy, n, lut_cap, st); break;             \
        case MIE_U16: rc = launch_b<uint16_t, R_>(b, tux, tuy, n, lut_cap, st); break;           \
        case MIE_I16: rc = launch_b<int16_t, R_>(b, tux, tuy, n, lut_cap, st); break;            \
        default: rc = launch_b<float, R_>(b, tux, tuy, n, lut_cap, st); break;                   \
    }
    switch (kux / 2) {
        case 1: MIE_CHAIN_B(1); break;
        case 2: MIE_CHAIN_B(2); break;
        case 3: MIE_CHAIN_B(3); break;
        default: MIE_CHAIN_B(4); break;
    }
#undef MIE_CHAIN_B
    return rc;
}

}  // extern "C"
