// chain_fast.cu — tuned kernels of the fused Gaussian -> CLAHE -> unsharp chain for
// 64x64-pixel CLAHE tiles (see chain_fast.cuh for the instruction-level tricks and
// chain.cu for the algorithm and the generic kernels these two must equal bit for bit).
#include "window.cuh"

namespace mie {

// ================================================================ chain_a (fast)
// One block (9 warps) per CLAHE tile:
//   row pass   : 72 rows x 4 segments = one item per thread; a thread loads 24 pixels of one row
//                with 64/128-bit loads, converts them, forms 16 horizontal sums -> s_mid;
//   col pass   : warps 0-7, 4 columns x 4 rows per thread out of s_mid;
//   epilogue   : lookup index -> 32-bit stores into the index plane; histogram bin ->
//                ATOMS.POPC.INC into the block histogram;
//   LUT        : warp 8 clips / redistributes / scans (8 bins per lane).
template <typename SrcT, int R, bool WIN>
__global__ void __launch_bounds__(kFastThreads)
chain_a_fast_kernel(ChainAArgs a, Taps wx, Taps wy, WinCvt cv) {
    constexpr int ROWS = kTile + 2 * R;
    // default-range integer pixels: blurred values are >= 0 and finite; windows (WIN) take the float rules
    constexpr bool NN = !(sizeof(SrcT) == 4) && !WIN;
    __shared__ __align__(16) float s_mid[ROWS * kPMa];
    __shared__ __align__(16) int s_hist[kBins + 8];  // [256] = dummy slot for ignored pixels

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < kBins + 8) s_hist[tid] = 0;

    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % a.g.gw), ty = (int)((tile / a.g.gw) % a.g.gh);
    const int64_t n = tile / ((int64_t)a.g.gw * a.g.gh);
    const int tx0 = tx * kTile, ty0 = ty * kTile;
    const int h = a.g.h, w = a.g.w;
    const SrcT* plane = (const SrcT*)a.src + n * a.ssn;

    // ---- horizontal pass, straight from global memory
    for (int i = tid; i < ROWS * 4; i += kFastThreads) {
        const int s = i & 3, r = i >> 2;
        const int sy = border_index(ty0 - R + r, h, a.border);
        float x[24];
        if (sy < 0) {
#pragma unroll
            for (int k = 0; k < 24; ++k) x[k] = 0.0f;
        } else {
            load_row24_win<SrcT, WIN>(plane + (int64_t)sy * a.ssh, tx0 + 16 * s, w, a.border, x, cv);
        }
        float* mrow = s_mid + r * kPMa + 8 * s;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float acc = __fmul_rn(wx.w[0], x[4 * k + j + 4 - R]);
#pragma unroll
                for (int t = 1; t <= 2 * R; ++t) acc = __fmaf_rn(wx.w[t], x[4 * k + j + 4 - R + t], acc);
                o[j] = acc;
            }
            // quad 4s+k: even quads at word 4*(2s + k/2), odd quads at 48 + 4*(2s + k/2)
            *reinterpret_cast<float4*>(mrow + ((k & 1) ? 48 : 0) + 4 * (k >> 1)) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();

    // ---- vertical pass + epilogue (warps 0..7)
    if (warp < 8) {
        const int q = tid & 15, rb = tid >> 4;
        const int qoff = quad_off(q);
        float4 win[4 + 2 * R];
#pragma unroll
        for (int k = 0; k < 4 + 2 * R; ++k)
            win[k] = *reinterpret_cast<const float4*>(s_mid + (rb * 4 + k) * kPMa + qoff);
        uint8_t* ip = a.idx + n * (int64_t)h * w + (int64_t)(ty0 + rb * 4) * w + tx0 + q * 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float g[4];
            col4_f32x2<R>(win, j, wy, g);
            *reinterpret_cast<uint32_t*>(ip + (int64_t)j * w) =
                pack_low_bytes(fast_idx_bits<NN>(g[0]), fast_idx_bits<NN>(g[1]), fast_idx_bits<NN>(g[2]),
                               fast_idx_bits<NN>(g[3]));
#pragma unroll
            for (int k = 0; k < 4; ++k) hist_add_nobranch(s_hist, fast_bin<NN>(g[k]));
        }
    }
    __syncthreads();
    if (warp == 8) warp_build_lut(s_hist, a.lp, a.luts + tile * kBins, lane);
}

// ================================================================ cell tables
// Interpolation cell (cy, cx), cy in [0, gh], cx in [0, gw], is the region between the centres of
// tiles (cy-1, cx-1) .. (cy, cx) (clamped at the image border).  For every grey level the cell table
// holds what the blend needs, ready to use: (tl - tr, tr, bl - br, br) as four half-width floats (see
// cell_word), 8 bytes per grey level, 2 KB per cell.  chain_b then needs
// ONE 64-bit shared-memory load per pixel and no integer unpacking.  A tiny launch between chain_a
// and chain_b.
template <int kMaxGw>   // 0: any grid width, serial walk
__global__ void __launch_bounds__(256)
chain_pack_cells_kernel(const uint8_t* __restrict__ luts, uint2* __restrict__ cells, int gh, int gw) {
    // one block per (image, cell row); thread = grey level; walks the gw + 1 cells of the row, carrying
    // the right-hand LUT entries of one cell over as the left-hand entries of the next
    const int cy = blockIdx.x;
    const int64_t n = blockIdx.y;
    const int jt = max(cy - 1, 0), jb = min(cy, gh - 1);
    const uint8_t* top = luts + (n * gh + jt) * (int64_t)gw * kBins + threadIdx.x;
    const uint8_t* bot = luts + (n * gh + jb) * (int64_t)gw * kBins + threadIdx.x;
    uint2* out = cells + (n * (gh + 1) + cy) * (int64_t)(gw + 1) * kBins + threadIdx.x;
    // all LUT bytes of the two tile rows first (independent loads in flight together: the serial version, one
    // dependent round trip per cell, was latency bound at 11.9 us for the config-2 batch), then the packing
    if constexpr (kMaxGw == 0) {
        int tl = top[0], bl = bot[0];
        for (int cx = 0; cx <= gw; ++cx) {
            const int ir = min(cx, gw - 1);
            const int tr = top[ir * kBins], br = bot[ir * kBins];
            uint2 e;
            e.x = cell_word(tl - tr, tr);
            e.y = cell_word(bl - br, br);
            out[cx * kBins] = e;
            tl = tr; bl = br;
        }
        return;
    }
    constexpr int N = kMaxGw > 0 ? kMaxGw : 1;
    uint8_t t[N], b[N];
#pragma unroll
    for (int i = 0; i < N; ++i)
        if (i < gw) { t[i] = __ldg(top + i * kBins); b[i] = __ldg(bot + i * kBins); }
    int tl = t[0], bl = b[0];
#pragma unroll
    for (int cx = 0; cx <= N; ++cx) {
        if (cx <= gw) {
            // right-hand tile of cell cx is tile min(cx, gw - 1): at cx == gw it is the carried-over left-hand tile
            const int tr = (cx < N && cx < gw) ? t[cx < N ? cx : 0] : tl;
            const int br = (cx < N && cx < gw) ? b[cx < N ? cx : 0] : bl;
            uint2 e;
            e.x = cell_word(tl - tr, tr);
            e.y = cell_word(bl - br, br);
            out[cx * kBins] = e;
            tl = tr; bl = br;
        }
    }
}

// ================================================================ chain_b (fast, 9-tap unsharp)
// One block per 64x64 output tile (aligned with the CLAHE tile grid, so the haloed 72x72 region
// touches exactly 2x2 interpolation cells):
//   tables : the block's four 1 KB cell tables -> shared memory (one 16-byte copy per thread);
//   C pass : CLAHE output C for every haloed pixel -> s_in;
//   row / col pass, epilogue: C + (C - blur(C)) -> quantise -> 64-bit stores.

template <typename DstT, bool WIN>
__global__ void __launch_bounds__(kFastThreads)
chain_b_fast_kernel(ChainBArgs a, const uint2* __restrict__ cells, AxisWeights aw, Taps wx, Taps wy, WinCvt cv) {
    constexpr int R = 4, E = kTile + 2 * R, PIN = TileSmem<R>::pin;
    extern __shared__ __align__(16) float smem[];
    float* s_in = smem;                                        // E x PIN
    float* s_mid = s_in + E * PIN;                             // E x kPMid (written after the C pass)
    uint2* s_cell = reinterpret_cast<uint2*>(s_mid);           // 4 cells x 256 entries: dead once the C pass
                                                               // is over, so it shares s_mid's storage
    float* s_w = s_mid + E * kPMid;                            // E weights

    const int tid = threadIdx.x;
    const int64_t tile = blockIdx.x;
    const int tx = (int)(tile % a.tiles_x), ty = (int)((tile / a.tiles_x) % a.tiles_y);
    const int64_t n = tile / ((int64_t)a.tiles_x * a.tiles_y);
    const int tx0 = tx * kTile, ty0 = ty * kTile;
    const int h = a.g.h, w = a.g.w, gh = a.g.gh, gw = a.g.gw;

    // ---- tables: cell (a, b) of this tile = global cell (ty + a, tx + b)
    if (tid < 256) {
        const int c = tid >> 6, part = tid & 63;  // 64 threads x 2 x 16 B per 2 KB cell table
        const uint4* src = reinterpret_cast<const uint4*>(
            cells + ((n * (gh + 1) + ty + (c >> 1)) * (int64_t)(gw + 1) + tx + (c & 1)) * kBins);
        uint4* dst4 = reinterpret_cast<uint4*>(s_cell + c * kBins);
        dst4[part] = __ldg(src + part);
        dst4[part + 64] = __ldg(src + part + 64);
    } else if (tid - 256 < E / 4) {
        const int k = (tid - 256) * 4;
        *reinterpret_cast<float4*>(s_w + k) = make_float4(aw.w[k], aw.w[k + 1], aw.w[k + 2], aw.w[k + 3]);
    }
    // ---- CLAHE output of the haloed tile: item = (row r, 8-column chunk u); chunk u = image
    //      columns gx0 .. gx0+7 with gx0 = tx0 - 4 + 8u (4-byte aligned).  The index words of the
    //      next item are fetched while the current one is computed (and the first fetch overlaps the
    //      table loads above), which hides the global-load latency of this pass.
    const uint8_t* iplane = a.idx + n * (int64_t)h * w;
    struct IdxChunk { uint32_t w0, w1; int sy; bool z0, z1; };
    auto fetch = [&](int i) {
        IdxChunk c;
        const int u = i % 9, r = i / 9;
        c.sy = border_index(ty0 - R + r, h, a.border);
        c.w0 = c.w1 = 0u; c.z0 = c.z1 = false;
        if (c.sy >= 0) {
            const uint8_t* irow = iplane + (int64_t)c.sy * w;
            const int gx0 = tx0 - 4 + 8 * u;
            if (gx0 < 0) {  // columns -4..-1 mirror onto 4,3,2,1
                c.w1 = __ldg(reinterpret_cast<const uint32_t*>(irow));
                if (a.border == MIE_BORDER_REFLECT)
                    c.w0 = __byte_perm(c.w1, __ldg(reinterpret_cast<const uint32_t*>(irow + 4)), 0x1234);
                else if (a.border == MIE_BORDER_REPLICATE) c.w0 = __byte_perm(c.w1, 0u, 0x0000);
                else c.z0 = true;
            } else if (gx0 + 8 > w) {  // columns w..w+3 mirror onto w-2..w-5
                c.w0 = __ldg(reinterpret_cast<const uint32_t*>(irow + gx0));
                if (a.border == MIE_BORDER_REFLECT)
                    c.w1 = __byte_perm(c.w0, __ldg(reinterpret_cast<const uint32_t*>(irow + gx0 - 4)), 0x7012);
                else if (a.border == MIE_BORDER_REPLICATE) c.w1 = __byte_perm(c.w0, 0u, 0x3333);
                else c.z1 = true;
            } else {
                c.w0 = __ldg(reinterpret_cast<const uint32_t*>(irow + gx0));
                c.w1 = __ldg(reinterpret_cast<const uint32_t*>(irow + gx0 + 4));
            }
        }
        return c;
    };
    IdxChunk cur = fetch(tid);
    __syncthreads();

    for (int i = tid; i < E * 9; i += kFastThreads) {
        IdxChunk nxt = cur;
        if (i + kFastThreads < E * 9) nxt = fetch(i + kFastThreads);
        const int u = i % 9, r = i / 9;
        float4 lo4 = make_float4(0.f, 0.f, 0.f, 0.f), hi4 = lo4;
        if (cur.sy >= 0) {
            const float wyv = s_w[r];
            // cell number (row cell * 2 + column cell) goes into byte 1 of the table index; the
            // column cell flips between haloed columns 35 and 36 (source column tx0 + 32)
            const uint32_t ca = (cur.sy >= ty0 + kTile / 2) ? 2u : 0u;
            const uint32_t cL = ca + (u >= 5 ? 1u : 0u), cH = ca + (u >= 4 ? 1u : 0u);
            const uint32_t w0 = cur.w0, w1 = cur.w1;
            const float4 wa = *reinterpret_cast<const float4*>(s_w + 8 * u);
            const float4 wb = *reinterpret_cast<const float4*>(s_w + 8 * u + 4);
            lo4.x = clahe_px(s_cell[__byte_perm(w0, cL, 0x7640)], wa.x, wyv);
            lo4.y = clahe_px(s_cell[__byte_perm(w0, cL, 0x7641)], wa.y, wyv);
            lo4.z = clahe_px(s_cell[__byte_perm(w0, cL, 0x7642)], wa.z, wyv);
            lo4.w = clahe_px(s_cell[__byte_perm(w0, cL, 0x7643)], wa.w, wyv);
            hi4.x = clahe_px(s_cell[__byte_perm(w1, cH, 0x7640)], wb.x, wyv);
            hi4.y = clahe_px(s_cell[__byte_perm(w1, cH, 0x7641)], wb.y, wyv);
            hi4.z = clahe_px(s_cell[__byte_perm(w1, cH, 0x7642)], wb.z, wyv);
            hi4.w = clahe_px(s_cell[__byte_perm(w1, cH, 0x7643)], wb.w, wyv);
            if (cur.z0) lo4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (cur.z1) hi4 = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float* dstp = s_in + r * PIN + 8 * u;
        *reinterpret_cast<float4*>(dstp) = lo4;
        *reinterpret_cast<float4*>(dstp + 4) = hi4;
        cur = nxt;
    }
    __syncthreads();

    // ---- horizontal pass out of s_in (lanes on consecutive rows: conflict-free LDS.128 / STS.128)
    for (int i = tid; i < E * 8; i += kFastThreads) {
        const int r = i % E, s = i / E;
        const float4* p = reinterpret_cast<const float4*>(s_in + r * PIN + s * 8);
        float win[16];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const float4 t = p[v];
            win[4 * v] = t.x; win[4 * v + 1] = t.y; win[4 * v + 2] = t.z; win[4 * v + 3] = t.w;
        }
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float acc = __fmul_rn(wx.w[0], win[j]);
#pragma unroll
            for (int t = 1; t <= 2 * R; ++t) acc = __fmaf_rn(wx.w[t], win[j + t], acc);
            o[j] = acc;
        }
        float4* q = reinterpret_cast<float4*>(s_mid + r * kPMid + s * 8);
        q[0] = make_float4(o[0], o[1], o[2], o[3]);
        q[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
    __syncthreads();

    // ---- vertical pass + unsharp + quantise (warps 0..7)
    if (tid < 256) {
        const int q = tid & 15, rb = tid >> 4;
        float4 win[4 + 2 * R];
#pragma unroll
        for (int k = 0; k < 4 + 2 * R; ++k)
            win[k] = *reinterpret_cast<const float4*>(s_mid + (rb * 4 + k) * kPMid + q * 4);
        DstT* op = (DstT*)a.dst + n * a.dsn + (int64_t)(ty0 + rb * 4) * a.dsh + tx0 + q * 4;
        const float* cp = s_in + (rb * 4 + R) * PIN + q * 4 + R;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float g[4];
            col4_f32x2<R>(win, j, wy, g);
            const float4 c = *reinterpret_cast<const float4*>(cp + j * PIN);
            float y[4];
            y[0] = __fadd_rn(c.x, __fsub_rn(c.x, g[0])); y[1] = __fadd_rn(c.y, __fsub_rn(c.y, g[1]));
            y[2] = __fadd_rn(c.z, __fsub_rn(c.z, g[2])); y[3] = __fadd_rn(c.w, __fsub_rn(c.w, g[3]));
            PixIO<DstT, WIN>::store4(op + (int64_t)j * a.dsh, y, cv);
        }
    }
}

// ================================================================ host side
int fast_chain_mode(const ClaheGeom& g, const Image& s, const Image& d, int kg, int ku, int border, float lo, float hi,
                    WinCvt* cv) {
    if (g.th != kTile || g.tw != kTile || g.hp != g.h || g.wp != g.w) return -1;
    if (kg < 3 || kg > 9 || ku < 3 || ku > 9) return -1;
    if (border == MIE_BORDER_CIRCULAR || border == MIE_BORDER_SYMMETRIC) return -1;
    if (!s.aligned(16) || !d.aligned(16)) return -1;   // 16-byte aligned rows for the vector loads / stores
    return range_mode(s.dtype, lo, hi, cv);
}

template <typename SrcT, bool WIN>
static int launch_a_t(const ChainAArgs& a, const Taps& wx, const Taps& wy, int R, unsigned blocks, cudaStream_t st,
                      const WinCvt& cv) {
    switch (R) {
        case 1: chain_a_fast_kernel<SrcT, 1, WIN><<<blocks, kFastThreads, 0, st>>>(a, wx, wy, cv); break;
        case 2: chain_a_fast_kernel<SrcT, 2, WIN><<<blocks, kFastThreads, 0, st>>>(a, wx, wy, cv); break;
        case 3: chain_a_fast_kernel<SrcT, 3, WIN><<<blocks, kFastThreads, 0, st>>>(a, wx, wy, cv); break;
        default: chain_a_fast_kernel<SrcT, 4, WIN><<<blocks, kFastThreads, 0, st>>>(a, wx, wy, cv); break;
    }
    return check_launch();
}

int launch_chain_a_fast(const ChainAArgs& a, int sd, const Taps& wx, const Taps& wy, int R, int64_t n,
                        cudaStream_t st, const WinCvt* win) {
    const unsigned blocks = (unsigned)(n * a.g.gh * a.g.gw);
    const WinCvt none = {};
    if (win) { MIE_DISPATCH_SRC(sd, return (launch_a_t<SrcT, true>(a, wx, wy, R, blocks, st, *win))); }
    else { MIE_DISPATCH_SRC(sd, return (launch_a_t<SrcT, false>(a, wx, wy, R, blocks, st, none))); }
    return MIE_OK;
}

int launch_pack_cells(const uint8_t* luts, void* cells, int64_t n, int gh, int gw, cudaStream_t st) {
    if (n > 65535) return MIE_E_SHAPE;
    dim3 pgrid((unsigned)(gh + 1), (unsigned)n);
    if (gw <= 8) chain_pack_cells_kernel<8><<<pgrid, 256, 0, st>>>(luts, (uint2*)cells, gh, gw);
    else if (gw <= 16) chain_pack_cells_kernel<16><<<pgrid, 256, 0, st>>>(luts, (uint2*)cells, gh, gw);
    else if (gw <= 32) chain_pack_cells_kernel<32><<<pgrid, 256, 0, st>>>(luts, (uint2*)cells, gh, gw);
    else chain_pack_cells_kernel<0><<<pgrid, 256, 0, st>>>(luts, (uint2*)cells, gh, gw);
    return check_launch();
}

size_t chain_cells_bytes(int64_t n, int gh, int gw) { return (size_t)n * (gh + 1) * (gw + 1) * kBins * 8; }

template <typename DstT, bool WIN>
static int launch_b_t(const ChainBArgs& b, const uint2* cells, const AxisWeights& aw, const Taps& wx,
                      const Taps& wy, unsigned blocks, cudaStream_t st, const WinCvt& cv) {
    constexpr int E = kTile + 8;
    constexpr size_t smem = (size_t)(E * TileSmem<4>::pin + E * kPMid + E) * 4;
    static_assert(E * kPMid * 4 >= 4 * kBins * 8, "cell tables must fit in the s_mid region");
    MIE_ENSURE_SMEM((chain_b_fast_kernel<DstT, WIN>), smem);
    chain_b_fast_kernel<DstT, WIN><<<blocks, kFastThreads, smem, st>>>(b, cells, aw, wx, wy, cv);
    return check_launch();
}

// Runs the cell-packing launch and the tuned chain_b (9-tap unsharp only).  `cells` must hold
// chain_cells_bytes(n, gh, gw) bytes.
int launch_chain_b_fast(const ChainBArgs& b, int dd, void* cells_raw, const Taps& wx, const Taps& wy, int64_t n,
                        cudaStream_t st, const WinCvt* win) {
    uint2* cells = (uint2*)cells_raw;
    int rc = launch_pack_cells(b.luts, cells, n, b.g.gh, b.g.gw, st);
    if (rc) return rc;
    AxisWeights aw;
    fill_axis_weights(aw);
    const unsigned blocks = (unsigned)(n * b.tiles_x * b.tiles_y);
    const WinCvt none = {};
    if (win) { MIE_DISPATCH_SRC(dd, return (launch_b_t<SrcT, true>(b, cells, aw, wx, wy, blocks, st, *win))); }
    else { MIE_DISPATCH_SRC(dd, return (launch_b_t<SrcT, false>(b, cells, aw, wx, wy, blocks, st, none))); }
    return MIE_OK;
}

}  // namespace mie
