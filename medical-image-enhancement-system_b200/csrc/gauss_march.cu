// gauss_march.cu — marching Gaussian blur / unsharp mask for the common geometry: square 9-tap kernel,
// image width a multiple of 128 (<= 1024), height a multiple of 64, default value range, 16-byte aligned
// rows.  Same arithmetic, bit for bit, as gauss.cu (and as the two blur stages of the fused chain); the
// schedule is the one of chain_march.cu: full-width bands of 64 rows walked two rows per step, source
// rows streamed through a bulk-copy (TMA) ring, row-pair buffers in shared memory, the vertical pass out
// of a register ring, packed fma.rn.f32x2 in both passes.  For unsharp the centre pixels of the rows that
// become complete are re-read from the row-pair buffers of four steps earlier.

#include "march.cuh"
#include "window.cuh"

namespace mie {

struct GaussMarchArgs {
    const void* src;
    void* dst;
    int64_t ssn, ssh, dsn, dsh;
    int h, w;
};

// WIN: integer value_range window (csrc/window.cuh) — the divide-free windowed conversion on the way in and the
// windowed quantisation on the way out; everything in between is the same fp32 arithmetic.
template <typename SrcT, typename DstT, int BORDER, bool UNSHARP, bool WIN, int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB)
gauss_march_kernel(GaussMarchArgs a, Taps wx, Taps wy, WinCvt cv) {
    typedef typename Fast<SrcT>::raw4 raw4;
    extern __shared__ __align__(16) float smem[];
    const int W = a.w, T = blockDim.x, h = a.h;
    const int pbuf = pairbuf_floats(T);
    float* s_buf = smem;                                             // 4 pair buffers
    int* s_off = reinterpret_cast<int*>(smem + 4 * pbuf);            // kMOffRows
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_off + kMOffRows);
    float* s_raw = reinterpret_cast<float*>(s_bar + kRawBars);       // kRawRows source rows (raw pixels)

    const int tid = threadIdx.x, warp = tid >> 5, nwarps = T >> 5;
    const int bands = h / kTile;
    const int ty = (int)(blockIdx.x % bands);
    const int64_t n = blockIdx.x / bands;
    const int ty0 = ty * kTile;
    fill_row_offsets<BORDER>(s_off, ty0, h, (int)a.ssh * (int)sizeof(SrcT), tid, T);
    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < kRawBars; ++b) mbar_init((uint32_t)__cvta_generic_to_shared(s_bar + b), 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const bool first_warp = warp == 0, last_warp = warp == nwarps - 1;
    const int row_bytes = W * (int)sizeof(SrcT);
    const uint32_t ring32 = (uint32_t)__cvta_generic_to_shared(s_raw);
    const uint32_t bar32 = (uint32_t)__cvta_generic_to_shared(s_bar);
    const char* plane0 = reinterpret_cast<const char*>((const SrcT*)a.src + n * a.ssn);
    // the producer is the first lane of warp 1 when there is one: warps 0 and nwarps-1 already carry the
    // image-border halo work, and every warp waits for the slowest one at the per-step barrier
    const int producer = nwarps > 2 ? 32 : 0;
    auto issue_batch = [&](const int b) {  // producer thread only
        const int4 o = *reinterpret_cast<const int4*>(s_off + kRawBatch * b);
        const int off[4] = {o.x, o.y, o.z, o.w};
        const uint32_t mb = bar32 + 8 * (b % kRawBars);
        int valid = 0;
#pragma unroll
        for (int j = 0; j < kRawBatch; ++j) valid += (BORDER != MIE_BORDER_CONSTANT || off[j] >= 0) ? 1 : 0;
        mbar_expect_tx(mb, (uint32_t)(valid * row_bytes));
#pragma unroll
        for (int j = 0; j < kRawBatch; ++j)
            if (BORDER != MIE_BORDER_CONSTANT || off[j] >= 0)
                bulk_g2s(ring32 + (uint32_t)(((kRawBatch * b + j) % kRawRows) * row_bytes), plane0 + (unsigned)off[j],
                         (uint32_t)row_bytes, mb);
    };
    if (tid == producer) {
#pragma unroll
        for (int b = 0; b < kRawBars; ++b) issue_batch(b);
    }
    f32x2 ring[kMRing][2];
    const char* my_raw = reinterpret_cast<const char*>(s_raw) + 4 * tid * (int)sizeof(SrcT);
    // -> packed (row 2p, row 2p + 1) pairs of the thread's four columns (the layout of the pair buffer); 16-bit pixels in
    // their default range are converted packed as well (chain_fast.cuh: cvt_pair4)
    uint32_t exp_magic = 0u;
    if constexpr (sizeof(SrcT) == 2 && !WIN) exp_magic = Fast<SrcT>::exp_magic();
    auto convert = [&](const int p, const int rslot, f32x2* xp) {
        if (p % 2 == 0) mbar_wait(bar32 + 8 * ((p / 2) % kRawBars), (uint32_t)((p / 2 / kRawBars) & 1));
        const raw4 r0 = *reinterpret_cast<const raw4*>(my_raw + (rslot % kRawRows) * row_bytes);
        const raw4 r1 = *reinterpret_cast<const raw4*>(my_raw + ((rslot + 1) % kRawRows) * row_bytes);
        if constexpr (sizeof(SrcT) == 2 && !WIN) {
            Fast<SrcT>::cvt_pair4(r0, r1, xp, exp_magic);
            if (BORDER == MIE_BORDER_CONSTANT) {
                const bool z0 = s_off[2 * p] < 0, z1 = s_off[2 * p + 1] < 0;
                if (z0 || z1) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float lo_, hi_;
                        f2_unpack(xp[k], lo_, hi_);
                        xp[k] = f2_pack(z0 ? 0.0f : lo_, z1 ? 0.0f : hi_);
                    }
                }
            }
        } else {
            float x0[4], x1[4];
            PixIO<SrcT, WIN>::cvt_raw4(r0, x0, cv);
            PixIO<SrcT, WIN>::cvt_raw4(r1, x1, cv);
            if (BORDER == MIE_BORDER_CONSTANT) {
                if (s_off[2 * p] < 0) x0[0] = x0[1] = x0[2] = x0[3] = 0.0f;
                if (s_off[2 * p + 1] < 0) x1[0] = x1[1] = x1[2] = x1[3] = 0.0f;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) xp[k] = f2_pack(x0[k], x1[k]);
        }
    };
    auto refill = [&](const int p) {
        const int b = (p - 1) / 2 + kRawBars;
        if (tid == producer && b < kMRows / kRawBatch) issue_batch(b);
    };
    DstT* op = (DstT*)a.dst + n * a.dsn + (int64_t)ty0 * a.dsh + 4 * tid;
    const int dsh = (int)a.dsh;

#pragma unroll
    for (int p = 0; p < kMPro; ++p) {
        f32x2 xp[4];
        convert(p, 2 * p, xp);
        float* buf = s_buf + (p % 4) * pbuf;
        pair_store_packed<BORDER>(buf, T, tid, first_warp, last_warp, xp);
        __syncthreads();
        if (p % 2 == 1) refill(p);
        pair_row_pass(buf, T, tid, wx, ring, 2 * p, xp);
    }
    for (int p0 = kMPro; p0 < kMPairs; p0 += kMUnroll) {
#pragma unroll
        for (int q = 0; q < kMUnroll; ++q) {
            const int p = p0 + q;
            f32x2 xp[4];
            convert(p, 2 * kMPro + 2 * q, xp);
            float* buf = s_buf + (q % 4) * pbuf;
            pair_store_packed<BORDER>(buf, T, tid, first_warp, last_warp, xp);
            __syncthreads();
            if (q % 2 == 1) refill(p);
            pair_row_pass(buf, T, tid, wx, ring, 2 * kMPro + 2 * q, xp);
            float g[4], c0[4], c1[4];
            if (UNSHARP) {  // centre pixels of rows (2p - 8, 2p - 7) + 4 = pair p - 2
                const float* cbuf = s_buf + ((q + 2) % 4) * pbuf;
                const float4 ca = *reinterpret_cast<const float4*>(cbuf + 4 * (tid + 1));
                const float4 cb = *reinterpret_cast<const float4*>(cbuf + 4 * (T + 2) + 4 * (tid + 1));
                c0[0] = ca.x; c0[1] = ca.z; c0[2] = cb.x; c0[3] = cb.z;
                c1[0] = ca.y; c1[1] = ca.w; c1[2] = cb.y; c1[3] = cb.w;
            }
            march_col_pass(ring, 2 * q, wy, g);
            if (UNSHARP) {
#pragma unroll
                for (int k = 0; k < 4; ++k) g[k] = __fadd_rn(c0[k], __fsub_rn(c0[k], g[k]));
            }
            PixIO<DstT, WIN>::store4(op, g, cv);
            op += dsh;
            march_col_pass(ring, 2 * q + 1, wy, g);
            if (UNSHARP) {
#pragma unroll
                for (int k = 0; k < 4; ++k) g[k] = __fadd_rn(c1[k], __fsub_rn(c1[k], g[k]));
            }
            PixIO<DstT, WIN>::store4(op, g, cv);
            op += dsh;
        }
    }
}

// The range mode of window.cuh (0, or 1 with *cv filled in) when the marching kernel covers the request, else -1.
int gauss_march_mode(const Image& s, const Image& d, int h, int w, int kx, int ky, int border, float lo, float hi,
                     WinCvt* cv) {
    if (kernel_policy(MIE_POLICY_GENERIC_GAUSS)) return -1;
    if (kx != 9 || ky != 9) return -1;
    if (w % 128 != 0 || w > 1024 || h % kTile != 0) return -1;
    if (border == MIE_BORDER_CIRCULAR || border == MIE_BORDER_SYMMETRIC) return -1;
    if (d.dtype != s.dtype && d.dtype != MIE_F32) return -1;
    if (!s.aligned(16) || !d.aligned(16)) return -1;
    if ((int64_t)h * s.sh * 4 >= (1LL << 31)) return -1;  // 32-bit source-row offsets
    return range_mode(s.dtype, lo, hi, cv);   // default range, or an integer window the host has verified
}

template <typename SrcT, typename DstT, int BORDER, bool WIN>
static int launch_gm_b(const GaussMarchArgs& a, const Taps& wx, const Taps& wy, int unsharp, unsigned blocks,
                       const WinCvt& cv, cudaStream_t st) {
    const int T = a.w / 4;
    const size_t smem = (size_t)(4 * 8 * (T + 2) + kMOffRows) * 4 + kRawBars * 8 + (size_t)kRawRows * a.w * sizeof(SrcT);
#ifndef MIE_G_MINB
#define MIE_G_MINB 5
#endif
    // W <= 512: 128 threads per block with the registers capped for MIE_G_MINB resident blocks per SM
#define MIE_GM_LAUNCH(U_, MAXT_, MINB_)                                                                        \
    do {                                                                                                       \
        MIE_ENSURE_SMEM((gauss_march_kernel<SrcT, DstT, BORDER, U_, WIN, MAXT_, MINB_>), 100 * 1024);          \
        gauss_march_kernel<SrcT, DstT, BORDER, U_, WIN, MAXT_, MINB_><<<blocks, T, smem, st>>>(a, wx, wy, cv); \
    } while (0)
    if (a.w <= 512) { if (unsharp) MIE_GM_LAUNCH(true, 128, MIE_G_MINB); else MIE_GM_LAUNCH(false, 128, MIE_G_MINB); }
    else { if (unsharp) MIE_GM_LAUNCH(true, 256, 2); else MIE_GM_LAUNCH(false, 256, 2); }
#undef MIE_GM_LAUNCH
    return check_launch();
}

template <typename SrcT, typename DstT, bool WIN>
static int launch_gm(const GaussMarchArgs& a, const Taps& wx, const Taps& wy, int border, int unsharp, unsigned blocks,
                     const WinCvt& cv, cudaStream_t st) {
    switch (border) {
        case MIE_BORDER_REFLECT: return launch_gm_b<SrcT, DstT, MIE_BORDER_REFLECT, WIN>(a, wx, wy, unsharp, blocks, cv, st);
        case MIE_BORDER_REPLICATE: return launch_gm_b<SrcT, DstT, MIE_BORDER_REPLICATE, WIN>(a, wx, wy, unsharp, blocks, cv, st);
        default: return launch_gm_b<SrcT, DstT, MIE_BORDER_CONSTANT, WIN>(a, wx, wy, unsharp, blocks, cv, st);
    }
}

int launch_gauss_march(const Image& s, const Image& d, int64_t n, int h, int w, const Taps& wx, const Taps& wy,
                       int border, int unsharp, int mode, const WinCvt& cv, cudaStream_t st) {
    GaussMarchArgs a;
    a.src = s.p; a.dst = d.out(); a.ssn = s.sn; a.ssh = s.sh; a.dsn = d.sn; a.dsh = d.sh; a.h = h; a.w = w;
    const int64_t blocks = n * (h / kTile);
    if (blocks > 2147483647LL) return MIE_E_SHAPE;
    if (mode == 1) {
        MIE_DISPATCH_SRC_DST(s.dtype, d.dtype, return (launch_gm<SrcT, DstT, true>(a, wx, wy, border, unsharp, (unsigned)blocks, cv, st)));
    } else {
        MIE_DISPATCH_SRC_DST(s.dtype, d.dtype, return (launch_gm<SrcT, DstT, false>(a, wx, wy, border, unsharp, (unsigned)blocks, cv, st)));
    }
    return MIE_OK;
}

}  // namespace mie
