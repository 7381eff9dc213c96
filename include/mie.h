/*
 * mie.h — C ABI of libmie_b200.so: the B200 (sm_100a) enhancement hot path.
 *
 * The reference repository (GregOratOr/medical-image-enhancement-system) ships no
 * code of its own (README.md and configs/__init__.py are 0 bytes); its hot path is
 * the set of third-party functions its dependency list names
 * (reference pyproject.toml:7-18 — kornia>=0.8.2 at :8, scikit-image>=0.26.0 at :12,
 * pins in uv.lock:219-230 and uv.lock:619-650).  Each entry point below therefore
 * cites the upstream function it replaces; there is no reference FFI to copy.
 *
 * Conventions
 *  - Every pointer named src/dst/workspace/luts/hist is a DEVICE pointer on the
 *    current CUDA device; `wx`, `wy`, `wspace` weight arrays are HOST pointers and
 *    are copied into kernel parameters at call time.
 *  - Images are batches of single-channel planes: plane i starts at
 *    base + i*stride_n, row y at + y*stride_h (strides in ELEMENTS), pixels
 *    contiguous within a row.  Multi-channel (B,C,H,W) tensors are passed as
 *    n = B*C planes (all ops here are per-channel).
 *  - dtype codes: MIE_U8, MIE_U16, MIE_I16, MIE_F32.  Integer pixels are mapped
 *    to [0,1] as  x01 = (float(v) - lo) / (hi - lo)  (IEEE fp32 ops, in that
 *    order) and mapped back as  rint(clamp(y,0,1) * (hi - lo)) + lo.  For F32
 *    planes lo/hi are ignored (kornia behaviour: caller supplies [0,1] data).
 *    dst_dtype must equal src_dtype or be MIE_F32.
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); nothing
 *    synchronises; no device memory is allocated or retained by the library.
 *  - Return 0 on success, a negative MIE_E_* for argument errors detected before
 *    launch, or a positive cudaError_t passed through.
 */
#ifndef MIE_H_
#define MIE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIE_ABI_VERSION 1

enum mie_dtype {
    MIE_U8 = 0, MIE_U16 = 1, MIE_I16 = 2, MIE_F32 = 3,
    MIE_F64 = 4   /* OUTPUT dtype of the scikit-image entry points only (skimage returns float64 for integer images) */
};

/* kornia border_type names: 'constant' (zeros), 'reflect' (mirror, edge not
 * repeated = scipy.ndimage 'mirror'), 'replicate' (= scipy 'nearest'), 'circular' (= scipy 'wrap').
 * MIE_BORDER_SYMMETRIC mirrors WITH the edge sample repeated (d c b a | a b c d | d c b a): scipy.ndimage's
 * 'reflect', the mode skimage.filters.unsharp_mask uses; accepted by mie_gaussian2d / mie_unsharp /
 * mie_median2d. */
enum mie_border {
    MIE_BORDER_CONSTANT = 0, MIE_BORDER_REFLECT = 1, MIE_BORDER_REPLICATE = 2, MIE_BORDER_CIRCULAR = 3,
    MIE_BORDER_SYMMETRIC = 4
};

/* CLAHE semantics selector. */
enum mie_clahe_semantics { MIE_CLAHE_KORNIA = 0, MIE_CLAHE_OPENCV = 1 };

enum mie_error {
    MIE_OK = 0,
    MIE_E_NULL = -1,        /* null pointer argument */
    MIE_E_DTYPE = -2,       /* unsupported dtype / dtype combination */
    MIE_E_SHAPE = -3,       /* non-positive or unsupported dimension */
    MIE_E_STRIDE = -4,      /* stride smaller than the row / plane */
    MIE_E_GRID = -5,        /* CLAHE grid entry <= 0 */
    MIE_E_PAD = -6,         /* required padding exceeds the image (kornia ValueError) */
    MIE_E_KERNEL = -7,      /* kernel size even, <= 0 or beyond the supported maximum */
    MIE_E_BORDER = -8,      /* unknown border mode, or halo >= image for reflect */
    MIE_E_WORKSPACE = -9,   /* workspace too small */
    MIE_E_RANGE = -10,      /* hi <= lo for an integer dtype */
    MIE_E_UNSUPPORTED = -11,/* valid request this build does not implement */
    MIE_E_ALIGN = -12,      /* workspace (or a buffer a tuned kernel needs aligned) is not 256-byte aligned */
    MIE_E_NCCL_BASE = -100  /* mie_halo_exchange_z: ncclResult_t r of a failed NCCL call is returned as -100 - r */
};

int mie_abi_version(void);

/* Kernel-selection policy (process-wide; a verification hook, not a tuning knob).  Every operator picks the tuned
 * sm_100a kernel whenever the request's geometry / dtype / alignment allows and a generic kernel otherwise; both
 * compute the same result bit for bit.  A set bit forces the generic variant for that operator although the tuned
 * one applies, so that tests can compare the two on the same input.  Replaces what round 1 read from MIE_*
 * environment variables: nothing in the library calls getenv().  mie_set_kernel_policy returns MIE_E_UNSUPPORTED
 * for unknown bits; call it while no other thread is inside the library. */
enum mie_kernel_policy {
    MIE_POLICY_DEFAULT = 0,
    MIE_POLICY_GENERIC_GAUSS = 1,          /* gauss_tile / gauss_generic kernels instead of the marching kernel */
    MIE_POLICY_GENERIC_CLAHE = 2,          /* per-tile histogram + generic interpolation kernels */
    MIE_POLICY_CLAHE_FLOAT_RULES = 4,      /* tuned CLAHE, but bins / indices from the float conversion, not the integer rules */
    MIE_POLICY_GENERIC_EQUALIZE = 8,
    MIE_POLICY_EQUALIZE_FLOAT_RULES = 16,
    MIE_POLICY_GENERIC_MEDIAN = 32,        /* forgetful-selection tile kernels instead of the packed marching kernels */
    MIE_POLICY_GENERIC_BILATERAL = 64,
    MIE_POLICY_GENERIC_NLM = 128,
    MIE_POLICY_CLAHE16_NO_CLUSTER = 256,   /* 65 536-bin CLAHE: one CTA per tile instead of a 2-CTA cluster */
    MIE_POLICY_CLAHE16_TWO_SWEEP = 512,    /* 65 536-bin CLAHE: the two-sweep kernel of tiles >= 65 536 pixels */
    MIE_POLICY_EQUALIZE_THREE_PASS = 1024, /* equalize: histogram / LUT / apply launches instead of the one-launch cluster kernel */
    MIE_POLICY_BILATERAL_EXACT_EXP = 2048, /* bilateral: the reproducible polynomial 2^t (bit-exact against the oracle) instead of MUFU.EX2 */
    MIE_POLICY_CLAHE16_FULL_LUTS = 4096,   /* 65 536-bin CLAHE: build all 65 536 LUT entries although the batch's largest pixel value is smaller */
    MIE_POLICY_EQUALIZE_SLAB = 8192,       /* equalize: the shared-memory slab (TMA) cluster kernel also for small planes (default: second read through L2) */
    MIE_POLICY_ALL = 16383
};
int mie_set_kernel_policy(unsigned mask);
unsigned mie_get_kernel_policy(void);
const char* mie_error_string(int code);
/* SM count / compute capability of the current device (for grid sizing, tests). */
int mie_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------ Gaussian / unsharp
 * Replaces kornia.filters.gaussian_blur2d(input, kernel_size, sigma, border_type,
 * separable=True) and kornia.filters.unsharp_mask(input, kernel_size, sigma,
 * border_type) (reference pyproject.toml:8; SURVEY.md §8(a) A3/A4).
 * wx (kx taps, horizontal) and wy (ky taps, vertical) are the normalised 1-D
 * weights; kx, ky odd, <= MIE_MAX_TAPS.  Horizontal pass first, then vertical; each
 * pass accumulates acc = w[0]*x[0]; acc = fma(w[i], x[i], acc) in tap order.
 * unsharp: out = x + (x - blur(x)).                                              */
#define MIE_MAX_TAPS 33
int mie_gaussian2d(const void* src, void* dst, int src_dtype, int dst_dtype,
                   int64_t n, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_h,
                   int64_t dst_stride_n, int64_t dst_stride_h,
                   const float* wx, int kx, const float* wy, int ky, int border,
                   float lo, float hi, void* stream);
int mie_unsharp(const void* src, void* dst, int src_dtype, int dst_dtype,
                int64_t n, int h, int w,
                int64_t src_stride_n, int64_t src_stride_h,
                int64_t dst_stride_n, int64_t dst_stride_h,
                const float* wx, int kx, const float* wy, int ky, int border,
                float lo, float hi, void* stream);

/* skimage.filters.unsharp_mask(image, radius, amount) (reference pyproject.toml:12; SURVEY.md §2.2,
 * §8(f) F3): out = x + amount * (x - blur(x)), computed as fma(amount, x - blur, x) (amount == 1 gives
 * mie_unsharp's result bit for bit); clip != 0 clamps the result to [0, 1] before any quantisation
 * (skimage without preserve_range).  skimage's blur is scipy.ndimage.gaussian_filter(sigma = radius,
 * mode = 'reflect' = MIE_BORDER_SYMMETRIC, truncate = 4): taps 2*int(4*radius + 0.5) + 1.            */
int mie_unsharp_amount(const void* src, void* dst, int src_dtype, int dst_dtype,
                       int64_t n, int h, int w,
                       int64_t src_stride_n, int64_t src_stride_h,
                       int64_t dst_stride_n, int64_t dst_stride_h,
                       const float* wx, int kx, const float* wy, int ky, int border,
                       float amount, int clip, float lo, float hi, void* stream);

/* ------------------------------------------------------------------ 3-D Gaussian / unsharp (whole volumes)
 * skimage.filters.gaussian(image, sigma, mode, truncate) and skimage.filters.unsharp_mask(image, radius, amount) on a
 * 3-D array: scipy.ndimage.gaussian_filter over all three axes of every (d, h, w) volume of the batch of n.
 * wx / wy / wz: kx / ky / kz normalised 1-D weights (HOST arrays, copied into kernel parameters); each count odd, 1 ..
 * MIE_MAX_TAPS (MIE_E_KERNEL otherwise); kz == 1 with weight 1.0 leaves z unfiltered (sigma_z == 0).  Pass order x,
 * then y, then z, each acc = w[0]*x[0]; acc = fma(w[t], x[t], acc) in tap order — so with kz == 1 the result equals
 * mie_gaussian2d / mie_unsharp_amount on every plane bit for bit.  Any border mode on any axis length, whatever the
 * radius (every source index is mirrored / wrapped as often as needed): MIE_E_BORDER for an unknown mode only.
 * Pixel mapping as mie_gaussian2d; dst_dtype is src_dtype or MIE_F32.  unsharp3d: out = fma(amount, x - blur, x),
 * clamped to [0, 1] before quantisation when clip != 0; skimage's blur is mode 'reflect' (MIE_BORDER_SYMMETRIC),
 * truncate 4.  Strides in elements; one launch, no workspace; n == 0 is a no-op.                               */
int mie_gaussian3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                   int64_t n, int d, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                   int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                   const float* wx, int kx, const float* wy, int ky, const float* wz, int kz,
                   int border, float lo, float hi, void* stream);
int mie_unsharp3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                  int64_t n, int d, int h, int w,
                  int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                  int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                  const float* wx, int kx, const float* wy, int ky, const float* wz, int kz,
                  int border, float amount, int clip, float lo, float hi, void* stream);

/* ------------------------------------------------------------------ CLAHE
 * Replaces kornia.enhance.equalize_clahe(input, clip_limit, grid_size)
 * (reference pyproject.toml:8; SURVEY.md §8(a) A1) and, with
 * semantics = MIE_CLAHE_OPENCV, cv::CLAHE (SURVEY.md §8(a) A1', Appendix A).
 * 256 bins.  gh x gw = grid_size (rows, cols).  clip_limit <= 0 disables clipping.
 *
 * Stage entry points (used by the parity tests to compare integer artefacts
 * bit-exactly, "teacher forcing"):
 *   mie_clahe_hist : raw per-tile histograms  hist[n][gh][gw][256] (uint32)
 *   mie_clahe_luts : clipped/redistributed/cumulated LUTs luts[n][gh][gw][256] (uint8)
 *   mie_clahe_apply: interpolation pass given LUTs
 *   mie_clahe      : luts + apply, LUTs kept in `workspace`.                       */
size_t mie_clahe_workspace_bytes(int64_t n, int h, int w, int gh, int gw);
int mie_clahe_hist(const void* src, int src_dtype, int64_t n, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_h,
                   int gh, int gw, int semantics, float lo, float hi,
                   uint32_t* hist, void* stream);
int mie_clahe_luts(const void* src, int src_dtype, int64_t n, int h, int w,
                   int64_t src_stride_n, int64_t src_stride_h,
                   int gh, int gw, double clip_limit, int semantics, float lo, float hi,
                   uint8_t* luts, void* stream);
int mie_clahe_apply(const void* src, void* dst, int src_dtype, int dst_dtype,
                    int64_t n, int h, int w,
                    int64_t src_stride_n, int64_t src_stride_h,
                    int64_t dst_stride_n, int64_t dst_stride_h,
                    int gh, int gw, int semantics, float lo, float hi,
                    const uint8_t* luts, void* stream);
int mie_clahe(const void* src, void* dst, int src_dtype, int dst_dtype,
              int64_t n, int h, int w,
              int64_t src_stride_n, int64_t src_stride_h,
              int64_t dst_stride_n, int64_t dst_stride_h,
              int gh, int gw, double clip_limit, int semantics, float lo, float hi,
              void* workspace, size_t workspace_bytes, void* stream);

/* 65 536-bin mode: semantics = MIE_CLAHE_OPENCV with MIE_U16 planes (cv::CLAHE on CV_16UC1; SURVEY.md
 * §8(a) A1', §8(f) F2) — no quantisation to 256 levels, bit-exact against cv2.  mie_clahe accepts it
 * (dst_dtype must be MIE_U16); the LUTs are uint16[n][gh][gw][65536] = mie_clahe16_lut_bytes(gh, gw)
 * per image, and `workspace` must hold the LUTs of at least ONE image: the batch is processed in groups
 * of floor(workspace_bytes / mie_clahe16_lut_bytes) images (larger groups are faster: fewer, fuller launches).
 * From 296 tiles on, mie_clahe bounds the LUTs by the batch's largest pixel value — one extra pass; LUT entries
 * above it are never looked up, so only the bins up to it are zeroed, swept and written (12-bit data in a 16-bit
 * container: 1/16 of the work, same output bits); the bound lives in 256 spare bytes behind the LUTs of the group
 * (a workspace without them gives one image of its group up).  mie_clahe16_luts is the stage entry point for
 * parity tests and always returns complete LUTs. */
size_t mie_clahe16_lut_bytes(int gh, int gw);
int mie_clahe16_luts(const void* src, int64_t n, int h, int w,
                     int64_t src_stride_n, int64_t src_stride_h,
                     int gh, int gw, double clip_limit, uint16_t* luts, void* stream);

/* ------------------------------------------------------------------ global equalisation
 * Replaces kornia.enhance.equalize(input) == torchvision equalize rule
 * (reference pyproject.toml:8,16; SURVEY.md §8(a) A2): 256-bin histogram of
 * trunc(x01*255), step=(N-last_nonzero)//255, lut[k]=clamp((cum[k-1]+step//2)//step),
 * identity when step==0.  workspace >= mie_equalize_workspace_bytes(n).           */
size_t mie_equalize_workspace_bytes(int64_t n);
int mie_equalize(const void* src, void* dst, int src_dtype, int dst_dtype,
                 int64_t n, int h, int w,
                 int64_t src_stride_n, int64_t src_stride_h,
                 int64_t dst_stride_n, int64_t dst_stride_h,
                 float lo, float hi, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ median
 * mie_median2d replaces kornia.filters.median_blur(input, kernel_size) (zero
 * padded, MIE_BORDER_CONSTANT) and skimage.filters.median on 2-D input
 * (MIE_BORDER_REPLICATE == scipy 'nearest'); SURVEY.md §8(a) A5.  kx, ky in {3,5,7}.
 * Pure selection: dst_dtype == src_dtype, bit-exact, no normalisation.
 * mie_median3d replaces skimage.filters.median on a 3-D volume ->
 * scipy.ndimage.median_filter(footprint=ones((3,3,3)), mode='nearest')
 * (reference pyproject.toml:12; SURVEY.md §8(a) A6): rank 13 of 27.  The volume is
 * d planes; halo_lo / halo_hi are the neighbouring slab's boundary planes
 * (h*w elements, row stride w) or NULL where the slab touches the volume face,
 * in which case `border` applies (REPLICATE or CONSTANT).                          */
int mie_median2d(const void* src, void* dst, int dtype, int64_t n, int h, int w,
                 int64_t src_stride_n, int64_t src_stride_h,
                 int64_t dst_stride_n, int64_t dst_stride_h,
                 int ky, int kx, int border, void* stream);
int mie_median3d(const void* src, void* dst, int dtype, int d, int h, int w,
                 int64_t src_stride_d, int64_t src_stride_h,
                 int64_t dst_stride_d, int64_t dst_stride_h,
                 const void* halo_lo, const void* halo_hi, int border, void* stream);

/* mie_sk_median / mie_sk_median3d: skimage.filters.median(image, footprint, mode, cval) with ANY boolean footprint
 * -> scipy.ndimage.median_filter(image, footprint=footprint, mode=mode, cval=cval), on n planes or n volumes
 * (reference pyproject.toml:12; SURVEY.md §8(a) A6).  Semantics VERIFIED against scipy 1.18.1
 * (tests/test_sk_median.py pins them on the CPU):
 *   out[p] = element count / 2 (0-based) of the sorted samples in[p + c - extent / 2] over the set cells c of the
 *   footprint (integer division per axis: even extents are legal and their centre sits at extent / 2), i.e. the upper
 *   median when count is even.  Samples outside the image follow `border` (MIE_BORDER_*: SYMMETRIC = scipy 'reflect',
 *   REFLECT = 'mirror', REPLICATE = 'nearest', CIRCULAR = 'wrap', folded as often as needed when the footprint is
 *   longer than the axis; CONSTANT = 'constant', where the sample is cval).  Pure selection: dst_dtype == src_dtype ==
 *   dtype, and every output is a sample or cval.  scipy's 'reflect' reads outside the image at offsets -2 n m (m >= 2)
 *   of an axis of length n > 1; the kernels fold those like every other offset (filters.median refuses footprints that
 *   reach them).  skimage.morphology.disk / ball (X^2 + Y^2 (+ Z^2) <= r^2) are RECALLED.  NaN in float images has no defined median (unspecified here as in
 *   scipy); with both -0.0 and +0.0 in a window the sign of a zero result may differ from scipy's.
 * footprint: HOST row-major uint8 mask of fy x fx (fz x fy x fx) cells, nonzero = set, read at call time.  Extents 1 ..
 * MIE_SK_MEDIAN_MAX_EXTENT (planes) or 1 .. MIE_SK_MEDIAN3D_MAX_EXTENT (volumes) per axis.
 * cval: the constant already cast to the image dtype as scipy casts it (the caller does the cast), so it must be
 * exactly representable: an integer in the dtype's range, or a float32 value (inf and NaN included).
 * Errors: MIE_E_KERNEL for an extent < 1 or above the bound, or a mask with no set cell; MIE_E_NULL for a null
 * footprint (or null src / dst with n > 0); MIE_E_BORDER for an unknown mode; MIE_E_RANGE for a cval that is not
 * representable; MIE_E_DTYPE, MIE_E_SHAPE and MIE_E_STRIDE as everywhere.  n == 0 is a no-op after the checks.
 * No workspace, no allocation and no host synchronisation (the footprint travels in the kernel parameters), so the
 * calls can be captured into a CUDA graph; 64-bit addressing. */
#define MIE_SK_MEDIAN_MAX_EXTENT 65
#define MIE_SK_MEDIAN3D_MAX_EXTENT 17
int mie_sk_median(const void* src, void* dst, int dtype, int64_t n, int h, int w,
                  int64_t src_stride_n, int64_t src_stride_h,
                  int64_t dst_stride_n, int64_t dst_stride_h,
                  const uint8_t* footprint, int fy, int fx, int border, double cval, void* stream);
int mie_sk_median3d(const void* src, void* dst, int dtype, int64_t n, int d, int h, int w,
                    int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                    int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                    const uint8_t* footprint, int fz, int fy, int fx, int border, double cval, void* stream);

/* ------------------------------------------------------------------ bilateral
 * Replaces kornia.filters.bilateral_blur(input, kernel_size, sigma_color,
 * sigma_space, border_type, color_distance_type) for single-channel planes
 * (SURVEY.md §8(a) A7).  wspace: ky*kx HOST floats (outer product of the
 * normalised 1-D Gaussians).  Weight = wspace * 2^(c2 * (d*d)) with the fixed-sequence exp2 of
 * csrc/bilateral.cu:mie_exp2n, c2 = fp32(-0.5 log2(e) / sigma_color^2), accumulated in row-major tap order
 * (num = fma(w, v, num); den += w), out = num / den.  ky, kx odd <= 15.           */
int mie_bilateral(const void* src, void* dst, int src_dtype, int dst_dtype,
                  int64_t n, int h, int w,
                  int64_t src_stride_n, int64_t src_stride_h,
                  int64_t dst_stride_n, int64_t dst_stride_h,
                  const float* wspace, int ky, int kx, float sigma_color, int border,
                  float lo, float hi, void* stream);

/* ------------------------------------------------------------------ non-local means
 * Replaces skimage.restoration.denoise_nl_means(image, patch_size, patch_distance, h,
 * fast_mode=True, sigma) on 2-D single-channel planes (reference pyproject.toml:12; SURVEY.md §8(a)
 * A8; BASELINE.json config 5).  Fast-mode semantics restated in csrc/nlm.cu: uniform patch weights,
 * search window [-patch_distance, patch_distance]^2 over the reflect-padded image, weight
 * exp(-max(D,0) / (h^2 s^2)) cut off at distance 5.  patch_size <= 9, patch_distance <= 16.
 * fp32 arithmetic, within rel 1e-5 of the float64 oracle (not bit-exact: exp is ex2.approx).       */
int mie_nlm(const void* src, void* dst, int src_dtype, int dst_dtype,
            int64_t n, int h, int w,
            int64_t src_stride_n, int64_t src_stride_h,
            int64_t dst_stride_n, int64_t dst_stride_h,
            int patch_size, int patch_distance, float h_param, float sigma,
            float lo, float hi, void* stream);

/* The same function with fast_mode=False: skimage's _nl_means_denoising_2d [RECALLED] — Gaussian patch weights
 * exp(-(di^2 + dj^2) / (2 ((s-1)/4)^2)) normalised by their sum and h^2, image reflect-padded by the patch radius
 * only, search window clipped at the image, cut-off test (distance > 5 -> weight 0) before every patch row.
 * float64 arithmetic in upstream's order.  dst_dtype: the source dtype, MIE_F32 or MIE_F64.  patch_size <= 15,
 * patch_distance <= 32 (MIE_E_KERNEL beyond).                                                              */
int mie_nlm_slow(const void* src, void* dst, int src_dtype, int dst_dtype,
                 int64_t n, int h, int w,
                 int64_t src_stride_n, int64_t src_stride_h,
                 int64_t dst_stride_n, int64_t dst_stride_h,
                 int patch_size, int patch_distance, double h_param, double sigma,
                 float lo, float hi, void* stream);

/* ------------------------------------------------------------------ quality metrics (SURVEY.md §8(f) F4)
 * Device-side reductions behind sewar.full_ref.mse / rmse / psnr / ssim (reference pyproject.toml:13,
 * pin uv.lock:692-700: sewar 0.4.6, numpy/scipy code, not installable here — semantics RECALLED).
 * Pixels are used raw (no [0,1] mapping).  `out` is a DEVICE array of n x 2 float64:
 *   mie_sqdiff_sums: out[i] = { sum (a-b)^2, sum |a-b| } of plane i  (integer planes: exact 64-bit sums)
 *   mie_ssim_sums  : out[i] = { sum ssim_map, sum cs_map } over the (h-ws+1) x (w-ws+1) 'valid' windows
 *                    of a ws x ws UNIFORM filter (sewar's default fltr_specs), ws <= 16:
 *                    mu = S/ws^2, var = S2/ws^2 - mu^2, cov = Sab/ws^2 - mu_a mu_b (window sums exact for
 *                    integer planes), ssim = (2 mu_a mu_b + c1)(2 cov + c2) / ((mu_a^2 + mu_b^2 + c1)
 *                    (var_a + var_b + c2)), cs = (2 cov + c2) / (var_a + var_b + c2), float64.
 * The caller divides by the pixel / window count (and takes sqrt / log10).  workspace >=
 * mie_metric_workspace_bytes(n, h, w, ws) with ws = 0 for mie_sqdiff_sums.  Reductions run in a
 * fixed order: results are bit-reproducible from run to run.                                        */
size_t mie_metric_workspace_bytes(int64_t n, int h, int w, int ws);
int mie_sqdiff_sums(const void* a, const void* b, int dtype, int64_t n, int h, int w,
                    int64_t a_stride_n, int64_t a_stride_h, int64_t b_stride_n, int64_t b_stride_h,
                    double* out, void* workspace, size_t workspace_bytes, void* stream);
int mie_ssim_sums(const void* a, const void* b, int dtype, int64_t n, int h, int w,
                  int64_t a_stride_n, int64_t a_stride_h, int64_t b_stride_n, int64_t b_stride_h,
                  int ws, double c1, double c2,
                  double* out, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ fused bilateral -> CLAHE (BASELINE.json config 4)
 * equalize_clahe(bilateral_blur(x01, (k, k), sigma_color, sigma_space, border), clip_limit, (gh, gw)), quantised once at
 * the end — the same bits as mie_bilateral (F32 out) -> mie_clahe, without the fp32 image in between: stage 1 writes the
 * CLAHE lookup index of every filtered pixel (1 byte) and accumulates the tile histograms, stage 2 turns histograms into
 * LUTs, stage 4 blends and quantises.  `stages` is a mask of 1 | 2 | 4 (7 = everything; single stages for timing).
 * Covered geometry (mie_bilateral_clahe_is_fused() == 1): k in {3,5,7,9}, CLAHE tiles that are multiples of 32 pixels and
 * need no padding, w % 4 == 0, w <= 4096, gw <= 32, integer pixels in their dtype's default range or float pixels;
 * anything else returns MIE_E_UNSUPPORTED (call mie_bilateral and mie_clahe).  wspace: k*k spatial weights (HOST).   */
size_t mie_bilateral_clahe_workspace_bytes(int64_t n, int h, int w, int gh, int gw);
int mie_bilateral_clahe_is_fused(int h, int w, int gh, int gw, int k, int dtype);
int mie_bilateral_clahe(const void* src, void* dst, int src_dtype, int dst_dtype,
                        int64_t n, int h, int w,
                        int64_t src_stride_n, int64_t src_stride_h,
                        int64_t dst_stride_n, int64_t dst_stride_h,
                        const float* wspace, int k, float sigma_color, int border,
                        int gh, int gw, double clip_limit, float lo, float hi, int stages,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ scikit-image exposure / restoration (F3)
 * skimage.exposure.equalize_adapthist(image, kernel_size, clip_limit, nbins), skimage.exposure.equalize_hist(image)
 * and skimage.restoration.denoise_bilateral(image, win_size, sigma_color, sigma_spatial, bins, mode, cval)
 * (reference pyproject.toml:12; SURVEY.md §2.2, Appendix B3/B4) — different algorithms from their kornia counterparts
 * above.  RECALLED semantics: the kernels follow oracle/mie_oracle.c:orc_sk_* bit for bit.  Every plane of the batch
 * is one image (skimage on a 2-D array).  dst_dtype: MIE_F64 (skimage's dtype for integer images) or MIE_F32 (the
 * float64 result rounded once).  Outputs are floats in [0, 1] (bilateral: on the img_as_float scale).
 *
 * mie_sk_equalize_adapthist: src u8 / u16 / i16 / f32; (kr, kc) = kernel_size in pixels (skimage default: max(dim/8, 1));
 *   nbins <= 4096.  Four launches: per-image min/max, one block per contextual region (histogram on 2^14 grey levels,
 *   iterative clip redistribution, mapping), interpolation (+ min/max of the result), final min-max rescale.
 * mie_sk_equalize_hist: src u8 / u16 / i16 (one bin per integer value between the image's min and max).
 * mie_sk_denoise_bilateral: src u8 / u16 / i16; win_size odd; mode 0 constant(cval) 1 edge 2 symmetric 3 reflect 4 wrap;
 *   color_luts: DEVICE float64 [n][bins] and range_lut: DEVICE float64 [win_size^2], built by the caller exactly as
 *   upstream builds them in Python; ranges: DEVICE int [n][2] = per-image (min, max) code.                              */
size_t mie_sk_adapthist_workspace_bytes(int64_t n, int h, int w, int kr, int kc, int nbins);
int mie_sk_equalize_adapthist(const void* src, void* dst, int src_dtype, int dst_dtype,
                              int64_t n, int h, int w,
                              int64_t src_stride_n, int64_t src_stride_h,
                              int64_t dst_stride_n, int64_t dst_stride_h,
                              int kr, int kc, double clip_limit, int nbins,
                              void* workspace, size_t workspace_bytes, void* stream);
/* mie_sk_equalize_adapthist3d: skimage.exposure.equalize_adapthist on a 3-D array — every (d, h, w) volume of the batch
 * is ONE image (mie_sk_equalize_adapthist treats each plane on its own).  Same dtypes, nbins range and error codes as
 * the 2-D entry point; (kd, kr, kc) = kernel_size in voxels (skimage default: max(dim/8, 1) per axis), kd*kr*kc <= 2^31-1.
 * Semantics, in volume coordinates (z, y, x):
 *   grey  = round_half_even(rescale_intensity(img_as_float(v), out_range=(0, 16383))) with min / max over the VOLUME
 *           (float64 for integer input, float32 for float32 input); bin = grey / (1 + 16384 / nbins);
 *   regions: ceil(d/kd) x ceil(h/kr) x ceil(w/kc) boxes anchored at the origin, completed past the far faces by numpy
 *           'reflect' padding (repeated reflection for pads longer than the axis); per region histogram -> clip_histogram
 *           with clim = max(int(clip_limit * kd*kr*kc), 1) (clip_limit <= 0: 65535, ASSUMED as in 2-D) ->
 *           map = int(min(cumsum * (16383 / (kd*kr*kc)) + 0, 16383));
 *   voxel (z, y, x) lies in block ((z + kd/2) / kd, ...) at position ((z + kd/2) % kd, ...); per axis it blends regions
 *           clamp(block - 1) and clamp(block) with weights (1 - c, c), c = pos / k (float64); the coefficient of edge
 *           (ez, ey, ex) is (wx[ex] * wy[ey]) * wz[ez]; acc += (float)(map * coef) in float32 over the edges in
 *           np.ndindex(2, 2, 2) order (z outermost); truncated to uint16;
 *   out   = rescale_intensity(out_range=(0, 1)) of that uint16 volume, min / max over the volume.
 * Launches: min / max, a code -> bin table per volume (integer input), one thread-block cluster per region (large
 * regions are counted by up to 8 CTAs and merged through distributed shared memory), trilinear blend (+ min / max),
 * rescale.  The workspace holds n * 65536 table entries whatever the dtype.                                           */
size_t mie_sk_adapthist3d_workspace_bytes(int64_t n, int d, int h, int w, int kd, int kr, int kc, int nbins);
int mie_sk_equalize_adapthist3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                                int64_t n, int d, int h, int w,
                                int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                                int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                                int kd, int kr, int kc, double clip_limit, int nbins,
                                void* workspace, size_t workspace_bytes, void* stream);
/* mie_sk_denoise_tv_chambolle / mie_sk_denoise_tv_chambolle3d: skimage.restoration.denoise_tv_chambolle(image, weight,
 * eps, max_num_iter) on every (h, w) plane (ndim 2, tau = 1/4) or every (d, h, w) volume (ndim 3, tau = 1/6) of the
 * batch; a (1, h, w) volume is therefore not a plane.  src u8 / u16 / i16 are computed in float64 on the img_as_float
 * scale (unsigned v / max, int16 (2 v + 1) / 65535), src f32 in float32; dst F64 or F32 (rounded once).
 * RECALLED semantics (upstream _denoise_tv_chambolle_nd; numpy twin tests/sk_tv_chambolle_twin.py), per pass i with
 * p = 0 on entry to pass 0, array axes a in order, every step one correctly rounded operation (no fma):
 *   d   = -(p0 + p1 [+ p2]), then d += p_a(x - e_a) where x_a >= 1, axis by axis;  out = image + d (pass 0: out = image)
 *   g_a = out(x + e_a) - out(x), 0 where x_a = n_a - 1;  norm = sqrt(g0^2 + g1^2 [+ g2^2])
 *   E   = (sum d^2 + weight * sum norm) / image.size;  p = (p - tau * g_a) / (1 + norm * (tau / weight))
 *   pass 0 sets E_init = E_previous = E; pass i > 0 stops if |E_previous - E| < eps * E_init, else E_previous = E.
 * The result is out of the last pass run (its p update is discarded): max_num_iter = 1 returns the float image, and a
 * constant image (E_init = 0) runs every pass and comes back unchanged.  In float32, tau and tau / weight (a float64
 * quotient) are rounded to float32 and weight * sum, eps * E_init are float32 products.  The two energy sums are taken
 * in float64 in a fixed order (numpy sums pairwise); they feed only the stopping test.  Every image stops on its own.
 * weight must be finite and > 0 (MIE_E_RANGE), max_num_iter >= 1 (MIE_E_SHAPE).  iters: DEVICE int32[n] receiving the
 * passes run per image, or NULL.  One launch per pass up to max_num_iter - 1 whatever the stopping point (a stopped
 * image's CTAs return at once), then one finishing launch; no host synchronisation and no allocation: all state lives in
 * the workspace (>= the query, 256-byte aligned) and is re-initialised by every call, so the call can be captured into
 * a CUDA graph.  The workspace holds two float copies of p: 2 * ndim * n * voxels * sizeof(float type) bytes plus a
 * little state. */
size_t mie_sk_tv_chambolle_workspace_bytes(int64_t n, int h, int w, int src_dtype);
size_t mie_sk_tv_chambolle3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype);
int mie_sk_denoise_tv_chambolle(const void* src, void* dst, int src_dtype, int dst_dtype,
                                int64_t n, int h, int w,
                                int64_t src_stride_n, int64_t src_stride_h,
                                int64_t dst_stride_n, int64_t dst_stride_h,
                                double weight, double eps, int max_num_iter, int* iters,
                                void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_denoise_tv_chambolle3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                                  int64_t n, int d, int h, int w,
                                  int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                                  int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                                  double weight, double eps, int max_num_iter, int* iters,
                                  void* workspace, size_t workspace_bytes, void* stream);
/* mie_sk_structural_similarity / mie_sk_structural_similarity3d: skimage.metrics.structural_similarity(im1, im2,
 * win_size, data_range, gaussian_weights, K1, K2, sigma, use_sample_covariance) on every (h, w) plane (ndim 2) or every
 * (d, h, w) volume (ndim 3) of the batch; a (1, h, w) volume is therefore not a plane (a 7x7x7 window needs d >= 7).
 * RECALLED semantics (upstream skimage/metrics/_structural_similarity.py, 0.26; numpy twin tests/sk_ssim_twin.py):
 *   F = float32 for f32 sources, float64 for u8 / u16 / i16 sources (RAW values, not img_as_float);
 *   filter = uniform_filter(size = win_size) or, gaussian_weights, gaussian(sigma, truncate = 3.5, mode = 'reflect');
 *   ux, uy, uxx, uyy, uxy = filter(a), filter(b), filter(a*a), filter(b*b), filter(a*b), products in F;
 *   vx = cov_norm (uxx - ux ux), vy = cov_norm (uyy - uy uy), vxy = cov_norm (uxy - ux uy);
 *   A1 = 2 ux uy + c1, A2 = 2 vxy + c2, B1 = ux^2 + uy^2 + c1, B2 = vx + vy + c2;  S = (A1 A2) / (B1 B2), all in F;
 *   mssim = mean(S cropped by (win_size - 1) / 2 on every side of every axis), in float64.
 * The caller computes cov_norm = NP / (NP - 1) with NP = win_size^ndim (1.0 without the sample covariance), c1 = (K1 R)^2
 * and c2 = (K2 R)^2 as upstream does in Python; for f32 sources they are rounded to float32, as NumPy 2 does.
 * scipy.ndimage's arithmetic (checked against scipy 1.18.1), which makes the map bit-exact: the 1-D pass runs along
 * axis 0, then 1, then 2, each line extended by half-sample symmetric reflection (d c b a | a b c d | d c b a, repeated
 * as often as needed) into float64, results rounded to F between passes.
 *   box (taps == NULL): tmp = sum of the first win_size extended samples, out[0] = tmp / win_size, then for i >= 1
 *        tmp += ext[i + win_size - 1] - ext[i - 1] and out[i] = tmp / win_size — a running sum over the whole line;
 *   Gaussian (taps = HOST float64 weights exp(-0.5 x^2 / sigma^2) / sum, x = -r .. r, ntaps = 2r + 1 odd, copied at
 *        call time): tmp = ext[c] w[r], then tmp += (ext[c + j] + ext[c - j]) w[j + r] for j = -r .. -1; no fma.
 *        win_size then only sets the crop and NP; the taps may reach beyond an axis.
 * map: NULL, or the S map (dst layout: its own strides), MIE_F64 for integer sources and MIE_F32 for f32 (MIE_E_DTYPE
 * otherwise).  mssim: DEVICE double[n], one value per image.  MIE_E_KERNEL for win_size or ntaps even, < 1 or
 * > MIE_MAX_TAPS; MIE_E_SHAPE for an image axis shorter than win_size.  The workspace (>= the query, 256-byte aligned)
 * does not grow with n or d beyond a fixed bound: the batch runs in chunks whose float buffers stay below 640 MiB
 * (plus 40 h w bytes for volumes, where a long volume's box z-pass carries its running sums between chunks).  Four
 * launches per chunk (three for planes), the per-image sums in a fixed order (same bits on every run); no host
 * synchronisation and no allocation, so the call can be captured into a CUDA graph.  n == 0 is a no-op. */
size_t mie_sk_structural_similarity_workspace_bytes(int64_t n, int h, int w, int src_dtype);
size_t mie_sk_structural_similarity3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype);
int mie_sk_structural_similarity(const void* a, const void* b, void* map, int src_dtype, int map_dtype,
                                 int64_t n, int h, int w,
                                 int64_t a_stride_n, int64_t a_stride_h,
                                 int64_t b_stride_n, int64_t b_stride_h,
                                 int64_t map_stride_n, int64_t map_stride_h,
                                 int win_size, const double* taps, int ntaps,
                                 double cov_norm, double c1, double c2, double* mssim,
                                 void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_structural_similarity3d(const void* a, const void* b, void* map, int src_dtype, int map_dtype,
                                   int64_t n, int d, int h, int w,
                                   int64_t a_stride_n, int64_t a_stride_d, int64_t a_stride_h,
                                   int64_t b_stride_n, int64_t b_stride_d, int64_t b_stride_h,
                                   int64_t map_stride_n, int64_t map_stride_d, int64_t map_stride_h,
                                   int win_size, const double* taps, int ntaps,
                                   double cov_norm, double c1, double c2, double* mssim,
                                   void* workspace, size_t workspace_bytes, void* stream);
/* mie_sk_ridge_filter / mie_sk_ridge_filter3d: skimage.filters.frangi / hessian / sato / meijering(image, sigmas, ...,
 * black_ridges, mode, cval) on every (h, w) plane (ndim 2) or every (d, h, w) volume (ndim 3) of the batch.
 * mie_sk_hessian_matrix / mie_sk_hessian_matrix3d: skimage.feature.hessian_matrix(image, sigma, mode, cval, order='rc',
 * use_gaussian_derivatives=True); mie_sk_hessian_eigvals: skimage.feature.hessian_matrix_eigvals.
 * RECALLED semantics (upstream skimage/filters/ridges.py and skimage/feature/corner.py, 0.26; numpy twin
 * tests/sk_ridges_twin.py):
 *   F = float32 for f32 sources, float64 for u8 / u16 / i16 sources.  The ridge filters take image.astype(F) on RAW
 *   values (negated when black_ridges == 0); hessian_matrix takes img_as_float (unsigned v / max, int16
 *   (2 v + 1) / 65535).
 *   Hessian: G_a = gaussian_filter(image, sigma, order = e_a, mode, cval), H_ab = gaussian_filter(G_a, sigma,
 *   order = e_b) for (a, b) in combinations_with_replacement(range(ndim), 2): H00 H01 H11, or H00 H01 H02 H11 H12 H22.
 *   Each gaussian_filter is a 1-D pass along axis 0, then 1, then 2, scipy's line arithmetic in float64 (checked
 *   against scipy 1.18.1): the line extended by `mode` (MIE_BORDER_*: CONSTANT = scipy 'constant' with cval, SYMMETRIC
 *   = 'reflect', REFLECT = 'mirror', REPLICATE = 'nearest', CIRCULAR = 'wrap', as often as needed), tmp = ext[c] w[r],
 *   then tmp += (ext[c + j] + ext[c - j]) w[j + r] (order 0) or (ext[c + j] - ext[c - j]) w[j + r] (order 1) for
 *   j = -r .. -1, no fma, rounded to F after each pass.  The elements are bit-exact.
 *   Eigenvalues, decreasing: 2-D (m + hs, m - hs), m = (H00 + H11) / 2, hs = sqrt(H01^2 + ((H00 - H11) / 2)^2) in F
 *   (bit-exact); 3-D cyclic Jacobi in float64, rounded to F (upstream: np.linalg.eigvalsh; both within a few ulp of
 *   the largest |eigenvalue|).
 *   filtered_max = 0; per sigma, in the order given: filtered_max = np.maximum(filtered_max, vals) with
 *   FRANGI:    e sorted by |e| (stable); l2 (, l3) = max(e[1:], 1e-10); 2-D r_a = inf, r_b = |e0| / l2; 3-D
 *              r_a = l2 / l3, r_b = |e0| / sqrt(l2 l3); s = sqrt(sum e^2); gamma < 0 (None): gamma = max(s) / 2 of the
 *              FIRST sigma, per image (1 if that is 0), reused for every sigma;
 *              vals = (1 - exp(-r_a^2 / 2 alpha^2)) exp(-r_b^2 / 2 beta^2) (1 - exp(-s^2 / 2 gamma^2)), in F;
 *   HESSIAN:   frangi (the caller passes gamma = 15), then out[out <= 0] = 1;
 *   SATO:      vals = sigma^2 * prod(max(e[:-1], 0)) ** (1 / (ndim - 1));
 *   MEIJERING: vals = the entry of largest |.| (first on ties) of circulant([1, alpha, ...]) @ e, clamped at 0, divided
 *              by its per-image max when that is > 0 (alpha: the caller passes 1 / (ndim + 1) for None).
 * Taps are HOST float64 arrays computed by the caller as scipy does (_gaussian_kernel1d(sigma, order,
 * int(4 sigma + 0.5))[::-1]), scale s at offset sum_{t < s} (2 radii[t] + 1) of taps0 (order 0) and taps1 (order 1),
 * copied at call time.  Errors: MIE_E_KERNEL for a radius < 0 or > MIE_SK_RIDGE_MAX_RADIUS, taps0 not symmetric or
 * taps1 not antisymmetric; MIE_E_RANGE for a sigma < 0 or not finite; MIE_E_NULL for null sigmas / radii / taps with
 * nscales > 0; MIE_E_SHAPE for nscales < 0; MIE_E_BORDER for an unknown mode; MIE_E_UNSUPPORTED for an unknown filter;
 * MIE_E_DTYPE for dst_dtype not MIE_F64 / MIE_F32 (the ridge filters; rounded once from F) or not F (hessian_matrix).
 * nscales == 0 writes zeros (HESSIAN: ones).  n == 0 is a no-op.
 * hessian_matrix writes element k of image i at dst + k dst_stride_e + i dst_stride_n + ... (dst_stride_e at least one
 * whole batch, MIE_E_STRIDE otherwise).  eigvals: h and eig DEVICE arrays of `dtype` (MIE_F32 or MIE_F64), element k
 * of voxel v at h[k h_stride_e + v] (ndim (ndim + 1) / 2 elements), eigenvalue k at eig[k eig_stride_e + v]; no
 * workspace.
 * Workspace (>= the query, 256-byte aligned): the batch runs in chunks of c = max(1, min(n, 2^24 / voxels, 65535))
 * images, all scales of a chunk before the next, so it does not grow with n:
 *   ridge, volumes:         9 align256(c voxels sizeof(F)) + 2 align256(8 c)
 *   ridge, planes:          4 align256(c voxels sizeof(F)) + align256(8 c voxels) + 2 align256(8 c)
 *   hessian_matrix:         5 (volumes) or 3 (planes) align256(c voxels sizeof(F))
 * — 9 F-sized images for one 512^3 volume.  Planes keep the running maximum in float64: upstream's first frangi
 * factor there is the float64 scalar 1 - exp(-inf), so its values are float64 from then on whatever F is.  Per scale: 24 pass launches for volumes (10 for planes) and one to three
 * epilogue launches.  The per-image maxima are integer atomicMax on the bits of non-negative values (same bits on
 * every run); no host synchronisation and no allocation, so the calls can be captured into a CUDA graph. */
#define MIE_SK_RIDGE_MAX_RADIUS 64
enum mie_sk_ridge { MIE_SK_FRANGI = 0, MIE_SK_HESSIAN = 1, MIE_SK_SATO = 2, MIE_SK_MEIJERING = 3 };
size_t mie_sk_ridge_filter_workspace_bytes(int64_t n, int h, int w, int src_dtype);
size_t mie_sk_ridge_filter3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype);
int mie_sk_ridge_filter(const void* src, void* dst, int src_dtype, int dst_dtype,
                        int64_t n, int h, int w,
                        int64_t src_stride_n, int64_t src_stride_h,
                        int64_t dst_stride_n, int64_t dst_stride_h,
                        int filter, int nscales, const double* sigmas, const int* radii,
                        const double* taps0, const double* taps1, int mode, double cval, int black_ridges,
                        double alpha, double beta, double gamma,
                        void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_ridge_filter3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                          int64_t n, int d, int h, int w,
                          int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                          int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h,
                          int filter, int nscales, const double* sigmas, const int* radii,
                          const double* taps0, const double* taps1, int mode, double cval, int black_ridges,
                          double alpha, double beta, double gamma,
                          void* workspace, size_t workspace_bytes, void* stream);
size_t mie_sk_hessian_matrix_workspace_bytes(int64_t n, int h, int w, int src_dtype);
size_t mie_sk_hessian_matrix3d_workspace_bytes(int64_t n, int d, int h, int w, int src_dtype);
int mie_sk_hessian_matrix(const void* src, void* dst, int src_dtype, int dst_dtype,
                          int64_t n, int h, int w,
                          int64_t src_stride_n, int64_t src_stride_h,
                          int64_t dst_stride_n, int64_t dst_stride_h, int64_t dst_stride_e,
                          int radius, const double* taps0, const double* taps1, int mode, double cval,
                          void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_hessian_matrix3d(const void* src, void* dst, int src_dtype, int dst_dtype,
                            int64_t n, int d, int h, int w,
                            int64_t src_stride_n, int64_t src_stride_d, int64_t src_stride_h,
                            int64_t dst_stride_n, int64_t dst_stride_d, int64_t dst_stride_h, int64_t dst_stride_e,
                            int radius, const double* taps0, const double* taps1, int mode, double cval,
                            void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_hessian_eigvals(const void* h, void* eig, int dtype, int ndim, int64_t count,
                           int64_t h_stride_e, int64_t eig_stride_e, void* stream);
size_t mie_sk_equalize_hist_workspace_bytes(int64_t n, int src_dtype);
int mie_sk_equalize_hist(const void* src, void* dst, int src_dtype, int dst_dtype,
                         int64_t n, int h, int w,
                         int64_t src_stride_n, int64_t src_stride_h,
                         int64_t dst_stride_n, int64_t dst_stride_h,
                         void* workspace, size_t workspace_bytes, void* stream);
int mie_sk_denoise_bilateral(const void* src, void* dst, int src_dtype, int dst_dtype,
                             int64_t n, int h, int w,
                             int64_t src_stride_n, int64_t src_stride_h,
                             int64_t dst_stride_n, int64_t dst_stride_h,
                             int win_size, int bins, int mode, double cval,
                             const double* color_luts, const double* range_lut, const int* ranges,
                             void* stream);

/* ------------------------------------------------------------------ z-halo exchange (BASELINE.json config 3)
 * The one exchange step of the path (SURVEY.md §8(e)): a volume sharded into z-slabs, one per rank, needs the
 * neighbouring slab's boundary plane on every interior face before mie_median3d(halo_lo, halo_hi) can run.
 * `nccl_comm` is the caller's ncclComm_t (passed as void*; from torch.distributed: ProcessGroupNCCL._comm_ptr())
 * whose rank numbering `rank` / `world` use.  Enqueues, in ONE NCCL group on `stream`:
 *     rank > 0        : ncclSend(first_plane -> rank-1), ncclRecv(halo_lo <- rank-1)
 *     rank < world-1  : ncclSend(last_plane  -> rank+1), ncclRecv(halo_hi <- rank+1)
 * plane_bytes each (h*w*element size; shipped as bytes).  Pointers of a missing neighbour may be NULL.  Every rank
 * of the communicator must make the call.  No allocation, no synchronisation; capturable into a CUDA graph.
 * NCCL is not linked into the library: the four entry points are resolved from the libnccl.so.2 already loaded into
 * the process, so the calls reach the same NCCL that created `nccl_comm`; MIE_E_UNSUPPORTED if there is none
 * (mie_halo_exchange_available() == 0).  world == 1 is a no-op.  NCCL failures: -100 - ncclResult_t. */
int mie_halo_exchange_available(void);
int mie_halo_exchange_z(void* nccl_comm, int rank, int world,
                        const void* first_plane, const void* last_plane,
                        void* halo_lo, void* halo_hi, size_t plane_bytes, void* stream);

/* Peer-load alternative to the exchange (one box, NVLink / NVSwitch): the halo pointers of mie_median3d may address the
 * NEIGHBOUR RANK's slab directly — its memory mapped into this process by CUDA IPC (mie_ipc_* below; from Python:
 * volume.PeerSlabPlan) — so the median kernel reads the two boundary planes over NVLink and no exchange is
 * launched at all.  This call enables the current device's access to `peer_device` (cudaDeviceEnablePeerAccess;
 * already-enabled is not an error); MIE_E_UNSUPPORTED when the two devices have no peer path. */
int mie_enable_peer_access(int peer_device);
/* CUDA IPC plumbing of the peer-load path (no torch types): mie_ipc_export writes the 64-byte cudaIpcMemHandle_t of the
 * allocation that contains dev_ptr and the pointer's byte offset inside it (the allocation base is resolved with the
 * driver's cuMemGetAddressRange, so pointers into a caching allocator's segment work); the handle travels to the
 * neighbour process by any means; mie_ipc_open — called there with the READER's device current — maps the allocation
 * (cudaIpcOpenMemHandle with lazy peer access) and returns its base; mie_ipc_close unmaps it. */
int mie_ipc_export(const void* dev_ptr, void* handle64, int64_t* offset_bytes);
int mie_ipc_open(const void* handle64, void** base_out);
int mie_ipc_close(void* base);

/* ------------------------------------------------------------------ fused chain (BASELINE.json config 2)
 * Gaussian denoise -> CLAHE -> unsharp mask in two launches; equals
 * mie_gaussian2d -> mie_clahe -> mie_unsharp (F32 intermediates) bit for bit.
 * wg*: denoise taps, wu*: unsharp taps.  Any geometry is accepted; shapes the
 * fused kernels do not cover run the same stages unfused inside the library,
 * using `workspace` for the fp32 intermediates.
 * `stages`: MIE_CHAIN_ALL runs the chain; MIE_CHAIN_STAGE_A / _B run only the
 * first / second launch of the fused path against the same workspace (used by
 * bench.py to time each kernel with CUDA events; MIE_E_UNSUPPORTED when the
 * geometry takes the unfused path).                                               */
enum mie_chain_stages {
    MIE_CHAIN_STAGE_A = 1, MIE_CHAIN_STAGE_B = 2, MIE_CHAIN_ALL = 3,
    /* schedule hints OR-ed into `stages` (tests / benchmarks): by default the marching kernels (one block per
     * 64-row band) serve jobs of >= 222 bands and the tile kernels (one block per 64x64 tile) smaller ones */
    MIE_CHAIN_PREFER_MARCH = 4, MIE_CHAIN_PREFER_TILES = 8
};
/* Which path (h, w, grid, kernel sizes) takes: 0 = stages run unfused (4 launches), 1 = generic
 * fused kernels (2 launches), 2 = tuned fused kernels for 64x64-pixel tiles and a 9-tap unsharp
 * (3 launches: chain_a, cell-table packing, chain_b; needs 16-byte aligned rows and the dtype's
 * default value range or a window mie_value_range_mode() reports as 1, otherwise 1 applies). */
int mie_chain_is_fused(int h, int w, int gh, int gw, int kgx, int kgy, int kux, int kuy);
/* How the tuned kernels treat the pixel mapping (lo, hi) of `dtype` (the value_range= extension of the Python
 * surface, SURVEY.md §8(b)): 0 = the dtype's default range (or float pixels); 1 = an integer window inside the
 * dtype's range whose divide-free conversion the host has checked against the IEEE quotient
 * (float(v) - lo) / (hi - lo) for EVERY code of the dtype — the tuned CLAHE / equalize / Gaussian / chain kernels
 * run it; -1 = neither (non-integer or out-of-range bounds, hi <= lo, or a code where the conversion would
 * differ): the generic kernels run it with the IEEE division.  Host-only; no CUDA call. */
int mie_value_range_mode(int dtype, float lo, float hi);
size_t mie_chain_workspace_bytes(int64_t n, int h, int w, int gh, int gw);
int mie_chain_gauss_clahe_unsharp(const void* src, void* dst, int src_dtype, int dst_dtype,
                                  int64_t n, int h, int w,
                                  int64_t src_stride_n, int64_t src_stride_h,
                                  int64_t dst_stride_n, int64_t dst_stride_h,
                                  const float* wgx, int kgx, const float* wgy, int kgy,
                                  int gh, int gw, double clip_limit,
                                  const float* wux, int kux, const float* wuy, int kuy,
                                  int border, float lo, float hi, int stages,
                                  void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MIE_H_ */
