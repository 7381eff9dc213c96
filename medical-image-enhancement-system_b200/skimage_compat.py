"""scikit-image call signatures over the same sm_100a kernels (SURVEY.md §2.2, §8(f) F3).

scikit-image >= 0.26.0 is the reference's second image-processing dependency (reference
pyproject.toml:12, pin uv.lock:619-650).  Its filters delegate to scipy.ndimage, whose Gaussian is the
kornia Gaussian with K = 2*int(truncate*sigma + 0.5) + 1 taps
(site-packages/scipy/ndimage/_filters.py:656-669, 745-747) and whose border modes map onto the ABI's:

    scipy / skimage mode   'nearest'    'reflect'     'mirror'    'constant'   'wrap'
    include/mie.h          REPLICATE    SYMMETRIC     REFLECT     CONSTANT     CIRCULAR

    gaussian(image, sigma, mode=, truncate=)            <- skimage.filters.gaussian
    unsharp_mask(image, radius, amount, preserve_range) <- skimage.filters.unsharp_mask
    median(image, footprint, mode=, cval=)              <- skimage.filters.median           (filters.py)
    disk(radius), ball(radius)                          <- skimage.morphology.disk / ball (median footprints)
    denoise_nl_means(image, ...)                        <- skimage.restoration.denoise_nl_means (filters.py)

Scale: skimage converts integer images to float with img_as_float (unsigned: v / max; signed: [-1, 1]).
Here integer tensors use this package's mapping x01 = (v - lo) / (hi - lo) with the dtype's full range
(uint8 / uint16: identical to img_as_float; int16: the affine image of skimage's scale) and come back in
the SAME integer dtype unless out_dtype=torch.float32 — the natural contract for 16-bit slices.  The
arithmetic is fp32 (skimage: float64 for integer input): agreement with scipy.ndimage is ~2e-7 abs on
[0,1] data (tests/test_skimage_compat.py).

gaussian / unsharp_mask filter every (H, W) plane on its own by default.  With volumetric=True they make skimage's
call on a 3-D array instead: every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor is blurred along z
as well, sigma / radius a scalar or (z, y, x).  One sm_100a kernel (csrc/gauss3d.cu) runs the x, y and z passes in that
order, so a zero z sigma reproduces the per-plane result bit for bit; agreement with scipy.ndimage.gaussian_filter on
3-D [0,1] data is to fp32 rounding (tests/test_gaussian3d.py).

    equalize_adapthist(image, kernel_size, clip_limit, nbins)  <- skimage.exposure.equalize_adapthist
    equalize_hist(image, nbins, mask)                          <- skimage.exposure.equalize_hist
    denoise_bilateral(image, win_size, sigma_color, sigma_spatial, bins, mode, cval)
                                                               <- skimage.restoration.denoise_bilateral
    denoise_tv_chambolle(image, weight, eps, max_num_iter)     <- skimage.restoration.denoise_tv_chambolle

These four have different algorithms from their kornia counterparts (SURVEY.md Appendix B3/B4) and their own
kernels (csrc/sk_exposure.cu, csrc/sk_bilateral.cu, csrc/sk_tv.cu).  They keep skimage's numerics — float64 arithmetic and a float64
result in [0, 1] for integer images (out_dtype=torch.float32 rounds it once) — and skimage's per-image semantics:
every (H, W) plane of the input is one image.  equalize_adapthist(..., volumetric=True) is skimage's call on a 3-D
array instead: every (D, H, W) volume is one image with 3-D contextual regions, and denoise_tv_chambolle(...,
volumetric=True) runs the 3-D algorithm on every volume.  RECALLED semantics, restated in oracle/skimage_twin.py (numpy,
array-level) and oracle/mie_oracle.c (per pixel), which agree bit for bit; tests/test_live_pins.py compares all of it
with the real package when it is importable.

    structural_similarity(im1, im2, win_size, data_range, gaussian_weights, full, K1, K2, sigma, use_sample_covariance)
                                                               <- skimage.metrics.structural_similarity

scores every plane, or with volumetric=True every (D, H, W) volume, as one image with upstream's 'reflect' windows and
sample covariance (csrc/sk_ssim.cu; RECALLED, numpy twin tests/sk_ssim_twin.py).  metrics.ssim is sewar's 2-D SSIM
('valid' windows, population variance) and gives different numbers.

    frangi / hessian / sato / meijering(image, sigmas, ..., black_ridges, mode, cval)  <- skimage.filters.*
    hessian_matrix(image, sigma, mode, cval, use_gaussian_derivatives=True)           <- skimage.feature.hessian_matrix
    hessian_matrix_eigvals(H_elems)                                  <- skimage.feature.hessian_matrix_eigvals

are the Hessian-based ridge (vesselness) filters, per plane or, volumetric=True, per volume (csrc/sk_ridges.cu;
RECALLED, numpy twin tests/sk_ridges_twin.py).  The Hessian elements are bit-exact against scipy.ndimage's arithmetic;
3-D eigenvalues come from a float64 Jacobi solver instead of LAPACK.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from ._ffi import (BORDER, DTYPE_CODE, MIE_F32, MIE_F64, SCIPY_MODES, as_planes, as_volumes, call, lib, new_out,
                   plane_layout, require_cuda, use_workspace, value_range_of, volume_layout)
from .filters import MAX_TAPS, denoise_nl_means, gaussian_blur2d, get_gaussian_kernel1d, median  # noqa: F401

__all__ = ["gaussian", "unsharp_mask", "median", "disk", "ball", "denoise_nl_means", "SCIPY_MODES", "equalize_adapthist", "equalize_hist",
           "denoise_bilateral", "denoise_tv_chambolle", "structural_similarity", "frangi", "hessian", "sato",
           "meijering", "hessian_matrix", "hessian_matrix_eigvals"]

def disk(radius: int, dtype=np.uint8) -> np.ndarray:
    """skimage.morphology.disk(radius) (RECALLED): the (2r+1)^2 uint8 mask X^2 + Y^2 <= r^2 over X, Y = -r .. r."""
    g = np.arange(-int(radius), int(radius) + 1)
    return np.asarray(g[:, None] ** 2 + g[None, :] ** 2 <= int(radius) ** 2, dtype=dtype)


def ball(radius: int, dtype=np.uint8) -> np.ndarray:
    """skimage.morphology.ball(radius) (RECALLED): the (2r+1)^3 uint8 mask X^2 + Y^2 + Z^2 <= r^2."""
    g = np.arange(-int(radius), int(radius) + 1)
    return np.asarray(g[:, None, None] ** 2 + g[None, :, None] ** 2 + g[None, None, :] ** 2 <= int(radius) ** 2,
                      dtype=dtype)


def _taps(sigma: float, truncate: float) -> int:
    if not float(sigma) > 0.0:
        raise ValueError("sigma must be positive")
    k = 2 * int(float(truncate) * float(sigma) + 0.5) + 1
    if k > MAX_TAPS:
        raise ValueError(f"sigma * truncate needs {k} taps; up to {MAX_TAPS} are supported")
    return k


def _mode(mode: str, cval: float) -> str:
    if mode not in SCIPY_MODES:
        raise ValueError(f"mode must be one of {sorted(SCIPY_MODES)}. Got {mode!r}")
    if mode == "constant" and cval != 0:
        raise NotImplementedError("mode='constant' supports cval=0 only")
    return SCIPY_MODES[mode]


def gaussian(image: torch.Tensor, sigma=1, *, mode: str = "nearest", cval=0, preserve_range: bool = False,
             truncate: float = 4.0, channel_axis=None, out=None, value_range=None, out_dtype=None,
             volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.gaussian on 2-D planes ((H,W), (C,H,W), (B,C,H,W): every plane on its own).
    `sigma`: scalar or (sigma_y, sigma_x).  `preserve_range` is accepted for signature compatibility:
    integer tensors are returned in their own dtype and range either way (see the module docstring).

    volumetric=True: the last three dimensions of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor form ONE volume, as
    skimage treats a 3-D array — blurred along z as well.  `sigma`: scalar or (sigma_z, sigma_y, sigma_x); an axis
    with sigma 0 is not filtered, so sigma (0, s, s) gives the per-plane result bit for bit."""
    if channel_axis is not None:
        raise NotImplementedError("planes are filtered separately; channel_axis is not supported")
    if out is not None:
        raise NotImplementedError("out= is not supported")
    if volumetric:
        return _gaussian3d(image, sigma, _mode(mode, cval), truncate, value_range, out_dtype, None)
    sy, sx = (sigma if isinstance(sigma, (tuple, list)) else (sigma, sigma))
    return gaussian_blur2d(image, (_taps(sy, truncate), _taps(sx, truncate)), (float(sy), float(sx)), _mode(mode, cval),
                           value_range=value_range, out_dtype=out_dtype)


def unsharp_mask(image: torch.Tensor, radius=1.0, amount=1.0, preserve_range: bool = False, *, channel_axis=None,
                 value_range=None, out_dtype=None, volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.unsharp_mask: image + amount * (image - gaussian(image, sigma=radius, mode='reflect')),
    clipped to [0, 1] on the normalised scale unless preserve_range (integer outputs saturate at the dtype's
    range in both cases).

    volumetric=True: every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor is one 3-D image, blurred
    over all three axes as skimage does for a 3-D array; `radius`: scalar or (r_z, r_y, r_x)."""
    if channel_axis is not None:
        raise NotImplementedError("planes are filtered separately; channel_axis is not supported")
    if volumetric:
        return _gaussian3d(image, radius, "symmetric", 4.0, value_range, out_dtype,
                           (float(amount), 0 if preserve_range else 1))
    require_cuda(image)
    k = _taps(radius, 4.0)
    x, n, h, w = as_planes(image)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    wk = get_gaussian_kernel1d(k, float(radius))
    call(x.device, "mie_unsharp_amount", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), wk.ctypes.data, k, wk.ctypes.data, k, BORDER["symmetric"], float(amount),
         0 if preserve_range else 1, lo, hi)
    return dst


def _axis_weights(sigma, truncate: float) -> np.ndarray:
    """1-D weights of one axis of a volume: sigma 0 leaves the axis unfiltered (scipy skips it)."""
    s = float(sigma)
    if s < 0.0 or s != s:
        raise ValueError("sigma must be non-negative")
    if s == 0.0:
        return np.ones(1, np.float32)
    k = _taps(s, truncate)
    return get_gaussian_kernel1d(k, s)


def _gaussian3d(image: torch.Tensor, sigma, border: str, truncate, value_range, out_dtype, unsharp) -> torch.Tensor:
    """mie_gaussian3d / mie_unsharp3d (unsharp = (amount, clip)) on every (D, H, W) volume of `image`."""
    x, n, d, h, w = as_volumes(image)
    if isinstance(sigma, (tuple, list)):
        if len(sigma) != 3:
            raise ValueError(f"volumetric=True takes a scalar sigma or (sigma_z, sigma_y, sigma_x); got {sigma!r}")
        sz, sy, sx = sigma
    else:
        sz = sy = sx = sigma
    wz, wy, wx = (_axis_weights(s, truncate) for s in (sz, sy, sx))
    require_cuda(x)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    args = (x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype], *volume_layout(n, d, h, w),
            wx.ctypes.data, wx.size, wy.ctypes.data, wy.size, wz.ctypes.data, wz.size, BORDER[border])
    if unsharp is None:
        call(x.device, "mie_gaussian3d", *args, lo, hi)
    else:
        call(x.device, "mie_unsharp3d", *args, unsharp[0], unsharp[1], lo, hi)
    return dst


# ---------------------------------------------------------------------------------------------- exposure / restoration
_OUT_CODE = {torch.float32: MIE_F32, torch.float64: MIE_F64}
_PAD_MODES = {"constant": 0, "edge": 1, "symmetric": 2, "reflect": 3, "wrap": 4}


def _float_default(x: torch.Tensor) -> torch.dtype:
    """skimage's result dtype: float32 for float32 images, float64 (img_as_float) for integer images."""
    return torch.float32 if x.dtype == torch.float32 else torch.float64


def _sk_kernel_size(shape, kernel_size):
    if kernel_size is None:
        return [max(int(s) // 8, 1) for s in shape]
    if isinstance(kernel_size, (int, float)):
        return [int(kernel_size)] * len(shape)
    if len(kernel_size) != len(shape):
        raise ValueError(f"Incorrect value of `kernel_size`: {kernel_size}")
    return [int(k) for k in kernel_size]


def equalize_adapthist(image: torch.Tensor, kernel_size=None, clip_limit: float = 0.01, nbins: int = 256, *,
                       out_dtype=None, volumetric: bool = False) -> torch.Tensor:
    """skimage.exposure.equalize_adapthist on every (H, W) plane of `image` ((H,W), (C,H,W), (B,C,H,W)).

    `kernel_size`: size of the contextual regions in PIXELS (int or (rows, cols); default max(dim // 8, 1)) — not a
    grid like kornia's.  `clip_limit` in [0, 1] is a fraction of the region's pixels; `nbins` <= 4096.
    Returns float64 (float32 for float32 input) in [0, 1] like skimage, or `out_dtype`.

    volumetric=True: the last three dimensions of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor form ONE volume, as
    skimage treats a 3-D array — 3-D contextual regions of `kernel_size` = (kd, kr, kc) voxels (an int is a cube;
    default max(dim // 8, 1) per axis), a trilinear blend of 8 region mappings, min / max over the whole volume."""
    if volumetric:
        return _equalize_adapthist3d(image, kernel_size, clip_limit, nbins, out_dtype)
    require_cuda(image)
    x, n, h, w = as_planes(image)
    kr, kc = _sk_kernel_size((h, w), kernel_size)
    if kr <= 0 or kc <= 0:
        raise ValueError("kernel_size entries must be positive")
    if not 0 < int(nbins) <= 4096:
        raise NotImplementedError("nbins must be in 1..4096")
    dst = new_out(x, out_dtype, _OUT_CODE, _float_default(x))
    ws = use_workspace(x.device, lib().mie_sk_adapthist_workspace_bytes(n, h, w, kr, kc, int(nbins)))
    call(x.device, "mie_sk_equalize_adapthist", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
         *plane_layout(n, h, w), kr, kc, float(clip_limit), int(nbins), ws.data_ptr(), ws.numel())
    return dst


def _equalize_adapthist3d(image: torch.Tensor, kernel_size, clip_limit, nbins, out_dtype) -> torch.Tensor:
    x, n, d, h, w = as_volumes(image)
    kd, kr, kc = _sk_kernel_size((d, h, w), kernel_size)
    if kd <= 0 or kr <= 0 or kc <= 0:
        raise ValueError("kernel_size entries must be positive")
    if not 0 < int(nbins) <= 4096:
        raise NotImplementedError("nbins must be in 1..4096")
    require_cuda(x)
    dst = new_out(x, out_dtype, _OUT_CODE, _float_default(x))
    ws = use_workspace(x.device, lib().mie_sk_adapthist3d_workspace_bytes(n, d, h, w, kd, kr, kc, int(nbins)))
    call(x.device, "mie_sk_equalize_adapthist3d", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
         *volume_layout(n, d, h, w), kd, kr, kc, float(clip_limit), int(nbins), ws.data_ptr(), ws.numel())
    return dst


def equalize_hist(image: torch.Tensor, nbins: int = 256, mask=None, *, out_dtype=None) -> torch.Tensor:
    """skimage.exposure.equalize_hist on every (H, W) plane of an INTEGER tensor: one bin per integer value between the
    plane's min and max (skimage ignores `nbins` for integer images), out = cdf[v] in float64."""
    if mask is not None:
        raise NotImplementedError("mask= is not supported")
    require_cuda(image)
    if image.dtype == torch.float32:
        raise NotImplementedError("equalize_hist is built for integer images (uint8 / uint16 / int16); float images use "
                                  "numpy.histogram's edge rules upstream")
    x, n, h, w = as_planes(image)
    dst = new_out(x, out_dtype, _OUT_CODE, torch.float64)
    ws = use_workspace(x.device, lib().mie_sk_equalize_hist_workspace_bytes(n, DTYPE_CODE[x.dtype]))
    call(x.device, "mie_sk_equalize_hist", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
         *plane_layout(n, h, w), ws.data_ptr(), ws.numel())
    return dst


def _as_float_codes(dtype: torch.dtype, codes: np.ndarray) -> np.ndarray:
    """skimage.util.img_as_float of integer codes (float64): unsigned v / max, int16 (2 v + 1) / 65535."""
    c = codes.astype(np.float64)
    if dtype == torch.uint8:
        return c / 255.0
    if dtype == torch.uint16:
        return c / 65535.0
    return (c * 2.0 + 1.0) / 65535.0


def denoise_bilateral(image: torch.Tensor, win_size=None, sigma_color=None, sigma_spatial: float = 1, bins: int = 10000,
                      mode: str = "constant", cval: float = 0, *, channel_axis=None, out_dtype=None) -> torch.Tensor:
    """skimage.restoration.denoise_bilateral on every (H, W) plane of an INTEGER tensor (single channel).

    The two look-up tables are built on the host exactly as upstream builds them in Python (numpy exp over
    linspace(0, max_value, bins) and over the window's hypot grid); per-plane min / max (and the standard deviation
    when sigma_color is None) are read back from the device for that — one small synchronisation per call.
    Returns float64 on skimage's img_as_float scale ([0, 1]; [-1, 1] for int16), or `out_dtype`."""
    if channel_axis is not None:
        raise NotImplementedError("planes are filtered separately; channel_axis is not supported")
    if mode not in _PAD_MODES:
        raise ValueError("Invalid mode specified.  Please use `constant`, `edge`, `wrap`, `symmetric` or `reflect`.")
    require_cuda(image)
    if image.dtype == torch.float32:
        raise NotImplementedError("denoise_bilateral is built for integer images (uint8 / uint16 / int16)")
    x, n, h, w = as_planes(image)
    if win_size is None:
        win_size = max(5, 2 * int(math.ceil(3 * sigma_spatial)) + 1)
    win_size = int(win_size)
    dst = new_out(x, out_dtype, _OUT_CODE, torch.float64)
    if n == 0:
        return dst
    planes = x.reshape(n, h * w)
    wide = planes.to(torch.int32)
    vmin, vmax = torch.aminmax(wide, dim=1)
    ranges = torch.stack([vmin, vmax], dim=1).to(torch.int32).contiguous()
    r_host = ranges.cpu().numpy()
    fmin = _as_float_codes(x.dtype, r_host[:, 0])
    fmax = _as_float_codes(x.dtype, r_host[:, 1])
    if sigma_color is None:   # image.std() of the float image, per plane
        if x.dtype == torch.int16:
            f = (wide.to(torch.float64) * 2.0 + 1.0) / 65535.0
        else:
            f = wide.to(torch.float64) / (255.0 if x.dtype == torch.uint8 else 65535.0)
        sig = f.std(dim=1, unbiased=False).cpu().numpy()
    else:
        sig = np.full(n, float(sigma_color), np.float64)
    max_value = np.where(fmin < 0, fmax - fmin, fmax)
    luts = np.ones((n, int(bins)), np.float64)
    for i in range(n):
        if r_host[i, 0] == r_host[i, 1] or not sig[i] > 0:
            continue   # flat plane: returned unchanged by the kernel
        values = np.linspace(0, max_value[i], int(bins), endpoint=False)
        luts[i] = np.exp(-0.5 * (values ** 2 / sig[i] ** 2))
    ext = (win_size - 1) // 2
    g = np.arange(-ext, ext + 1)
    rr, cc = np.meshgrid(g, g, indexing="ij")
    spatial = np.exp(-0.5 * (np.hypot(rr, cc) ** 2 / float(sigma_spatial) ** 2)).ravel()
    d_luts = torch.from_numpy(np.ascontiguousarray(luts)).to(x.device)
    d_spatial = torch.from_numpy(np.ascontiguousarray(spatial)).to(x.device)
    call(x.device, "mie_sk_denoise_bilateral", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
         *plane_layout(n, h, w), win_size, int(bins), _PAD_MODES[mode], float(cval), d_luts.data_ptr(),
         d_spatial.data_ptr(), ranges.data_ptr())
    return dst


def denoise_tv_chambolle(image: torch.Tensor, weight: float = 0.1, eps: float = 2e-4, max_num_iter: int = 200, *,
                         channel_axis=None, out_dtype=None, volumetric: bool = False) -> torch.Tensor:
    """skimage.restoration.denoise_tv_chambolle on every (H, W) plane of `image` ((H,W), (C,H,W), (B,C,H,W)), each
    plane one 2-D image with its own energy and stopping point.

    volumetric=True: every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor is one 3-D image, as skimage
    treats a 3-D array.  Integer images are computed in float64 on the img_as_float scale, float32 images in float32;
    returns that float dtype, or `out_dtype`.  The iteration runs on the device with no host synchronisation."""
    return _denoise_tv_chambolle(image, weight, eps, max_num_iter, channel_axis, out_dtype, volumetric, None)


_INT_DATA_RANGE = {torch.uint8: 255, torch.uint16: 65535, torch.int16: 65535}   # skimage dtype_range max - min
_SSIM_KWARGS = ("K1", "K2", "sigma", "use_sample_covariance")


def _ssim_taps(sigma: float, truncate: float) -> np.ndarray:
    """scipy.ndimage's Gaussian weights in float64: exp(-0.5 / sigma^2 * x^2) / sum over x = -r .. r,
    r = int(truncate * sigma + 0.5); a sigma scipy does not filter with (<= 1e-15) is the single weight 1."""
    if sigma <= 1e-15:
        return np.ones(1, np.float64)
    r = int(truncate * sigma + 0.5)
    x = np.arange(-r, r + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return phi / phi.sum()


def structural_similarity(im1: torch.Tensor, im2: torch.Tensor, *, win_size=None, gradient: bool = False,
                          data_range=None, channel_axis=None, gaussian_weights: bool = False, full: bool = False,
                          volumetric: bool = False, **kwargs):
    """skimage.metrics.structural_similarity of every (H, W) plane of im1 against the same plane of im2 ((H,W), (C,H,W),
    (B,C,H,W)); with volumetric=True, of every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor as one
    3-D image (7x7x7 windows by default).  kwargs: K1, K2, sigma, use_sample_covariance, as upstream.

    Integer images are scored on their raw values in float64 (data_range defaults to the dtype's range), float32 images
    in float32 (data_range required).  Returns a Python float for a single image, else a float64 CPU tensor shaped like
    the leading dimensions; full=True returns (mssim, S) with S a CUDA tensor of the input's shape (float64 for integer
    input, float32 for float32).  Bit-exact maps against scipy.ndimage's arithmetic (include/mie.h)."""
    unknown = set(kwargs) - set(_SSIM_KWARGS)
    if unknown:
        raise TypeError(f"unexpected keyword arguments {sorted(unknown)}")
    for name, t in (("im1", im1), ("im2", im2)):
        if not isinstance(t, torch.Tensor) or t.dtype not in DTYPE_CODE:
            raise TypeError(f"{name} must be a uint8, uint16, int16 or float32 torch.Tensor")
    if im1.shape != im2.shape:
        raise ValueError("Input images must have the same dimensions.")
    if gradient:
        raise NotImplementedError("gradient=True is not supported")
    if channel_axis is not None:
        raise NotImplementedError("images are scored separately; channel_axis is not supported")
    if im1.dtype != im2.dtype:
        raise NotImplementedError(f"im1 and im2 must have the same dtype; got {im1.dtype} and {im2.dtype}")
    K1, K2, sigma = float(kwargs.get("K1", 0.01)), float(kwargs.get("K2", 0.03)), float(kwargs.get("sigma", 1.5))
    if K1 < 0:
        raise ValueError("K1 must be positive")
    if K2 < 0:
        raise ValueError("K2 must be positive")
    if sigma < 0:
        raise ValueError("sigma must be positive")
    use_sample_covariance = kwargs.get("use_sample_covariance", True)
    truncate = 3.5
    if win_size is None:
        win_size = 2 * int(truncate * sigma + 0.5) + 1 if gaussian_weights else 7
    win_size = int(win_size)
    ndim = 3 if volumetric else 2
    if not ndim <= im1.dim() <= ndim + 2:
        raise ValueError(f"expected (H,W), (C,H,W) or (B,C,H,W) with volumetric=False, (D,H,W), (B,D,H,W) or "
                         f"(B,C,D,H,W) with volumetric=True; got shape {tuple(im1.shape)}")
    dims = tuple(int(s) for s in im1.shape[-ndim:])
    if any(s < win_size for s in dims):
        raise ValueError("win_size exceeds image extent. Either ensure that your images are at least 7x7; or pass "
                         "win_size explicitly in the function call, with an odd value less than or equal to the smaller "
                         "side of your images.")
    if win_size % 2 != 1:
        raise ValueError("Window size must be odd.")
    if data_range is None:
        if im1.dtype == torch.float32:
            raise ValueError("Since skimage 0.18, data_range must be supplied for floating-point inputs.")
        data_range = _INT_DATA_RANGE[im1.dtype]
    taps = _ssim_taps(sigma, truncate) if gaussian_weights else None
    if win_size > MAX_TAPS or (taps is not None and taps.size > MAX_TAPS):
        raise NotImplementedError(f"windows of up to {MAX_TAPS} taps are supported")
    NP = win_size ** ndim
    cov_norm = NP / (NP - 1) if use_sample_covariance else 1.0
    C1 = (K1 * data_range) ** 2
    C2 = (K2 * data_range) ** 2
    require_cuda(im1, "im1")
    require_cuda(im2, "im2")
    if im1.device != im2.device:
        raise ValueError("im1 and im2 must be on the same device")
    if volumetric:
        a, n, d, h, w = as_volumes(im1)
    else:
        a, n, h, w = as_planes(im1)
    b = im2.contiguous()
    code = DTYPE_CODE[a.dtype]
    map_dtype = _float_default(a)
    S = torch.empty(a.shape, dtype=map_dtype, device=a.device) if full else None
    mssim = torch.empty(n, dtype=torch.float64, device=a.device)
    L = lib()
    if volumetric:
        entry, layout = "mie_sk_structural_similarity3d", (*volume_layout(n, d, h, w), d * h * w, h * w, w)
        nbytes = L.mie_sk_structural_similarity3d_workspace_bytes(n, d, h, w, code)
    else:
        entry, layout = "mie_sk_structural_similarity", (*plane_layout(n, h, w), h * w, w)
        nbytes = L.mie_sk_structural_similarity_workspace_bytes(n, h, w, code)
    ws = use_workspace(a.device, nbytes)
    call(a.device, entry, a.data_ptr(), b.data_ptr(), None if S is None else S.data_ptr(), code, _OUT_CODE[map_dtype],
         *layout, win_size, None if taps is None else taps.ctypes.data, 0 if taps is None else taps.size,
         float(cov_norm), float(C1), float(C2), mssim.data_ptr(), ws.data_ptr(), ws.numel())
    lead = tuple(a.shape[:-ndim])
    result = float(mssim.item()) if not lead else mssim.cpu().reshape(lead)
    return (result, S) if full else result


def _denoise_tv_chambolle(image, weight, eps, max_num_iter, channel_axis, out_dtype, volumetric, iters):
    """denoise_tv_chambolle; `iters`: None or a CUDA int32 tensor of one entry per image receiving the passes run."""
    if channel_axis is not None:
        raise NotImplementedError("planes are denoised separately; channel_axis is not supported")
    if not float(weight) > 0.0 or not math.isfinite(float(weight)):
        raise ValueError("weight must be a positive finite number")
    if int(max_num_iter) < 1:
        raise ValueError("max_num_iter must be at least 1")
    L = lib()
    if volumetric:
        x, n, d, h, w = as_volumes(image)
        require_cuda(x)
        entry, layout = "mie_sk_denoise_tv_chambolle3d", volume_layout(n, d, h, w)
        nbytes = L.mie_sk_tv_chambolle3d_workspace_bytes(n, d, h, w, DTYPE_CODE[x.dtype])
    else:
        require_cuda(image)
        x, n, h, w = as_planes(image)
        entry, layout = "mie_sk_denoise_tv_chambolle", plane_layout(n, h, w)
        nbytes = L.mie_sk_tv_chambolle_workspace_bytes(n, h, w, DTYPE_CODE[x.dtype])
    dst = new_out(x, out_dtype, _OUT_CODE, _float_default(x))
    if iters is not None and (iters.dtype != torch.int32 or iters.numel() != n or iters.device != x.device):
        raise ValueError(f"iters must be an int32 tensor of {n} entries on {x.device}")
    ws = use_workspace(x.device, nbytes)
    call(x.device, entry, x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype], *layout, float(weight),
         float(eps), int(max_num_iter), None if iters is None else iters.data_ptr(), ws.data_ptr(), ws.numel())
    return dst


# ---------------------------------------------------------------------------------------------- ridge filters
RIDGE_MAX_RADIUS = 64   # MIE_SK_RIDGE_MAX_RADIUS: sigma < 16 at scipy's truncate of 4
_RIDGE_FILTER = {"frangi": 0, "hessian": 1, "sato": 2, "meijering": 3}


def _gaussian_kernel1d(sigma: float, order: int, radius: int) -> np.ndarray:
    """scipy.ndimage's _gaussian_kernel1d (float64), transcribed so that the taps are scipy's bit for bit."""
    exponent_range = np.arange(order + 1)
    sigma2 = sigma * sigma
    x = np.arange(-radius, radius + 1)
    phi_x = np.exp(-0.5 / sigma2 * x ** 2)
    phi_x = phi_x / phi_x.sum()
    if order == 0:
        return phi_x
    q = np.zeros(order + 1)
    q[0] = 1
    D = np.diag(exponent_range[1:], 1)
    P = np.diag(np.ones(order) / -sigma2, -1)
    Q_deriv = D + P
    for _ in range(order):
        q = Q_deriv.dot(q)
    q = (x[:, None] ** exponent_range).dot(q)
    return q * phi_x


def _hessian_taps(sigma: float):
    """(radius, order-0 taps, order-1 taps) of gaussian_filter(sigma, order, truncate=4.0) in correlation order:
    scipy's gaussian_filter1d correlates with _gaussian_kernel1d(sigma, order, int(4 sigma + 0.5))[::-1]."""
    sigma = float(sigma)
    if sigma < 0.0 or sigma != sigma:
        raise ValueError("Sigma values less than zero are not valid")
    if sigma == 0.0:
        raise NotImplementedError("sigma 0 (scipy then skips the derivative) is not supported")
    r = int(4.0 * sigma + 0.5)
    if r > RIDGE_MAX_RADIUS:
        raise NotImplementedError(f"sigma {sigma} needs a filter radius of {r}; up to {RIDGE_MAX_RADIUS} is supported")
    return r, np.ascontiguousarray(_gaussian_kernel1d(sigma, 0, r)[::-1]), \
        np.ascontiguousarray(_gaussian_kernel1d(sigma, 1, r)[::-1])


def _ridge_border(mode: str) -> int:
    if mode not in SCIPY_MODES:
        raise ValueError(f"mode must be one of {sorted(SCIPY_MODES)}. Got {mode!r}")
    return BORDER[SCIPY_MODES[mode]]


def _ridge_image(image: torch.Tensor, volumetric: bool):
    """-> (dense tensor, n, d, h, w, layout arguments, entry point suffix)."""
    if volumetric:
        x, n, d, h, w = as_volumes(image)
        require_cuda(x)
        return x, n, d, h, w, volume_layout(n, d, h, w), "3d"
    require_cuda(image)
    x, n, h, w = as_planes(image)
    return x, n, 1, h, w, plane_layout(n, h, w), ""


def _ridge(image, name, sigmas, mode, cval, black_ridges, alpha, beta, gamma, out_dtype, volumetric):
    sig = [float(s) for s in np.asarray(sigmas, dtype=np.float64).ravel()]
    if any(s < 0.0 for s in sig):
        raise ValueError("Sigma values less than zero are not valid")
    taps = [_hessian_taps(s) for s in sig]
    border = _ridge_border(mode)
    x, n, d, h, w, layout, nd = _ridge_image(image, volumetric)
    dst = new_out(x, out_dtype, _OUT_CODE, _float_default(x))
    code = DTYPE_CODE[x.dtype]
    L = lib()
    if nd:
        nbytes = L.mie_sk_ridge_filter3d_workspace_bytes(n, d, h, w, code)
    else:
        nbytes = L.mie_sk_ridge_filter_workspace_bytes(n, h, w, code)
    sig_a = np.asarray(sig, np.float64)
    radii = np.asarray([t[0] for t in taps], np.int32)
    t0 = np.concatenate([t[1] for t in taps]) if taps else np.zeros(1)
    t1 = np.concatenate([t[2] for t in taps]) if taps else np.zeros(1)
    ws = use_workspace(x.device, nbytes)
    call(x.device, "mie_sk_ridge_filter" + nd, x.data_ptr(), dst.data_ptr(), code, _OUT_CODE[dst.dtype], *layout,
         _RIDGE_FILTER[name], len(sig), sig_a.ctypes.data, radii.ctypes.data, t0.ctypes.data, t1.ctypes.data, border,
         float(cval), int(bool(black_ridges)), float(alpha), float(beta), -1.0 if gamma is None else abs(float(gamma)),
         ws.data_ptr(), ws.numel())
    return dst


def _scales(sigmas, scale_range, scale_step):
    if scale_range is not None and scale_step is not None:
        return np.arange(scale_range[0], scale_range[1], scale_step)
    return sigmas


def frangi(image: torch.Tensor, sigmas=range(1, 10, 2), scale_range=None, scale_step=None, alpha=0.5, beta=0.5,
           gamma=None, black_ridges=True, mode="reflect", cval=0, *, out_dtype=None,
           volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.frangi on every (H, W) plane of `image` ((H,W), (C,H,W), (B,C,H,W)), each plane one image; with
    volumetric=True on every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor.  gamma=None takes half the
    largest Hessian norm of the first sigma, per image.  Integer images are filtered on their raw values in float64,
    float32 images in float32; returns that float dtype, or `out_dtype` (float64 or float32, rounded once)."""
    return _ridge(image, "frangi", _scales(sigmas, scale_range, scale_step), mode, cval, black_ridges, alpha, beta,
                  gamma, out_dtype, volumetric)


def hessian(image: torch.Tensor, sigmas=range(1, 10, 2), scale_range=None, scale_step=None, alpha=0.5, beta=0.5,
            gamma=15, black_ridges=True, mode="reflect", cval=0, *, out_dtype=None,
            volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.hessian: frangi with gamma=15, then every value <= 0 set to 1.  Layout and dtypes as frangi."""
    return _ridge(image, "hessian", _scales(sigmas, scale_range, scale_step), mode, cval, black_ridges, alpha, beta,
                  gamma, out_dtype, volumetric)


def sato(image: torch.Tensor, sigmas=range(1, 10, 2), black_ridges=True, mode="reflect", cval=0, *, out_dtype=None,
         volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.sato.  Layout and dtypes as frangi."""
    return _ridge(image, "sato", sigmas, mode, cval, black_ridges, 0.0, 0.0, None, out_dtype, volumetric)


def meijering(image: torch.Tensor, sigmas=range(1, 10, 2), alpha=None, black_ridges=True, mode="reflect", cval=0, *,
              out_dtype=None, volumetric: bool = False) -> torch.Tensor:
    """skimage.filters.meijering (alpha=None: 1 / (ndim + 1)); every scale is divided by its own per-image maximum.
    Layout and dtypes as frangi."""
    if alpha is None:
        alpha = 1 / ((3 if volumetric else 2) + 1)
    return _ridge(image, "meijering", sigmas, mode, cval, black_ridges, alpha, 0.0, None, out_dtype, volumetric)


def hessian_matrix(image: torch.Tensor, sigma=1, mode="constant", cval=0, order="rc", use_gaussian_derivatives=None,
                   *, volumetric: bool = False) -> list:
    """skimage.feature.hessian_matrix(..., use_gaussian_derivatives=True) of every plane (or, volumetric=True, every
    volume): [H00, H01, H11] or [H00, H01, H02, H11, H12, H22], CUDA tensors of the input's shape on the img_as_float
    scale (float64 for integer input, float32 for float32), bit-exact against scipy.ndimage's arithmetic."""
    if use_gaussian_derivatives is not True:
        raise NotImplementedError("only use_gaussian_derivatives=True is built (the np.gradient path is not)")
    if order == "xy":
        raise NotImplementedError("order='xy' is not supported")
    if order != "rc":
        raise ValueError("order must be 'rc' or 'xy'")
    if isinstance(sigma, (tuple, list)):
        raise NotImplementedError("one sigma for every axis is supported")
    r, t0, t1 = _hessian_taps(sigma)
    border = _ridge_border(mode)
    x, n, d, h, w, layout, nd = _ridge_image(image, volumetric)
    ndim = 3 if nd else 2
    dt = _float_default(x)
    out = torch.empty((ndim * (ndim + 1) // 2, *x.shape), dtype=dt, device=x.device)
    code = DTYPE_CODE[x.dtype]
    L = lib()
    if nd:
        nbytes = L.mie_sk_hessian_matrix3d_workspace_bytes(n, d, h, w, code)
    else:
        nbytes = L.mie_sk_hessian_matrix_workspace_bytes(n, h, w, code)
    ws = use_workspace(x.device, nbytes)
    call(x.device, "mie_sk_hessian_matrix" + nd, x.data_ptr(), out.data_ptr(), code, _OUT_CODE[dt], *layout,
         x.numel(), r, t0.ctypes.data, t1.ctypes.data, border, float(cval), ws.data_ptr(), ws.numel())
    return list(out.unbind(0))


def hessian_matrix_eigvals(H_elems) -> torch.Tensor:
    """skimage.feature.hessian_matrix_eigvals: the eigenvalues of every voxel in decreasing order, a CUDA tensor of
    shape (ndim, *H_elems[0].shape).  3 elements: 2-D (upstream's closed form, bit-exact); 6: 3-D (cyclic Jacobi in
    float64, rounded to the elements' dtype)."""
    H_elems = list(H_elems)
    ndim = {3: 2, 6: 3}.get(len(H_elems))
    if ndim is None:
        raise ValueError(f"expected the 3 (2-D) or 6 (3-D) Hessian elements; got {len(H_elems)}")
    first = H_elems[0]
    for t in H_elems:
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype not in (torch.float32, torch.float64):
            raise TypeError("H_elems must be float32 or float64 CUDA tensors")
        if t.shape != first.shape or t.dtype != first.dtype or t.device != first.device:
            raise ValueError("H_elems must share shape, dtype and device")
    h = torch.stack([t.contiguous() for t in H_elems])
    eig = torch.empty((ndim, *first.shape), dtype=first.dtype, device=first.device)
    count = first.numel()
    call(first.device, "mie_sk_hessian_eigvals", h.data_ptr(), eig.data_ptr(), _OUT_CODE[first.dtype], ndim, count,
         count, count)
    return eig
