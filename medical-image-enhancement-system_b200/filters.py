"""Denoising / sharpening operators with kornia's (and, for N-D median, skimage's)
call signatures, backed by the sm_100a kernels behind include/mie.h.

  gaussian_blur2d, unsharp_mask, median_blur, bilateral_blur
      <- kornia.filters.*            (reference pyproject.toml:8;  SURVEY.md §8(a) A3,A4,A5,A7)
  median
      <- skimage.filters.median      (reference pyproject.toml:12; SURVEY.md §8(a) A6), any footprint and scipy mode

Integer tensors are accepted directly (see enhance.py for the mapping rule).
"""
from __future__ import annotations

import math

import numpy as np
import torch

from ._ffi import (BORDER, DTYPE_CODE, MIE_F64, SCIPY_MODES, as_planes, call, check_out, new_out, plane_layout,
                   require_cuda, value_range_of, volume_layout)

__all__ = ["get_gaussian_kernel1d", "gaussian_blur2d", "unsharp_mask", "median_blur", "bilateral_blur", "median"]

MAX_TAPS = 33


def get_gaussian_kernel1d(kernel_size: int, sigma: float) -> np.ndarray:
    """kornia.filters.get_gaussian_kernel1d: x = arange(K) - K//2 (+0.5 when K is
    even); exp(-x^2 / (2 sigma^2)) normalised to sum 1.  Evaluated in float64 on the
    host and rounded once to float32 (the weights are kernel parameters)."""
    k = int(kernel_size)
    if k <= 0:
        raise TypeError(f"kernel_size must be a positive integer. Got {kernel_size}")
    x = np.arange(k, dtype=np.float64) - k // 2
    if k % 2 == 0:
        x = x + 0.5
    g = np.exp(-(x * x) / (2.0 * float(sigma) ** 2))
    return np.ascontiguousarray((g / g.sum()).astype(np.float32))


def _pair_int(v, name):
    if isinstance(v, (tuple, list)):
        if len(v) != 2:
            raise TypeError(f"{name} must be an int or a pair. Got {v}")
        a, b = int(v[0]), int(v[1])
    else:
        a = b = int(v)
    return a, b


def _pair_float(v, name):
    if isinstance(v, torch.Tensor):
        v = v.detach().flatten().tolist()
        if len(v) == 1:
            v = v[0]
        elif len(v) != 2:
            raise NotImplementedError(f"per-sample {name} tensors are not supported; pass a float or a (y, x) pair")
    if isinstance(v, (tuple, list)):
        if len(v) != 2:
            raise TypeError(f"{name} must be a float or a pair. Got {v}")
        return float(v[0]), float(v[1])
    return float(v), float(v)


def _check_kernel(ky, kx):
    for k in (ky, kx):
        if k <= 0 or k % 2 == 0:
            raise ValueError(f"kernel_size must be odd and positive. Got {(ky, kx)}")
        if k > MAX_TAPS:
            raise ValueError(f"kernel_size up to {MAX_TAPS} is supported. Got {(ky, kx)}")


def _border(border_type: str) -> int:
    if border_type not in BORDER:
        raise ValueError(f"border_type must be one of {sorted(BORDER)}. Got {border_type}")
    return BORDER[border_type]


def _separable(fn_name, input, kernel_size, sigma, border_type, value_range, out_dtype):
    ky, kx = _pair_int(kernel_size, "kernel_size")
    _check_kernel(ky, kx)
    sy, sx = _pair_float(sigma, "sigma")
    _border(border_type)
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    wx, wy = get_gaussian_kernel1d(kx, sx), get_gaussian_kernel1d(ky, sy)
    call(x.device, fn_name, x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), wx.ctypes.data, kx, wy.ctypes.data, ky, _border(border_type), lo, hi)
    return dst


def gaussian_blur2d(input: torch.Tensor, kernel_size, sigma, border_type: str = "reflect", separable: bool = True,
                    *, value_range=None, out_dtype=None) -> torch.Tensor:
    """kornia.filters.gaussian_blur2d.  kernel_size (ky, kx) and sigma (sy, sx) as in kornia.
    `separable=False` computes the same separable result (a Gaussian is rank 1)."""
    return _separable("mie_gaussian2d", input, kernel_size, sigma, border_type, value_range, out_dtype)


def unsharp_mask(input: torch.Tensor, kernel_size, sigma, border_type: str = "reflect", *, value_range=None,
                 out_dtype=None) -> torch.Tensor:
    """kornia.filters.unsharp_mask: input + (input - gaussian_blur2d(input))."""
    return _separable("mie_unsharp", input, kernel_size, sigma, border_type, value_range, out_dtype)


def median_blur(input: torch.Tensor, kernel_size, *, border_type: str = "constant") -> torch.Tensor:
    """kornia.filters.median_blur: zero-padded window, lower median; same dtype out.
    border_type='replicate' gives skimage/scipy 'nearest' and cv2.medianBlur borders."""
    require_cuda(input)
    ky, kx = _pair_int(kernel_size, "kernel_size")
    x, n, h, w = as_planes(input)
    dst = torch.empty_like(x)
    call(x.device, "mie_median2d", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(n, h, w), ky, kx,
         _border(border_type))
    return dst


def bilateral_blur(input: torch.Tensor, kernel_size, sigma_color, sigma_space, border_type: str = "reflect",
                   color_distance_type: str = "l1", *, value_range=None, out_dtype=None) -> torch.Tensor:
    """kornia.filters.bilateral_blur on single-channel planes ('l1' and 'l2' coincide
    for one channel; multi-channel inputs are filtered per channel)."""
    if color_distance_type not in ("l1", "l2"):
        raise ValueError("color_distance_type only accepts l1 or l2")
    require_cuda(input)
    ky, kx = _pair_int(kernel_size, "kernel_size")
    _check_kernel(ky, kx)
    sy, sx = _pair_float(sigma_space, "sigma_space")
    if isinstance(sigma_color, torch.Tensor):
        sigma_color = float(sigma_color.flatten()[0])
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    wsp = np.ascontiguousarray(
        (get_gaussian_kernel1d(ky, sy)[:, None] * get_gaussian_kernel1d(kx, sx)[None, :]).astype(np.float32))
    call(x.device, "mie_bilateral", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), wsp.ctypes.data, ky, kx, float(sigma_color), _border(border_type), lo, hi)
    return dst


def denoise_nl_means(image: torch.Tensor, patch_size: int = 7, patch_distance: int = 11, h: float = 0.1,
                     channel_axis=None, fast_mode: bool = True, sigma: float = 0.0, *, preserve_range: bool = False,
                     value_range=None, out_dtype=None) -> torch.Tensor:
    """skimage.restoration.denoise_nl_means on 2-D planes ((H,W), (C,H,W), (B,C,H,W): every plane is
    filtered on its own).  `fast_mode=True` (default): uniform patch weights, separable sliding sums, fp32 (within
    rel 1e-5 of the float64 oracle).  `fast_mode=False`: upstream's slow mode — Gaussian patch weights, search window
    clipped at the image, cut-off test before every patch row — in float64 and upstream's operation order;
    out_dtype may then also be torch.float64 (what skimage returns for integer images).  `h` and `sigma`
    are on the [0,1] scale of the normalised image, as in skimage after img_as_float; integer tensors
    use this package's normalisation (value_range, default the dtype's range) and come back in the same
    dtype unless out_dtype says otherwise.  `preserve_range` is accepted for signature compatibility and
    only meaningful for float tensors (which are never rescaled here)."""
    if channel_axis is not None:
        raise NotImplementedError("multichannel non-local means is not supported (planes are filtered separately)")
    require_cuda(image)
    x, n, hh, ww = as_planes(image)
    lo, hi = value_range_of(x, value_range)
    if not fast_mode:
        dst = new_out(x, out_dtype, (x.dtype, torch.float32, torch.float64))
        code = MIE_F64 if dst.dtype == torch.float64 else DTYPE_CODE[dst.dtype]
        call(x.device, "mie_nlm_slow", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], code, *plane_layout(n, hh, ww),
             int(patch_size), int(patch_distance), float(h), float(sigma), lo, hi)
        return dst
    dst = new_out(x, out_dtype)
    call(x.device, "mie_nlm", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, hh, ww), int(patch_size), int(patch_distance), float(h), float(sigma), lo, hi)
    return dst


MEDIAN_MAX_EXTENT = {2: 65, 3: 17}   # MIE_SK_MEDIAN_MAX_EXTENT, MIE_SK_MEDIAN3D_MAX_EXTENT (include/mie.h)
_INT_RANGE = {torch.uint8: (0, 255), torch.uint16: (0, 65535), torch.int16: (-32768, 32767)}


def median_cval(dtype: torch.dtype, cval, two_cell_box: bool = False) -> float:
    """`cval` cast to the image dtype the way scipy.ndimage.median_filter casts it (checked against scipy 1.18.1):
    float32 images round it to float32 (1e300 -> inf); integer images truncate it towards zero to a 32-bit integer
    and keep its low bits (uint8: 300 -> 44, -1 -> 255; int16: -2.5 -> -2), before selection.  Outside the 32-bit
    range, or not finite, scipy's result is the platform's out-of-range conversion: NotImplementedError.
    `two_cell_box`: a footprint of two set cells and no unset one.  scipy then runs its separable maximum filter, which
    compares the double cval and casts the result: a cval below the dtype's range never wins (the dtype minimum
    does the same), and one above it is NotImplementedError (the cast result does not depend on the pixels)."""
    c = float(cval)
    if dtype == torch.float32:
        with np.errstate(over="ignore"):
            return float(np.float32(c))
    lo, hi = _INT_RANGE[dtype]
    if not math.isfinite(c) or not -2.0 ** 31 <= math.trunc(c) < 2.0 ** 31:
        raise NotImplementedError(f"cval {cval!r} is outside the 32-bit range: scipy's cast of it to {dtype} is "
                                  "platform-defined")
    if two_cell_box:
        if c > hi:
            raise NotImplementedError(f"cval {cval!r} above the {dtype} range with a two-cell footprint is not supported")
        return float(max(math.trunc(c), lo))
    return float((math.trunc(c) - lo) % (hi - lo + 1) + lo)


def _as_footprint(footprint) -> np.ndarray:
    if isinstance(footprint, torch.Tensor):
        footprint = footprint.detach().cpu().numpy()
    return np.ascontiguousarray(np.asarray(footprint, dtype=bool))


def median(image: torch.Tensor, footprint=None, out=None, mode: str = "nearest", cval: float = 0.0,
           behavior: str = "ndimage", *, halo_lo=None, halo_hi=None, peer_halos: bool = False) -> torch.Tensor:
    """skimage.filters.median on a 2-D image or a 3-D volume -> scipy.ndimage.median_filter(image, footprint, mode=mode,
    cval=cval): element count // 2 of the sorted window.  `footprint`: None (all-ones 3^ndim), or any numpy array,
    torch tensor or nested list of the image's ndim, extents up to 65 (planes) or 17 (volumes); e.g.
    skimage_compat.disk(r) / ball(r).  Modes 'nearest', 'reflect', 'mirror', 'wrap' and 'constant' (cval cast as
    median_cval describes).

    The default footprint in 'nearest', or in 'constant' with cval 0, runs mie_median2d / mie_median3d; every other
    call runs mie_sk_median / mie_sk_median3d.  `halo_lo` / `halo_hi` (default footprint only): the neighbouring
    slab's boundary plane when the volume is one z-slab of a sharded volume (see volume.py); with `peer_halos=True`
    they may live on another GPU of the box (the neighbour rank's slab mapped by CUDA IPC: the kernel reads them over
    NVLink)."""
    require_cuda(image)
    if behavior != "ndimage":
        raise NotImplementedError("behavior='rank' is not supported")
    if mode not in SCIPY_MODES:
        raise NotImplementedError(f"mode {mode!r} is not supported ({', '.join(SCIPY_MODES)})")
    if image.dim() not in (2, 3):
        raise ValueError("median expects a 2-D image or a 3-D volume")
    ndim = image.dim()
    box3 = footprint is None
    if not box3:
        fp = _as_footprint(footprint)
        if fp.ndim != ndim:
            raise RuntimeError(f"footprint.ndim ({fp.ndim}) must match len(axes) ({ndim})")
        count = int(fp.sum())
        if count == 0:
            raise RuntimeError("rank not within filter footprint size")
        if max(fp.shape) > MEDIAN_MAX_EXTENT[ndim]:
            raise NotImplementedError(f"footprint extents up to {MEDIAN_MAX_EXTENT[ndim]} are supported for a {ndim}-D "
                                      f"image; got {fp.shape}")
        box3 = fp.shape == (3,) * ndim and count == fp.size
        if mode == "reflect" and any(1 < n <= e // 8 for n, e in zip(image.shape, fp.shape)):
            # scipy maps offset -2 n m (m >= 2) of an axis of length n to index -1 in 'reflect' mode and reads memory
            # outside the image there
            raise NotImplementedError(f"mode 'reflect' with footprint {fp.shape} reaches 4 times beyond an axis of "
                                      f"image {tuple(image.shape)}, where scipy's result is undefined")
    cv = 0.0
    if mode == "constant":
        cv = median_cval(image.dtype, cval, not box3 and count == 2 and count == fp.size)
    default = box3 and (mode == "nearest" or (mode == "constant" and cv == 0.0))
    x = image.contiguous()
    dst = torch.empty_like(x) if out is None else check_out(x, out, (x.dtype,))
    if out is not None and out.untyped_storage().data_ptr() == x.untyped_storage().data_ptr():
        lo, hi = max(out.data_ptr(), x.data_ptr()), min(out.data_ptr() + out.numel() * out.element_size(),
                                                        x.data_ptr() + x.numel() * x.element_size())
        if lo < hi:
            raise ValueError("out must not overlap the input: the median kernels read neighbours they have not written yet")
    border = BORDER[SCIPY_MODES[mode]]
    if not default:
        if halo_lo is not None or halo_hi is not None or peer_halos:
            raise NotImplementedError("slab halos are supported with the default footprint only")
        fp8 = np.ones((3,) * ndim, np.uint8) if footprint is None else fp.astype(np.uint8)
        if ndim == 2:
            call(x.device, "mie_sk_median", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(1, *x.shape),
                 fp8.ctypes.data, *fp8.shape, border, cv)
        else:
            call(x.device, "mie_sk_median3d", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype],
                 *volume_layout(1, *x.shape), fp8.ctypes.data, *fp8.shape, border, cv)
        return dst
    if x.dim() == 2:
        call(x.device, "mie_median2d", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(1, *x.shape),
             3, 3, border)
    else:
        d, h, w = x.shape
        for hp in (halo_lo, halo_hi):
            if hp is not None and (hp.shape != (h, w) or hp.dtype != x.dtype or not hp.is_contiguous()
                                   or (hp.device != x.device and not (peer_halos and hp.is_cuda))):
                raise ValueError("halo planes must be contiguous (H, W) tensors of the volume's dtype on its device")
        # one volume of d dense planes: mie_median3d takes (d, h, w) and the plane strides
        call(x.device, "mie_median3d", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(d, h, w),
             halo_lo.data_ptr() if halo_lo is not None else None, halo_hi.data_ptr() if halo_hi is not None else None,
             border)
    return dst
