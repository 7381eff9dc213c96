"""Denoising / sharpening operators with kornia's (and, for N-D median, skimage's)
call signatures, backed by the sm_100a kernels behind include/mie.h.

  gaussian_blur2d, unsharp_mask, median_blur, bilateral_blur
      <- kornia.filters.*            (reference pyproject.toml:8;  SURVEY.md §8(a) A3,A4,A5,A7)
  median
      <- skimage.filters.median      (reference pyproject.toml:12; SURVEY.md §8(a) A6)

Integer tensors are accepted directly (see enhance.py for the mapping rule).
"""
from __future__ import annotations

import numpy as np
import torch

from ._ffi import (BORDER, DTYPE_CODE, MIE_F64, as_planes, call, check_out, new_out, plane_layout, require_cuda,
                   value_range_of)

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


_MEDIAN_MODES = {"nearest": "replicate", "constant": "constant"}


def median(image: torch.Tensor, footprint=None, out=None, mode: str = "nearest", cval: float = 0.0,
           behavior: str = "ndimage", *, halo_lo=None, halo_hi=None, peer_halos: bool = False) -> torch.Tensor:
    """skimage.filters.median on a 2-D image (3x3 default) or 3-D volume (3x3x3 default)
    -> scipy.ndimage.median_filter semantics (rank n//2).  Footprints: None or an all-ones
    box of the default size.  `halo_lo` / `halo_hi`: the neighbouring slab's boundary
    plane when the volume is one z-slab of a sharded volume (see volume.py); with `peer_halos=True` they may live on
    another GPU of the box (the neighbour rank's slab mapped by CUDA IPC: the kernel reads them over NVLink)."""
    require_cuda(image)
    if behavior != "ndimage":
        raise NotImplementedError("behavior='rank' is not supported")
    if mode not in _MEDIAN_MODES:
        raise NotImplementedError(f"mode {mode!r} is not supported (nearest, constant)")
    if mode == "constant" and cval != 0.0:
        raise NotImplementedError("constant mode supports cval=0 only")
    if image.dim() not in (2, 3):
        raise ValueError("median expects a 2-D image or a 3-D volume")
    if footprint is not None:
        fp = np.asarray(footprint.cpu() if isinstance(footprint, torch.Tensor) else footprint)
        if fp.shape != (3,) * image.dim() or not fp.all():
            raise NotImplementedError("only the default all-ones 3^ndim footprint is supported")
    border = BORDER[_MEDIAN_MODES[mode]]
    x = image.contiguous()
    dst = torch.empty_like(x) if out is None else check_out(x, out, (x.dtype,))
    if out is not None and out.untyped_storage().data_ptr() == x.untyped_storage().data_ptr():
        lo, hi = max(out.data_ptr(), x.data_ptr()), min(out.data_ptr() + out.numel() * out.element_size(),
                                                        x.data_ptr() + x.numel() * x.element_size())
        if lo < hi:
            raise ValueError("out must not overlap the input: the median kernels read neighbours they have not written yet")
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
