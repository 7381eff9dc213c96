"""scikit-image call signatures over the same sm_100a kernels (SURVEY.md §2.2, §8(f) F3).

scikit-image >= 0.26.0 is the reference's second image-processing dependency (reference
pyproject.toml:12, pin uv.lock:619-650).  Its filters delegate to scipy.ndimage, whose Gaussian is the
kornia Gaussian with K = 2*int(truncate*sigma + 0.5) + 1 taps
(site-packages/scipy/ndimage/_filters.py:656-669, 745-747) and whose border modes map onto the ABI's:

    scipy / skimage mode   'nearest'    'reflect'     'mirror'    'constant'   'wrap'
    include/mie.h          REPLICATE    SYMMETRIC     REFLECT     CONSTANT     CIRCULAR

    gaussian(image, sigma, mode=, truncate=)            <- skimage.filters.gaussian
    unsharp_mask(image, radius, amount, preserve_range) <- skimage.filters.unsharp_mask
    median(image, ...)                                  <- skimage.filters.median           (filters.py)
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
"""
from __future__ import annotations

import math

import numpy as np
import torch

from ._ffi import BORDER, DTYPE_CODE, MIE_F32, MIE_F64, as_planes, check, lib, require_cuda, stream_ptr, value_range_of
from .filters import MAX_TAPS, _out_like, denoise_nl_means, gaussian_blur2d, get_gaussian_kernel1d, median  # noqa: F401

__all__ = ["gaussian", "unsharp_mask", "median", "denoise_nl_means", "SCIPY_MODES", "equalize_adapthist", "equalize_hist",
           "denoise_bilateral", "denoise_tv_chambolle"]

SCIPY_MODES = {"nearest": "replicate", "reflect": "symmetric", "mirror": "reflect", "constant": "constant",
               "wrap": "circular"}


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
    dst = _out_like(x, out_dtype)
    wk = get_gaussian_kernel1d(k, float(radius))
    with torch.cuda.device(x.device):
        check(lib().mie_unsharp_amount(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype], n, h, w,
                                       h * w, w, h * w, w, wk.ctypes.data, k, wk.ctypes.data, k, BORDER["symmetric"],
                                       float(amount), 0 if preserve_range else 1, lo, hi, stream_ptr(x.device)))
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


def _check_volume(image) -> None:
    if not isinstance(image, torch.Tensor):
        raise TypeError(f"input must be a torch.Tensor, got {type(image)}")
    if not 3 <= image.dim() <= 5:
        raise ValueError(f"volumetric=True expects (D,H,W), (B,D,H,W) or (B,C,D,H,W); got shape {tuple(image.shape)}")


def _gaussian3d(image: torch.Tensor, sigma, border: str, truncate, value_range, out_dtype, unsharp) -> torch.Tensor:
    """mie_gaussian3d / mie_unsharp3d (unsharp = (amount, clip)) on every (D, H, W) volume of `image`."""
    _check_volume(image)
    if isinstance(sigma, (tuple, list)):
        if len(sigma) != 3:
            raise ValueError(f"volumetric=True takes a scalar sigma or (sigma_z, sigma_y, sigma_x); got {sigma!r}")
        sz, sy, sx = sigma
    else:
        sz = sy = sx = sigma
    wz, wy, wx = (_axis_weights(s, truncate) for s in (sz, sy, sx))
    require_cuda(image)
    x = image.contiguous()
    d, h, w = (int(s) for s in x.shape[-3:])
    n = x.numel() // (d * h * w) if d * h * w else 0
    lo, hi = value_range_of(x, value_range)
    dst = _out_like(x, out_dtype)
    args = (x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype], n, d, h, w, d * h * w, h * w, w,
            d * h * w, h * w, w, wx.ctypes.data, wx.size, wy.ctypes.data, wy.size, wz.ctypes.data, wz.size, BORDER[border])
    with torch.cuda.device(x.device):
        if unsharp is None:
            check(lib().mie_gaussian3d(*args, lo, hi, stream_ptr(x.device)))
        else:
            check(lib().mie_unsharp3d(*args, unsharp[0], unsharp[1], lo, hi, stream_ptr(x.device)))
    return dst


# ---------------------------------------------------------------------------------------------- exposure / restoration
_OUT_CODE = {torch.float32: MIE_F32, torch.float64: MIE_F64}
_PAD_MODES = {"constant": 0, "edge": 1, "symmetric": 2, "reflect": 3, "wrap": 4}


def _sk_out(x: torch.Tensor, out_dtype, default):
    dt = default if out_dtype is None else out_dtype
    if dt not in _OUT_CODE:
        raise TypeError("out_dtype must be torch.float32 or torch.float64")
    return torch.empty(x.shape, dtype=dt, device=x.device)


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
    dst = _sk_out(x, out_dtype, torch.float32 if x.dtype == torch.float32 else torch.float64)
    L = lib()
    ws = torch.empty(max(L.mie_sk_adapthist_workspace_bytes(n, h, w, kr, kc, int(nbins)), 1), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(L.mie_sk_equalize_adapthist(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype], n, h, w,
                                          h * w, w, h * w, w, kr, kc, float(clip_limit), int(nbins), ws.data_ptr(), ws.numel(),
                                          stream_ptr(x.device)))
    return dst


def _equalize_adapthist3d(image: torch.Tensor, kernel_size, clip_limit, nbins, out_dtype) -> torch.Tensor:
    if not isinstance(image, torch.Tensor):
        raise TypeError(f"input must be a torch.Tensor, got {type(image)}")
    if not 3 <= image.dim() <= 5:
        raise ValueError(f"volumetric=True expects (D,H,W), (B,D,H,W) or (B,C,D,H,W); got shape {tuple(image.shape)}")
    d, h, w = (int(s) for s in image.shape[-3:])
    kd, kr, kc = _sk_kernel_size((d, h, w), kernel_size)
    if kd <= 0 or kr <= 0 or kc <= 0:
        raise ValueError("kernel_size entries must be positive")
    if not 0 < int(nbins) <= 4096:
        raise NotImplementedError("nbins must be in 1..4096")
    require_cuda(image)
    x = image.contiguous()
    n = x.numel() // (d * h * w) if d * h * w else 0
    dst = _sk_out(x, out_dtype, torch.float32 if x.dtype == torch.float32 else torch.float64)
    L = lib()
    ws = torch.empty(max(L.mie_sk_adapthist3d_workspace_bytes(n, d, h, w, kd, kr, kc, int(nbins)), 1), dtype=torch.uint8,
                     device=x.device)
    with torch.cuda.device(x.device):
        check(L.mie_sk_equalize_adapthist3d(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype], n, d, h,
                                            w, d * h * w, h * w, w, d * h * w, h * w, w, kd, kr, kc, float(clip_limit),
                                            int(nbins), ws.data_ptr(), ws.numel(), stream_ptr(x.device)))
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
    dst = _sk_out(x, out_dtype, torch.float64)
    L = lib()
    ws = torch.empty(max(L.mie_sk_equalize_hist_workspace_bytes(n, DTYPE_CODE[x.dtype]), 1), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(L.mie_sk_equalize_hist(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype], n, h, w,
                                     h * w, w, h * w, w, ws.data_ptr(), ws.numel(), stream_ptr(x.device)))
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
    dst = _sk_out(x, out_dtype, torch.float64)
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
    with torch.cuda.device(x.device):
        check(lib().mie_sk_denoise_bilateral(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype], n, h, w,
                                             h * w, w, h * w, w, win_size, int(bins), _PAD_MODES[mode], float(cval),
                                             d_luts.data_ptr(), d_spatial.data_ptr(), ranges.data_ptr(), stream_ptr(x.device)))
    return dst


def denoise_tv_chambolle(image: torch.Tensor, weight: float = 0.1, eps: float = 2e-4, max_num_iter: int = 200, *,
                         channel_axis=None, out_dtype=None, volumetric: bool = False) -> torch.Tensor:
    """skimage.restoration.denoise_tv_chambolle on every (H, W) plane of `image` ((H,W), (C,H,W), (B,C,H,W)), each
    plane one 2-D image with its own energy and stopping point.

    volumetric=True: every (D, H, W) volume of a (D,H,W), (B,D,H,W) or (B,C,D,H,W) tensor is one 3-D image, as skimage
    treats a 3-D array.  Integer images are computed in float64 on the img_as_float scale, float32 images in float32;
    returns that float dtype, or `out_dtype`.  The iteration runs on the device with no host synchronisation."""
    return _denoise_tv_chambolle(image, weight, eps, max_num_iter, channel_axis, out_dtype, volumetric, None)


def _denoise_tv_chambolle(image, weight, eps, max_num_iter, channel_axis, out_dtype, volumetric, iters):
    """denoise_tv_chambolle; `iters`: None or a CUDA int32 tensor of one entry per image receiving the passes run."""
    if channel_axis is not None:
        raise NotImplementedError("planes are denoised separately; channel_axis is not supported")
    if not float(weight) > 0.0 or not math.isfinite(float(weight)):
        raise ValueError("weight must be a positive finite number")
    if int(max_num_iter) < 1:
        raise ValueError("max_num_iter must be at least 1")
    if volumetric:
        _check_volume(image)
    require_cuda(image)
    L = lib()
    if volumetric:
        x = image.contiguous()
        d, h, w = (int(s) for s in x.shape[-3:])
        n = x.numel() // (d * h * w) if d * h * w else 0
        nbytes = L.mie_sk_tv_chambolle3d_workspace_bytes(n, d, h, w, DTYPE_CODE[x.dtype])
    else:
        x, n, h, w = as_planes(image)
        nbytes = L.mie_sk_tv_chambolle_workspace_bytes(n, h, w, DTYPE_CODE[x.dtype])
    dst = _sk_out(x, out_dtype, torch.float32 if x.dtype == torch.float32 else torch.float64)
    if iters is not None and (iters.dtype != torch.int32 or iters.numel() != n or iters.device != x.device):
        raise ValueError(f"iters must be an int32 tensor of {n} entries on {x.device}")
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=x.device)
    it = None if iters is None else iters.data_ptr()
    with torch.cuda.device(x.device):
        if volumetric:
            check(L.mie_sk_denoise_tv_chambolle3d(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
                                                  n, d, h, w, d * h * w, h * w, w, d * h * w, h * w, w, float(weight),
                                                  float(eps), int(max_num_iter), it, ws.data_ptr(), ws.numel(),
                                                  stream_ptr(x.device)))
        else:
            check(L.mie_sk_denoise_tv_chambolle(x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], _OUT_CODE[dst.dtype],
                                                n, h, w, h * w, w, h * w, w, float(weight), float(eps), int(max_num_iter),
                                                it, ws.data_ptr(), ws.numel(), stream_ptr(x.device)))
    return dst
