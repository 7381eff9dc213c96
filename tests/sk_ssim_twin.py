"""numpy twin of skimage.metrics.structural_similarity — TEST INFRASTRUCTURE ONLY (never imported by the package).

**RECALLED**: `structural_similarity` is a literal transcription of upstream's function (0.26,
skimage/metrics/_structural_similarity.py) as the author remembers it, on scipy.ndimage; scikit-image is not installable
here, so nothing in it is pinned against upstream until tests/test_sk_ssim.py::test_live_pin_against_skimage can run.
Integer images are used with their raw values as float64 (not img_as_float); float32 images stay float32, and NumPy 2's
weak Python scalars then round cov_norm, C1 and C2 to float32 as upstream's arithmetic does.

`uniform_line` / `gaussian_line` transcribe scipy.ndimage's 1-D line loops (uniform_filter1d, gaussian_filter1d with
mode='reflect'), vectorised over every other axis: the arithmetic csrc/sk_ssim.cu implements.  `filter_axes` runs them
along axis 0, 1, 2 with the values rounded to the array's dtype between passes, as scipy's N-D filters do."""
from __future__ import annotations

import numpy as np
from scipy.ndimage import gaussian_filter, uniform_filter

TRUNCATE = 3.5
DTYPE_RANGE = {np.uint8: (0, 255), np.uint16: (0, 65535), np.int16: (-32768, 32767)}


def gaussian_weights(sigma: float, truncate: float = TRUNCATE) -> np.ndarray:
    """scipy's _gaussian_kernel1d(sigma, 0, int(truncate * sigma + 0.5)) in float64."""
    r = int(truncate * float(sigma) + 0.5)
    x = np.arange(-r, r + 1)
    phi = np.exp(-0.5 / (float(sigma) * float(sigma)) * x ** 2)
    return phi / phi.sum()


def _extended(x: np.ndarray, axis: int, before: int, after: int) -> np.ndarray:
    """The line extended in 'reflect' mode (d c b a | a b c d | d c b a, repeated as needed), as float64, axis first."""
    n = x.shape[axis]
    idx = np.arange(-before, n + after) % (2 * n)
    idx = np.where(idx < n, idx, 2 * n - 1 - idx)
    return np.moveaxis(np.take(x, idx, axis=axis).astype(np.float64), axis, 0)


def uniform_line(x: np.ndarray, size: int, axis: int = -1) -> np.ndarray:
    """uniform_filter1d(x, size, axis, mode='reflect') for odd size: running sum in float64, cast to x's dtype."""
    r = size // 2
    n = x.shape[axis]
    ext = _extended(x, axis, r, r)
    out = np.empty((n,) + ext.shape[1:], np.float64)
    tmp = np.zeros(ext.shape[1:], np.float64)
    for j in range(size):
        tmp = tmp + ext[j]
    out[0] = tmp / size
    for i in range(1, n):
        tmp = tmp + (ext[i + size - 1] - ext[i - 1])
        out[i] = tmp / size
    return np.moveaxis(out, 0, axis).astype(x.dtype)


def gaussian_line(x: np.ndarray, weights: np.ndarray, axis: int = -1) -> np.ndarray:
    """gaussian_filter1d(x, sigma, axis, mode='reflect') given its symmetric float64 weights: scipy's symmetric
    correlation tmp = ext[c] w[r]; tmp += (ext[c + j] + ext[c - j]) w[j + r] for j = -r .. -1, cast to x's dtype."""
    r = weights.size // 2
    n = x.shape[axis]
    ext = _extended(x, axis, r, r)
    out = np.empty((n,) + ext.shape[1:], np.float64)
    for i in range(n):
        c = i + r
        tmp = ext[c] * weights[r]
        for j in range(-r, 0):
            tmp = tmp + (ext[c + j] + ext[c - j]) * weights[j + r]
        out[i] = tmp
    return np.moveaxis(out, 0, axis).astype(x.dtype)


def filter_axes(x: np.ndarray, line, *args) -> np.ndarray:
    """The 1-D filter along axis 0, then 1, ... — values in x's dtype between passes."""
    for ax in range(x.ndim):
        x = line(x, *args, axis=ax)
    return x


def structural_similarity(im1, im2, *, win_size=None, data_range=None, gaussian_weights=False, full=False, **kwargs):
    """-> mssim, or (mssim, S) with full=True.  Single-channel, no gradient: the subset the package implements."""
    im1, im2 = np.asarray(im1), np.asarray(im2)
    if im1.shape != im2.shape:
        raise ValueError("Input images must have the same dimensions.")
    K1 = kwargs.pop("K1", 0.01)
    K2 = kwargs.pop("K2", 0.03)
    sigma = kwargs.pop("sigma", 1.5)
    if K1 < 0:
        raise ValueError("K1 must be positive")
    if K2 < 0:
        raise ValueError("K2 must be positive")
    if sigma < 0:
        raise ValueError("sigma must be positive")
    use_sample_covariance = kwargs.pop("use_sample_covariance", True)

    if gaussian_weights:
        truncate = TRUNCATE
    if win_size is None:
        if gaussian_weights:
            r = int(truncate * sigma + 0.5)
            win_size = 2 * r + 1
        else:
            win_size = 7

    if np.any((np.asarray(im1.shape) - win_size) < 0):
        raise ValueError("win_size exceeds image extent.")
    if not (win_size % 2 == 1):
        raise ValueError("Window size must be odd.")

    if data_range is None:
        if np.issubdtype(im1.dtype, np.floating):
            raise ValueError("data_range must be supplied for floating-point inputs.")
        dmin, dmax = DTYPE_RANGE[im1.dtype.type]
        data_range = dmax - dmin

    ndim = im1.ndim
    if gaussian_weights:
        def filter_func(x):
            return gaussian_filter(x, sigma, mode="reflect", truncate=truncate)
    else:
        def filter_func(x):
            return uniform_filter(x, size=win_size)

    float_type = np.float32 if im1.dtype == np.float32 else np.float64
    im1 = im1.astype(float_type, copy=False)
    im2 = im2.astype(float_type, copy=False)

    NP = win_size ** ndim
    if use_sample_covariance:
        cov_norm = NP / (NP - 1)
    else:
        cov_norm = 1.0

    ux = filter_func(im1)
    uy = filter_func(im2)
    uxx = filter_func(im1 * im1)
    uyy = filter_func(im2 * im2)
    uxy = filter_func(im1 * im2)
    vx = cov_norm * (uxx - ux * ux)
    vy = cov_norm * (uyy - uy * uy)
    vxy = cov_norm * (uxy - ux * uy)

    R = data_range
    C1 = (K1 * R) ** 2
    C2 = (K2 * R) ** 2

    A1, A2, B1, B2 = (
        2 * ux * uy + C1,
        2 * vxy + C2,
        ux ** 2 + uy ** 2 + C1,
        vx + vy + C2,
    )
    D = B1 * B2
    S = (A1 * A2) / D

    pad = (win_size - 1) // 2
    mssim = S[tuple(slice(pad, s - pad) for s in S.shape)].mean(dtype=np.float64)
    if full:
        return mssim, S
    return mssim
