"""numpy twin of skimage.filters.frangi / hessian / sato / meijering and skimage.feature.hessian_matrix /
hessian_matrix_eigvals — TEST INFRASTRUCTURE ONLY (never imported by the package).

**RECALLED**: the functions below are literal transcriptions of upstream (0.26, skimage/filters/ridges.py,
skimage/feature/corner.py) as remembered, on scipy.ndimage.gaussian_filter and np.linalg.eigvalsh; scikit-image is not
installable here, so nothing in them is pinned against upstream until
tests/test_sk_ridges.py::test_live_pin_against_skimage can run.  Each recalled choice is marked RECALLED.

`sym_line` / `anti_line` transcribe scipy.ndimage's 1-D correlation loops for symmetric (order 0) and antisymmetric
(order 1) Gaussian weights, vectorised over every other axis, in all five modes: the arithmetic csrc/sk_ridges.cu
implements."""
from __future__ import annotations

from itertools import combinations_with_replacement

import numpy as np
from scipy import linalg
from scipy.ndimage import gaussian_filter

TRUNCATE = 4.0   # RECALLED: scipy's default truncate, sigma unscaled


def _index(i: np.ndarray, n: int, mode: str) -> np.ndarray:
    """Source index of extended coordinate i on an axis of length n (-1: cval), scipy's extension rules."""
    i = np.asarray(i)
    if mode == "constant":
        return np.where((i >= 0) & (i < n), i, -1)
    if mode == "nearest":
        return np.clip(i, 0, n - 1)
    if mode == "wrap":
        return i % n
    if mode == "reflect":     # d c b a | a b c d | d c b a
        m = i % (2 * n)
        return np.where(m < n, m, 2 * n - 1 - m)
    if mode == "mirror":      # d c b | a b c d | c b a
        if n == 1:
            return np.zeros_like(i)
        p = 2 * (n - 1)
        m = i % p
        return np.where(m < n, m, p - m)
    raise ValueError(mode)


def _extended(x: np.ndarray, axis: int, r: int, mode: str, cval: float) -> np.ndarray:
    n = x.shape[axis]
    idx = _index(np.arange(-r, n + r), n, mode)
    ext = np.take(x, np.maximum(idx, 0), axis=axis).astype(np.float64)
    ext = np.moveaxis(ext, axis, 0)
    ext[idx < 0] = cval
    return ext


def _line(x, weights, axis, mode, cval, sign):
    r = weights.size // 2
    n = x.shape[axis]
    ext = _extended(x, axis, r, mode, cval)
    out = np.empty((n,) + ext.shape[1:], np.float64)
    for i in range(n):
        c = i + r
        tmp = ext[c] * weights[r]
        for j in range(-r, 0):
            tmp = tmp + ((ext[c + j] + ext[c - j]) if sign > 0 else (ext[c + j] - ext[c - j])) * weights[j + r]
        out[i] = tmp
    return np.moveaxis(out, 0, axis).astype(x.dtype)


def sym_line(x, weights, axis=-1, mode="reflect", cval=0.0):
    """scipy's correlate1d loop for symmetric weights: tmp = ext[c] w[r]; tmp += (ext[c + j] + ext[c - j]) w[j + r]."""
    return _line(x, weights, axis, mode, cval, 1)


def anti_line(x, weights, axis=-1, mode="reflect", cval=0.0):
    """The same for antisymmetric weights: tmp += (ext[c + j] - ext[c - j]) w[j + r]."""
    return _line(x, weights, axis, mode, cval, -1)


def img_as_float(image: np.ndarray) -> np.ndarray:
    image = np.asarray(image)
    if image.dtype == np.uint8:
        return image.astype(np.float64) / 255.0
    if image.dtype == np.uint16:
        return image.astype(np.float64) / 65535.0
    if image.dtype == np.int16:
        return (image.astype(np.float64) * 2.0 + 1.0) / 65535.0
    return image


def _float_type(dtype) -> type:
    return np.float32 if np.dtype(dtype) == np.float32 else np.float64


def hessian_matrix(image, sigma=1, mode="constant", cval=0, order="rc", use_gaussian_derivatives=True):
    """RECALLED: img_as_float, then gradients G_a = gaussian_filter(image, sigma, order=e_a) and
    H_ab = gaussian_filter(G_a, sigma, order=e_b) for (a, b) in combinations_with_replacement(range(ndim), 2)."""
    assert use_gaussian_derivatives and order == "rc"
    image = img_as_float(image)
    image = image.astype(_float_type(image.dtype), copy=False)
    ndim = image.ndim
    orders = [tuple(1 if a == b else 0 for b in range(ndim)) for a in range(ndim)]
    gradients = [gaussian_filter(image, sigma, order=orders[a], mode=mode, cval=cval, truncate=TRUNCATE)
                 for a in range(ndim)]
    return [gaussian_filter(gradients[a], sigma, order=orders[b], mode=mode, cval=cval, truncate=TRUNCATE)
            for a, b in combinations_with_replacement(range(ndim), 2)]


def hessian_matrix_eigvals(H_elems):
    """RECALLED: 2-D closed form (m + hs, m - hs); 3-D np.linalg.eigvalsh reversed to decreasing order."""
    if len(H_elems) == 3:
        M00, M01, M11 = H_elems
        m = (M00 + M11) / 2
        hs = np.sqrt(M01 ** 2 + ((M00 - M11) / 2) ** 2)
        eigs = np.empty((2, *M00.shape), M00.dtype)
        eigs[:] = (m + hs, m - hs)
        return eigs
    H00, H01, H02, H11, H12, H22 = H_elems
    mats = np.stack([np.stack([H00, H01, H02], -1), np.stack([H01, H11, H12], -1), np.stack([H02, H12, H22], -1)], -2)
    eigs = np.linalg.eigvalsh(mats)[..., ::-1]
    return np.moveaxis(eigs, -1, 0)


def _hessian_eigvals(image, sigma, mode, cval):
    return hessian_matrix_eigvals(hessian_matrix(image, sigma, mode=mode, cval=cval, use_gaussian_derivatives=True))


def _check_sigmas(sigmas):
    if any(s < 0 for s in sigmas):   # RECALLED
        raise ValueError("Sigma values less than zero are not valid")


def frangi(image, sigmas=range(1, 10, 2), scale_range=None, scale_step=None, alpha=0.5, beta=0.5, gamma=None,
           black_ridges=True, mode="reflect", cval=0):
    """RECALLED: gamma=None is set from the FIRST sigma's s and reused; ties of |lambda| keep the decreasing order."""
    if scale_range is not None and scale_step is not None:
        sigmas = np.arange(scale_range[0], scale_range[1], scale_step)
    sigmas = list(sigmas)
    _check_sigmas(sigmas)
    image = np.asarray(image)
    image = image.astype(_float_type(image.dtype), copy=False)
    if not black_ridges:
        image = -image
    filtered_max = np.zeros_like(image)
    for sigma in sigmas:
        eigvals = _hessian_eigvals(image, sigma, mode, cval)
        eigvals = np.take_along_axis(eigvals, abs(eigvals).argsort(0, kind="stable"), 0)
        lambda1 = eigvals[0]
        if image.ndim == 2:
            (lambda2,) = np.maximum(eigvals[1:], 1e-10)
            r_a = np.inf
            r_b = abs(lambda1) / lambda2
        else:
            lambda2, lambda3 = np.maximum(eigvals[1:], 1e-10)
            r_a = lambda2 / lambda3
            r_b = abs(lambda1) / np.sqrt(lambda2 * lambda3)
        s = np.sqrt((eigvals ** 2).sum(0))
        if gamma is None:
            gamma = s.max() / 2
            if gamma == 0:
                gamma = 1
        vals = 1.0 - np.exp(-r_a ** 2 / (2 * alpha ** 2))
        vals *= np.exp(-r_b ** 2 / (2 * beta ** 2))
        vals *= 1.0 - np.exp(-s ** 2 / (2 * gamma ** 2))
        filtered_max = np.maximum(filtered_max, vals)
    return filtered_max


def hessian(image, sigmas=range(1, 10, 2), scale_range=None, scale_step=None, alpha=0.5, beta=0.5, gamma=15,
            black_ridges=True, mode="reflect", cval=0):
    filtered = frangi(image, sigmas=sigmas, scale_range=scale_range, scale_step=scale_step, alpha=alpha, beta=beta,
                      gamma=gamma, black_ridges=black_ridges, mode=mode, cval=cval)
    filtered[filtered <= 0] = 1
    return filtered


def sato(image, sigmas=range(1, 10, 2), black_ridges=True, mode="reflect", cval=0):
    sigmas = list(sigmas)
    _check_sigmas(sigmas)
    image = np.asarray(image)
    image = image.astype(_float_type(image.dtype), copy=False)
    if not black_ridges:
        image = -image
    filtered_max = np.zeros_like(image)
    for sigma in sigmas:
        eigvals = _hessian_eigvals(image, sigma, mode, cval)
        eigvals = eigvals[:-1]
        vals = sigma ** 2 * np.prod(np.maximum(eigvals, 0), 0) ** (1 / len(eigvals))
        filtered_max = np.maximum(filtered_max, vals)
    return filtered_max


def meijering(image, sigmas=range(1, 10, 2), alpha=None, black_ridges=True, mode="reflect", cval=0):
    sigmas = list(sigmas)
    _check_sigmas(sigmas)
    image = np.asarray(image)
    image = image.astype(_float_type(image.dtype), copy=False)
    if not black_ridges:
        image = -image
    if alpha is None:
        alpha = 1 / (image.ndim + 1)
    mtx = linalg.circulant([1, *[alpha] * (image.ndim - 1)]).astype(image.dtype)
    filtered_max = np.zeros_like(image)
    for sigma in sigmas:
        eigvals = _hessian_eigvals(image, sigma, mode, cval)
        vals = np.tensordot(mtx, eigvals, 1)
        vals = np.take_along_axis(vals, abs(vals).argmax(0)[None], 0).squeeze(0)
        vals = np.maximum(vals, 0)
        max_val = vals.max()
        if max_val > 0:
            vals /= max_val
        filtered_max = np.maximum(filtered_max, vals)
    return filtered_max
