"""numpy twin of skimage.restoration.denoise_tv_chambolle — TEST INFRASTRUCTURE ONLY (never imported by the package).

**RECALLED**: a literal transcription of upstream's `_denoise_tv_chambolle_nd` as the author remembers the 0.26
sources; scikit-image is not installable here, so nothing in it is pinned against upstream until
tests/test_tv_chambolle.py::test_live_pin_against_skimage can run.  Integer images go through img_as_float
(oracle/skimage_twin.py); float32 images stay float32, and NumPy 2's weak Python scalars then round tau, tau / weight,
weight * sum and eps * E_init to float32 exactly as upstream does.

Two extras over upstream: the number of passes run (the returned `out` is that of the last one), and the smallest
relative distance between |E_previous - E| and eps * E_init over the stopping tests made, so that a test can assert
that its case is far from a tie, where a different summation order could change the iteration count."""
from __future__ import annotations

import numpy as np

from skimage_twin import img_as_float


def denoise_tv_chambolle(image, weight=0.1, eps=2e-4, max_num_iter=200):
    """-> (out, passes run, tie margin).  The margin is inf when the threshold eps * E_init is 0 (no test can pass)."""
    image = img_as_float(np.asarray(image))
    ndim = image.ndim
    p = np.zeros((ndim,) + image.shape, dtype=image.dtype)
    g = np.zeros_like(p)
    d = np.zeros_like(image)
    margin = np.inf
    i = 0
    while i < max_num_iter:
        if i > 0:
            d = -p.sum(0)
            slices_d = [slice(None)] * ndim
            slices_p = [slice(None)] * (ndim + 1)
            for ax in range(ndim):
                slices_d[ax] = slice(1, None)
                slices_p[ax + 1] = slice(0, -1)
                slices_p[0] = ax
                d[tuple(slices_d)] += p[tuple(slices_p)]
                slices_d[ax] = slice(None)
                slices_p[ax + 1] = slice(None)
            out = image + d
        else:
            out = image
        E = (d ** 2).sum()
        slices_g = [slice(None)] * (ndim + 1)
        for ax in range(ndim):
            slices_g[ax + 1] = slice(0, -1)
            slices_g[0] = ax
            g[tuple(slices_g)] = np.diff(out, axis=ax)
            slices_g[ax + 1] = slice(None)
        norm = np.sqrt((g ** 2).sum(axis=0))[np.newaxis, ...]
        E += weight * norm.sum()
        tau = 1.0 / (2.0 * ndim)
        norm *= tau / weight
        norm += 1.0
        p -= tau * g
        p /= norm
        E /= float(image.size)
        if i == 0:
            E_init = E
            E_previous = E
        else:
            threshold = eps * E_init
            if threshold != 0:
                margin = min(margin, abs(float(np.abs(E_previous - E)) - float(threshold)) / abs(float(threshold)))
            if np.abs(E_previous - E) < threshold:
                break
            else:
                E_previous = E
        i += 1
    return out, min(i + 1, max_num_iter), margin
