"""numpy front end of tests/gaussian3d_oracle.c: skimage.filters.gaussian / unsharp_mask on (..., D, H, W) volumes,
restated per voxel in C.  TEST INFRASTRUCTURE ONLY (imported by tests/test_gaussian3d.py, never by the package).

The C file includes oracle/mie_oracle.c whole and adds the z pass, so the x and y passes are the 2-D oracle's.  The
library is compiled with the oracle's flags into the temporary directory (named by a hash of both sources and the
flags), never into the source tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle as O   # puts oracle/ on sys.path (for `build`), and gives the weights, border codes and scipy modes
from build import CFLAGS  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "gaussian3d_oracle.c")
ORACLE_SRC = os.path.join(os.path.dirname(HERE), "oracle", "mie_oracle.c")

_lib = None
_p, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float


def _build() -> str:
    h = hashlib.sha256()
    for path in (SRC, ORACLE_SRC):
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(CFLAGS).encode())
    uid = os.getuid() if hasattr(os, "getuid") else 0
    lib = os.path.join(tempfile.gettempdir(), f"mie_gaussian3d_oracle_{uid}_{h.hexdigest()[:16]}.so")
    if os.path.exists(lib):
        return lib
    gcc = shutil.which("gcc")
    if gcc is None:
        raise RuntimeError("gcc not found: cannot build the 3-D Gaussian oracle")
    tmp = f"{lib}.tmp{os.getpid()}"
    r = subprocess.run([gcc, *CFLAGS, SRC, "-o", tmp, "-lm"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"3-D Gaussian oracle build failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib)
    return lib


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_build())
        L.orc_gaussian3d_ex.argtypes = [_p, _p, _i64, _i, _i, _i, _p, _i, _p, _i, _p, _i, _i, _i, _f, _i]
        L.orc_gaussian3d_ex.restype = _i
        _lib = L
    return _lib


def gaussian_taps3d(sigma, truncate=4.0):
    """Per-axis weights (z, y, x) of skimage.filters.gaussian on a 3-D array: K = 2*int(truncate*sigma + 0.5) + 1
    taps; an axis with sigma == 0 is not filtered (one tap of weight 1.0)."""
    sig = tuple(sigma) if isinstance(sigma, (tuple, list)) else (sigma,) * 3
    out = []
    for s in sig:
        s = float(s)
        if s == 0.0:
            out.append(np.ones(1, np.float32))
        else:
            out.append(O.gaussian_kernel1d(2 * int(float(truncate) * s + 0.5) + 1, s))
    return out


def sep3d(x01, wz, wy, wx, border_type, unsharp=0, amount=1.0, clip=0):
    """orc_gaussian3d_ex on (..., D, H, W) float32 volumes: x pass, y pass, z pass."""
    x = np.ascontiguousarray(x01, np.float32)
    if x.ndim < 3:
        raise ValueError("expected (..., D, H, W)")
    d, h, w = x.shape[-3:]
    n = int(np.prod(x.shape[:-3], dtype=np.int64)) if x.ndim > 3 else 1
    wz, wy, wx = (np.ascontiguousarray(a, np.float32) for a in (wz, wy, wx))
    out = np.empty_like(x)
    rc = lib().orc_gaussian3d_ex(O._ptr(x), O._ptr(out), n, d, h, w, O._ptr(wx), wx.size, O._ptr(wy), wy.size,
                                 O._ptr(wz), wz.size, O.BORDERS[border_type], int(unsharp), float(amount), int(clip))
    if rc != 0:
        raise RuntimeError(f"3-D Gaussian oracle error {rc}")
    return out


def skimage_gaussian3d(x01, sigma=1.0, mode="nearest", truncate=4.0):
    """skimage.filters.gaussian on (..., D, H, W) float volumes, every (D, H, W) volume one 3-D image."""
    wz, wy, wx = gaussian_taps3d(sigma, truncate)
    return sep3d(x01, wz, wy, wx, O.SCIPY_MODES[mode])


def skimage_unsharp_mask3d(x01, radius=1.0, amount=1.0, preserve_range=False):
    """skimage.filters.unsharp_mask on (..., D, H, W) [0,1] volumes: x + amount (x - gaussian(x, radius,
    mode='reflect')) over all three axes, clipped to [0,1] unless preserve_range."""
    wz, wy, wx = gaussian_taps3d(radius, 4.0)
    return sep3d(x01, wz, wy, wx, "symmetric", 1, amount, 0 if preserve_range else 1)
