"""numpy front end of tests/sk_adapthist3d_oracle.c: skimage.exposure.equalize_adapthist on ONE 3-D volume, restated
per voxel in C.  TEST INFRASTRUCTURE ONLY (imported by tests/test_skimage_adapthist3d.py, never by the package).

The C file includes oracle/mie_oracle.c whole and adds the 3-D contextual-region stage, so the grey and rescale stages
are the very functions the 2-D oracle runs.  The library is compiled with the oracle's flags into the temporary
directory (named by a hash of both sources and the flags), never into the source tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle as O   # puts oracle/ on sys.path (for `build`), and gives the dtype codes and kernel-size rule
from build import CFLAGS  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sk_adapthist3d_oracle.c")
ORACLE_SRC = os.path.join(os.path.dirname(HERE), "oracle", "mie_oracle.c")

_lib = None
_p, _i, _d = C.c_void_p, C.c_int, C.c_double


def _build() -> str:
    h = hashlib.sha256()
    for path in (SRC, ORACLE_SRC):
        with open(path, "rb") as f:
            h.update(f.read())
    h.update(" ".join(CFLAGS).encode())
    uid = os.getuid() if hasattr(os, "getuid") else 0
    lib = os.path.join(tempfile.gettempdir(), f"mie_sk_adapthist3d_oracle_{uid}_{h.hexdigest()[:16]}.so")
    if os.path.exists(lib):
        return lib
    gcc = shutil.which("gcc")
    if gcc is None:
        raise RuntimeError("gcc not found: cannot build the volumetric CLAHE oracle")
    tmp = f"{lib}.tmp{os.getpid()}"
    r = subprocess.run([gcc, *CFLAGS, SRC, "-o", tmp, "-lm"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"volumetric CLAHE oracle build failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib)
    return lib


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(_build())
        L.orc_sk_adapthist_grey.argtypes, L.orc_sk_adapthist_grey.restype = [_p, _i, _i, _i, _p], _i
        L.orc_sk_clahe3d.argtypes, L.orc_sk_clahe3d.restype = [_p, _i, _i, _i, _i, _i, _i, _d, _i, _p, _p], _i
        L.orc_sk_rescale01.argtypes, L.orc_sk_rescale01.restype = [_p, _i, _i, _i, _p], _i
        _lib = L
    return _lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _check(rc: int):
    if rc != 0:
        raise RuntimeError(f"oracle error {rc}")


def sk_equalize_adapthist3d(volume, kernel_size=None, clip_limit=0.01, nbins=256, return_stages=False):
    """skimage.exposure.equalize_adapthist on ONE (D, H, W) volume: one image with 3-D contextual regions of
    kernel_size = (kd, kr, kc) voxels (int: a cube; default max(dim // 8, 1) per axis), min / max over the volume.
    Stages: grey (2^14 levels), clahe (uint16), maps (region mappings, int64)."""
    x = np.ascontiguousarray(volume)
    if x.ndim != 3 or x.dtype not in O._DT:
        raise ValueError("expected one 3-D volume of dtype uint8 / uint16 / int16 / float32")
    d, h, w = x.shape
    kd, kr, kc = O.sk_adapthist_kernel(x.shape, kernel_size)
    L = lib()
    grey = np.empty(x.shape, np.uint16)
    _check(L.orc_sk_adapthist_grey(_ptr(x), O._DT[x.dtype], d * h, w, _ptr(grey)))   # flat: d * h rows
    c = np.empty(x.shape, np.uint16)
    maps = np.empty((-(-d // kd), -(-h // kr), -(-w // kc), nbins), np.int64)
    _check(L.orc_sk_clahe3d(_ptr(grey), d, h, w, kd, kr, kc, float(clip_limit), int(nbins), _ptr(c), _ptr(maps)))
    f32 = x.dtype == np.float32
    out = np.empty(x.shape, np.float32 if f32 else np.float64)
    _check(L.orc_sk_rescale01(_ptr(c), d * h, w, int(f32), _ptr(out)))
    if return_stages:
        return out, {"grey": grey, "clahe": c, "maps": maps}
    return out
