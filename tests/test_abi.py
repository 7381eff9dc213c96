"""CPU-side checks of the C-ABI boundary: the library loads without a GPU, exports every
symbol include/mie.h declares, and the Python mirror rejects bad arguments like kornia does."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "mie.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mie_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import mie_b200
    from mie_b200 import _ffi

    lib = ctypes.CDLL(_ffi.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mie.h but not exported"
    assert set(names) == set(_ffi.SIGNATURES), "ctypes signature table out of sync with include/mie.h"
    assert mie_b200._lib().mie_abi_version() == 1


def test_error_strings():
    from mie_b200 import _ffi

    L = _ffi.lib()
    assert L.mie_error_string(0) == b"ok"
    for code in range(-12, 0):
        assert L.mie_error_string(code) != b"unknown error"
    with pytest.raises(ValueError):
        _ffi.check(-6)
    with pytest.raises(TypeError):
        _ffi.check(-2)
    with pytest.raises(NotImplementedError):
        _ffi.check(-11)


def test_workspace_queries_need_no_gpu():
    from mie_b200 import _ffi

    L = _ffi.lib()
    # LUTs (256 B per tile) + packed cell tables of the tuned interpolation pass (2 KB per cell)
    assert L.mie_clahe_workspace_bytes(256, 512, 512, 8, 8) == 256 * 64 * 256 + 256 * 81 * 2048
    assert L.mie_clahe16_lut_bytes(8, 8) == 64 * 65536 * 2
    assert L.mie_chain_workspace_bytes(2, 64, 64, 2, 2) == 2 * 4 * 256 + 2 * 64 * 64 * 4
    assert L.mie_chain_workspace_bytes(0, 64, 64, 2, 2) == 0


def test_argument_errors_match_kornia_types():
    import mie_b200 as M

    x = torch.zeros(1, 1, 16, 16)
    with pytest.raises(TypeError):
        M.equalize_clahe(x, 2, (8, 8))  # clip_limit must be float
    with pytest.raises(TypeError):
        M.equalize_clahe(x, 2.0, [8, 8])  # grid_size must be a tuple
    with pytest.raises(TypeError):
        M.equalize_clahe(x, 2.0, (8, 8, 8))
    with pytest.raises(TypeError):
        M.equalize_clahe(x, 2.0, (8.0, 8))
    with pytest.raises(ValueError):
        M.equalize_clahe(x, 2.0, (0, 8))
    with pytest.raises(NotImplementedError):
        M.equalize_clahe(x, 2.0, (8, 8), slow_and_differentiable=True)
    # no CPU path: CPU tensors are refused loudly
    with pytest.raises(RuntimeError, match="no CPU path"):
        M.equalize_clahe(x, 2.0, (8, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        M.gaussian_blur2d(x, 9, 1.0)
    with pytest.raises(ValueError):
        M.gaussian_blur2d(x.to(torch.float32), 4, 1.0)  # even kernel


def test_host_side_argument_validation_of_the_abi():
    """Argument errors are detected on the host before any launch (no GPU needed)."""
    from mie_b200 import _ffi

    L = _ffi.lib()
    import numpy as np

    w = np.ones(9, np.float32) / 9
    fake = 0x1000  # never dereferenced: validation fails first
    args = dict(n=1, h=64, w=64)
    # reflect halo >= image
    rc = L.mie_gaussian2d(fake, fake, 3, 3, 1, 4, 4, 16, 4, 16, 4, w.ctypes.data, 9, w.ctypes.data, 9, 1, 0.0, 1.0, None)
    assert rc == -8
    rc = L.mie_gaussian2d(fake, fake, 3, 3, 1, 64, 64, 4096, 64, 4096, 64, w.ctypes.data, 8, w.ctypes.data, 9, 1, 0.0,
                          1.0, None)
    assert rc == -7
    rc = L.mie_gaussian2d(None, fake, 3, 3, 1, 64, 64, 4096, 64, 4096, 64, w.ctypes.data, 9, w.ctypes.data, 9, 1, 0.0,
                          1.0, None)
    assert rc == -1
    rc = L.mie_gaussian2d(fake, fake, 1, 0, 1, 64, 64, 4096, 64, 4096, 64, w.ctypes.data, 9, w.ctypes.data, 9, 1, 0.0,
                          65535.0, None)
    assert rc == -2  # u16 -> u8 not allowed
    rc = L.mie_clahe_luts(fake, 3, 1, 20, 20, 400, 20, 0, 8, 2.0, 0, 0.0, 1.0, fake, None)
    assert rc == -5
    rc = L.mie_clahe_luts(fake, 3, 1, 3, 3, 9, 3, 8, 8, 2.0, 0, 0.0, 1.0, fake, None)
    assert rc == -6  # kornia: cannot compute tiles
    rc = L.mie_clahe(fake, fake, 1, 1, 1, 64, 64, 4096, 64, 4096, 64, 8, 8, 2.0, 0, 0.0, 65535.0, fake, 10, None)
    assert rc == -9
    rc = L.mie_clahe_luts(fake, 1, 1, 64, 64, 4096, 64, 8, 8, 2.0, 0, 5.0, 5.0, fake, None)
    assert rc == -10


def test_newer_entry_points_reject_bad_arguments_before_any_launch():
    """Argument validation of the metrics / skimage-signature / median / chain entry points runs on the host,
    so it can be checked without a GPU (pointers are never dereferenced when validation fails)."""
    import numpy as np
    from mie_b200 import _ffi

    L = _ffi.lib()
    fake = 0x1000
    w9 = np.ones(9, np.float32) / 9
    # metrics: window larger than the image, unknown dtype, undersized workspace, n == 0 is a no-op
    assert L.mie_ssim_sums(fake, fake, 1, 1, 8, 8, 64, 8, 64, 8, 11, 1.0, 1.0, fake, fake, 1 << 20, None) == -7
    assert L.mie_ssim_sums(fake, fake, 1, 1, 64, 64, 4096, 64, 4096, 64, 17, 1.0, 1.0, fake, fake, 1 << 20, None) == -7
    assert L.mie_sqdiff_sums(fake, fake, 7, 1, 8, 8, 64, 8, 64, 8, fake, fake, 1 << 20, None) == -2
    assert L.mie_sqdiff_sums(fake, fake, 1, 1, 64, 64, 4096, 64, 4096, 64, fake, fake, 1, None) == -9
    assert L.mie_sqdiff_sums(None, None, 1, 0, 64, 64, 4096, 64, 4096, 64, None, None, 0, None) == 0
    assert L.mie_metric_workspace_bytes(2, 64, 64, 11) == 2 * 4 * 2 * 8      # 2 planes x (2x2 window tiles) x 2 doubles
    assert L.mie_metric_workspace_bytes(2, 8, 8, 11) == 0                    # window does not fit
    # unsharp with amount: symmetric border accepted by validation (fails later only on the null stream launch),
    # unknown border rejected
    assert L.mie_unsharp_amount(fake, fake, 3, 3, 1, 64, 64, 4096, 64, 4096, 64, w9.ctypes.data, 9, w9.ctypes.data, 9,
                                9, 1.5, 1, 0.0, 1.0, None) == -8
    assert L.mie_unsharp_amount(fake, fake, 3, 3, 0, 64, 64, 4096, 64, 4096, 64, w9.ctypes.data, 9, w9.ctypes.data, 9,
                                4, 1.5, 1, 0.0, 1.0, None) == 0             # empty batch, symmetric border: fine
    # median: even kernel, circular border
    assert L.mie_median2d(fake, fake, 1, 1, 64, 64, 4096, 64, 4096, 64, 4, 4, 0, None) == -7
    assert L.mie_median2d(fake, fake, 1, 1, 64, 64, 4096, 64, 4096, 64, 3, 3, 3, None) == -8
    assert L.mie_median3d(fake, fake, 1, 4, 64, 64, 4096, 64, 4096, 64, None, None, 1, None) == -8   # reflect: not for volumes
    # chain: unknown bits in the stages mask; schedule hints are legal
    assert L.mie_chain_gauss_clahe_unsharp(fake, fake, 1, 1, 0, 512, 512, 262144, 512, 262144, 512, w9.ctypes.data, 9,
                                           w9.ctypes.data, 9, 8, 8, 2.0, w9.ctypes.data, 9, w9.ctypes.data, 9, 1, 0.0,
                                           65535.0, 16, fake, 0, None) == -11
    assert L.mie_chain_gauss_clahe_unsharp(fake, fake, 1, 1, 0, 512, 512, 262144, 512, 262144, 512, w9.ctypes.data, 9,
                                           w9.ctypes.data, 9, 8, 8, 2.0, w9.ctypes.data, 9, w9.ctypes.data, 9, 1, 0.0,
                                           65535.0, 3 | 4, fake, 0, None) == 0


def test_median2d_rejects_unknown_dtype_codes_before_the_tuned_kernels():
    """The 3x3 / 5x5 tuned median kernels are chosen by dtype: an unknown code must be refused before that choice,
    as it is for the generic 7x7 path.  With a GPU the pointers are a real buffer, so a wrongly launched kernel
    stays inside it."""
    from mie_b200 import _ffi

    L = _ffi.lib()
    if torch.cuda.is_available():
        bufs = [torch.zeros(64 * 64 * 4, dtype=torch.uint8, device="cuda") for _ in range(2)]
        src, dst = (b.data_ptr() for b in bufs)
    else:
        src = dst = 0x10000
    for dtype in (4, 7, -1):
        for k in (3, 5, 7):
            assert L.mie_median2d(src, dst, dtype, 1, 64, 64, 4096, 64, 4096, 64, k, k, 0, None) == -2, (dtype, k)
    if torch.cuda.is_available():
        torch.cuda.synchronize()


def test_round2_advice_validation_paths():
    """ADVICE round 1: a misaligned workspace is refused (MIE_E_ALIGN) instead of faulting in a 32-bit / 128-bit
    access, and the 65 536-bin CLAHE validates the grid before it enters a division (was SIGFPE through the C ABI)."""
    import numpy as np
    from mie_b200 import _ffi

    L = _ffi.lib()
    w9 = np.ones(9, np.float32) / 9
    fake = 0x10000
    need = L.mie_chain_workspace_bytes(1, 512, 512, 8, 8)
    common = (1, 512, 512, 262144, 512, 262144, 512, w9.ctypes.data, 9, w9.ctypes.data, 9, 8, 8, 2.0, w9.ctypes.data, 9,
              w9.ctypes.data, 9, 1, 0.0, 65535.0, 3)
    assert L.mie_chain_gauss_clahe_unsharp(fake, fake, 1, 1, *common, fake + 1, need, None) == -12
    assert L.mie_chain_gauss_clahe_unsharp(fake, fake, 1, 1, *common, fake + 128, need, None) == -12
    with pytest.raises(ValueError):
        _ffi.check(-12)
    # mie_clahe, uint16 + OpenCV semantics (65 536 bins): zero / negative grids and shapes return codes
    for gh, gw, code in ((0, 8, -5), (8, 0, -5), (-3, 8, -5)):
        assert L.mie_clahe(fake, fake, 1, 1, 1, 64, 64, 4096, 64, 4096, 64, gh, gw, 2.0, 1, 0.0, 65535.0, fake, 1 << 20,
                           None) == code
    assert L.mie_clahe(fake, fake, 1, 1, 1, 0, 64, 4096, 64, 4096, 64, 8, 8, 2.0, 1, 0.0, 65535.0, fake, 1 << 20, None) == -3


def _fma32(a, b, c):
    """float32 fma through exact rational arithmetic (numpy has no fmaf)."""
    from fractions import Fraction
    import numpy as np
    return np.float32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def test_value_range_mode_is_a_host_query_and_its_verdicts_hold():
    """mie_value_range_mode (include/mie.h) needs no GPU.  Its verdicts: the dtype default -> 0, an integer window inside
    the dtype -> 1 (after the exhaustive host check), anything else -> -1.  For an accepted window the divide-free
    conversion of csrc/window.cuh is re-evaluated here on a sample of codes against the IEEE quotient the oracle uses."""
    import numpy as np
    import mie_b200 as M
    L = M._ffi.lib()
    U8, U16, I16, F32 = 0, 1, 2, 3
    assert L.mie_value_range_mode(U16, 0.0, 65535.0) == 0
    assert L.mie_value_range_mode(I16, -32768.0, 32767.0) == 0
    assert L.mie_value_range_mode(U8, 0.0, 255.0) == 0
    assert L.mie_value_range_mode(F32, 0.0, 1.0) == 0 and L.mie_value_range_mode(F32, -3.0, 7.5) == 0
    assert L.mie_value_range_mode(I16, -1024.0, 3071.0) == 1          # the HU window of config 3
    assert L.mie_value_range_mode(U16, 0.0, 4095.0) == 1              # 12-bit occupancy of a uint16 container
    assert L.mie_value_range_mode(U8, 16.0, 235.0) == 1
    assert L.mie_value_range_mode(I16, -1000.5, 3000.0) == -1         # non-integer bound
    assert L.mie_value_range_mode(U16, -1.0, 4095.0) == -1            # outside the dtype
    assert L.mie_value_range_mode(U8, 0.0, 256.0) == -1
    assert L.mie_value_range_mode(U16, 100.0, 100.0) == -1            # hi <= lo
    assert L.mie_value_range_mode(7, 0.0, 1.0) == -1                  # unknown dtype
    assert M.value_range_mode(torch.int16) == "default"
    assert M.value_range_mode(torch.int16, (-1024, 3071)) == "window"
    assert M.value_range_mode(torch.int16, (-1000.5, 3000.0)) == "generic"
    assert M.value_range_mode(torch.float32, (5, 9)) == "default"
    with pytest.raises(ValueError):
        M.value_range_mode(torch.uint16, (10, 10))
    with pytest.raises(TypeError):
        M.value_range_mode(torch.float64)

    # the conversion itself, int16 in the HU window: a = (2^23 + v + 32768) - (2^23 + 32768 + lo) is exact,
    # q0 = a * r, q = fma(fma(-rg, q0, a), r, q0) must equal (float(v) - lo) / rg
    lo, hi = np.float32(-1024.0), np.float32(3071.0)
    rg = np.float32(hi - lo)
    r = np.float32(1.0) / rg
    rng = np.random.default_rng(0)
    codes = np.concatenate([np.array([-32768, -1025, -1024, -1023, 0, 3070, 3071, 3072, 32767]),
                            rng.integers(-32768, 32768, 400)])
    for v in codes:
        exact = (np.float32(v) - lo) / rg
        a = np.float32(np.float32(8388608.0 + float(v) + 32768.0) - np.float32(8388608.0 + 32768.0 + float(lo)))
        q0 = np.float32(a * r)
        q = _fma32(_fma32(-rg, q0, a), r, q0)
        assert q == exact, (v, q, exact)
