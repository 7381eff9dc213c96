"""Host-side stride validation of every C-ABI entry point that takes strides (no GPU needed; pointers are fake and
never dereferenced because every call here either fails validation or has an empty batch).

include/mie.h: plane i at base + i*stride_n, row y at + y*stride_h, in elements.  A row stride below the width, or a
plane stride that makes plane i+1 start inside plane i's last row, is MIE_E_STRIDE — for the source and the
destination separately, and for the slice stride of the volume entry points.  The tightest legal plane stride is
(h - 1) * stride_h + w, one element less is refused.  An empty batch is a no-op whatever its (legal) layout."""
import numpy as np
import pytest

E_STRIDE = -4
FAKE = 0x10000   # 256-byte aligned, never dereferenced
H, W = 64, 64
PAD = W + 48     # a legal padded row stride
TAPS9 = np.ones(9, np.float32) / 9
WSP9 = np.ones(81, np.float32) / 81


def _lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def _t():
    return TAPS9.ctypes.data


# Each entry: name -> (call(n, s, d) -> rc, has_destination).  s = (ssn, ssh), d = (dsn, dsh); every other argument
# valid, so the stride check decides.
def _planes_ops():
    L = _lib()
    ws = 1 << 30
    U16, F32 = 1, 3
    return {
        "mie_gaussian2d": (lambda n, s, d: L.mie_gaussian2d(FAKE, FAKE, U16, U16, n, H, W, *s, *d, _t(), 9, _t(), 9, 1,
                                                            0.0, 65535.0, None), True),
        "mie_unsharp": (lambda n, s, d: L.mie_unsharp(FAKE, FAKE, U16, U16, n, H, W, *s, *d, _t(), 9, _t(), 9, 1, 0.0,
                                                      65535.0, None), True),
        "mie_unsharp_amount": (lambda n, s, d: L.mie_unsharp_amount(FAKE, FAKE, U16, U16, n, H, W, *s, *d, _t(), 9, _t(),
                                                                    9, 4, 1.5, 1, 0.0, 65535.0, None), True),
        "mie_clahe_hist": (lambda n, s, d: L.mie_clahe_hist(FAKE, U16, n, H, W, *s, 8, 8, 0, 0.0, 65535.0, FAKE, None),
                           False),
        "mie_clahe_luts": (lambda n, s, d: L.mie_clahe_luts(FAKE, U16, n, H, W, *s, 8, 8, 2.0, 0, 0.0, 65535.0, FAKE,
                                                            None), False),
        "mie_clahe_apply": (lambda n, s, d: L.mie_clahe_apply(FAKE, FAKE, U16, U16, n, H, W, *s, *d, 8, 8, 0, 0.0,
                                                              65535.0, FAKE, None), True),
        "mie_clahe": (lambda n, s, d: L.mie_clahe(FAKE, FAKE, F32, F32, n, H, W, *s, *d, 8, 8, 2.0, 0, 0.0, 1.0, FAKE,
                                                  ws, None), True),
        "mie_clahe[opencv u16]": (lambda n, s, d: L.mie_clahe(FAKE, FAKE, U16, U16, n, H, W, *s, *d, 8, 8, 2.0, 1, 0.0,
                                                              65535.0, FAKE, ws, None), True),
        "mie_clahe16_luts": (lambda n, s, d: L.mie_clahe16_luts(FAKE, n, H, W, *s, 8, 8, 2.0, FAKE, None), False),
        "mie_equalize": (lambda n, s, d: L.mie_equalize(FAKE, FAKE, U16, U16, n, H, W, *s, *d, 0.0, 65535.0, FAKE, ws,
                                                        None), True),
        "mie_median2d": (lambda n, s, d: L.mie_median2d(FAKE, FAKE, U16, n, H, W, *s, *d, 3, 3, 0, None), True),
        "mie_median3d": (lambda n, s, d: L.mie_median3d(FAKE, FAKE, U16, n, H, W, *s, *d, None, None, 2, None), True),
        "mie_bilateral": (lambda n, s, d: L.mie_bilateral(FAKE, FAKE, U16, U16, n, H, W, *s, *d, WSP9.ctypes.data, 9, 9,
                                                          0.1, 1, 0.0, 65535.0, None), True),
        "mie_nlm": (lambda n, s, d: L.mie_nlm(FAKE, FAKE, U16, F32, n, H, W, *s, *d, 5, 6, 0.1, 0.0, 0.0, 65535.0, None),
                    True),
        "mie_nlm_slow": (lambda n, s, d: L.mie_nlm_slow(FAKE, FAKE, U16, F32, n, H, W, *s, *d, 5, 4, 0.1, 0.0, 0.0,
                                                        65535.0, None), True),
        # metrics: the second image takes the destination's place
        "mie_sqdiff_sums": (lambda n, s, d: L.mie_sqdiff_sums(FAKE, FAKE, U16, n, H, W, *s, *d, FAKE, FAKE, ws, None),
                            True),
        "mie_ssim_sums": (lambda n, s, d: L.mie_ssim_sums(FAKE, FAKE, U16, n, H, W, *s, *d, 7, 6.5, 58.5, FAKE, FAKE, ws,
                                                          None), True),
        "mie_bilateral_clahe": (lambda n, s, d: L.mie_bilateral_clahe(FAKE, FAKE, U16, U16, n, H, W, *s, *d,
                                                                      WSP9.ctypes.data, 9, 0.1, 1, 2, 2, 2.0, 0.0,
                                                                      65535.0, 7, FAKE, ws, None), True),
        "mie_sk_equalize_adapthist": (lambda n, s, d: L.mie_sk_equalize_adapthist(FAKE, FAKE, U16, 4, n, H, W, *s, *d, 8,
                                                                                  8, 0.01, 256, FAKE, ws, None), True),
        "mie_sk_equalize_hist": (lambda n, s, d: L.mie_sk_equalize_hist(FAKE, FAKE, U16, 4, n, H, W, *s, *d, FAKE, ws,
                                                                        None), True),
        "mie_sk_denoise_bilateral": (lambda n, s, d: L.mie_sk_denoise_bilateral(FAKE, FAKE, U16, 4, n, H, W, *s, *d, 5,
                                                                                1000, 2, 0.0, FAKE, FAKE, FAKE, None),
                                     True),
        "mie_chain_gauss_clahe_unsharp": (lambda n, s, d: L.mie_chain_gauss_clahe_unsharp(
            FAKE, FAKE, U16, U16, n, H, W, *s, *d, _t(), 9, _t(), 9, 8, 8, 2.0, _t(), 9, _t(), 9, 1, 0.0, 65535.0, 3,
            FAKE, ws, None), True),
    }


PLANE_OPS = ["mie_gaussian2d", "mie_unsharp", "mie_unsharp_amount", "mie_clahe_hist", "mie_clahe_luts", "mie_clahe_apply",
             "mie_clahe", "mie_clahe[opencv u16]", "mie_clahe16_luts", "mie_equalize", "mie_median2d", "mie_median3d",
             "mie_bilateral", "mie_nlm", "mie_nlm_slow", "mie_sqdiff_sums", "mie_ssim_sums", "mie_bilateral_clahe",
             "mie_sk_equalize_adapthist", "mie_sk_equalize_hist", "mie_sk_denoise_bilateral",
             "mie_chain_gauss_clahe_unsharp"]


def _tight(ssh):
    return (H - 1) * ssh + W


@pytest.mark.parametrize("name", PLANE_OPS)
def test_too_small_strides_are_refused(name):
    call, has_dst = _planes_ops()[name]
    ok = (_tight(PAD), PAD)
    bad_cases = [
        ("source row stride w - 1", 1, (H * (W - 1), W - 1), ok),
        ("source plane stride one short of the last row", 2, (_tight(PAD) - 1, PAD), ok),
        ("source plane stride one short, dense rows", 2, (_tight(W) - 1, W), ok),
    ]
    if has_dst:
        bad_cases += [
            ("destination row stride w - 1", 1, ok, (H * (W - 1), W - 1)),
            ("destination plane stride one short of the last row", 2, ok, (_tight(PAD) - 1, PAD)),
            ("destination plane stride one short, dense rows", 2, ok, (_tight(W) - 1, W)),
        ]
    for what, n, s, d in bad_cases:
        assert call(n, s, d) == E_STRIDE, f"{name}: {what}"


@pytest.mark.parametrize("name", PLANE_OPS)
def test_empty_batch_with_a_padded_layout_is_a_no_op(name):
    call, _ = _planes_ops()[name]
    assert call(0, ((H + 3) * PAD, PAD), (_tight(PAD), PAD)) == 0, name
    assert call(0, (_tight(W + 1) + 3, W + 1), ((H + 3) * PAD, PAD)) == 0, name


# ---------------------------------------------------------------------------------------------------------- volumes
D = 5


def _volume_ops():
    L = _lib()
    U16 = 1
    return {
        "mie_gaussian3d": lambda n, s, d: L.mie_gaussian3d(FAKE, FAKE, U16, U16, n, D, H, W, *s, *d, _t(), 9, _t(), 9,
                                                           _t(), 9, 4, 0.0, 65535.0, None),
        "mie_unsharp3d": lambda n, s, d: L.mie_unsharp3d(FAKE, FAKE, U16, U16, n, D, H, W, *s, *d, _t(), 9, _t(), 9,
                                                         _t(), 9, 4, 1.5, 1, 0.0, 65535.0, None),
        "mie_sk_equalize_adapthist3d": lambda n, s, d: L.mie_sk_equalize_adapthist3d(
            FAKE, FAKE, U16, 4, n, D, H, W, *s, *d, 2, 8, 8, 0.01, 256, FAKE, 1 << 30, None),
    }


def _vol(ssh, ssd=None, ssn=None):
    """(ssn, ssd, ssh): the tightest legal slice / volume strides unless given."""
    ssd = (H - 1) * ssh + W if ssd is None else ssd
    ssn = (D - 1) * ssd + (H - 1) * ssh + W if ssn is None else ssn
    return ssn, ssd, ssh


@pytest.mark.parametrize("name", ["mie_gaussian3d", "mie_unsharp3d", "mie_sk_equalize_adapthist3d"])
def test_volume_strides_too_small_are_refused(name):
    call = _volume_ops()[name]
    ok = _vol(PAD)
    tight_d = (H - 1) * PAD + W
    bad = [
        ("row stride w - 1", 1, _vol(W - 1), ok),
        ("slice stride one short of the last row", 1, _vol(PAD, ssd=tight_d - 1, ssn=D * tight_d), ok),
        ("volume stride one short of the last slice's last row", 2, _vol(PAD, ssn=(D - 1) * tight_d + (H - 1) * PAD + W - 1),
         ok),
        ("volume stride ignoring the padded slices", 2, _vol(PAD, ssd=(H + 3) * PAD, ssn=D * H * W), ok),
    ]
    bad += [(f"destination {what}", n, d, s) for what, n, s, d in bad]
    for what, n, s, d in bad:
        assert call(n, s, d) == E_STRIDE, f"{name}: {what}"


@pytest.mark.parametrize("name", ["mie_gaussian3d", "mie_unsharp3d", "mie_sk_equalize_adapthist3d"])
def test_volume_empty_batch_with_a_padded_layout_is_a_no_op(name):
    call = _volume_ops()[name]
    padded = _vol(PAD, ssd=(H + 3) * PAD, ssn=(D + 1) * (H + 3) * PAD)
    assert call(0, padded, _vol(W + 1, ssd=H * (W + 1) + 3, ssn=D * (H * (W + 1) + 3) + 5)) == 0, name
