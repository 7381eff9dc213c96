"""Hessian-based ridge filters on planes and whole volumes (skimage_compat.frangi / hessian / sato / meijering,
hessian_matrix, hessian_matrix_eigvals; mie_sk_ridge_filter*, mie_sk_hessian_matrix*, mie_sk_hessian_eigvals).

CPU: scipy.ndimage's line loops as the twin (tests/sk_ridges_twin.py) transcribes them, pinned against the installed
scipy; the package's taps; the twin's 2-D closed form against eigvalsh; the ABI's host validation; the Python argument
errors.  GPU: Hessian elements and 2-D eigenvalues bit for bit, 3-D eigenvalues and filter outputs within bounds argued
below, every dtype, mode and the filters' options, non-dense layouts, repeatable bits, graph capture, a batch beyond 2^31
elements and a 512^3 volume.

Tolerances.  The Hessian elements are bit-exact, so in 2-D the eigenvalues are too and the filters differ from the twin
only by exp (CUDA's and numpy's differ by at most an ulp or two) and, for meijering, numpy's BLAS order in tensordot:
a few ulp of values <= 1, hence 1e-14 (relative to the output's maximum for sato and meijering, whose values scale
with sigma^2 and the Hessian).  In 3-D the eigenvalues come from different solvers: each is within
E = 64 eps max|lambda| of eigvalsh's (eps of float64, of float32 for float32 images; checked directly below).  frangi's
factors are smooth in the eigenvalues away from a reordering by |lambda|, with derivatives bounded by the ratios they
take; at E ~ 1e-14 max|lambda| that leaves the outputs within 1e-9.  Where the twin's order by |lambda| (meijering:
its argmax of |.|) is decided by a gap below 2E, the two may pick different eigenvalues and the outputs differ by O(1):
those voxels are counted, printed and allowed up to 1e-5 of the voxels.  float32 images are compared at 1e-4: the float32
eigenvalue error (64 eps32 ~ 8e-6 relative) dominates.  Two places are not smooth and get their own bound:
- sato in 3-D takes sqrt(max(e0, 0) max(e1, 0)); an eigenvalue within E of 0 moves it by up to
  sigma^2 sqrt(E (|e0| + |e1| + E)), which is the per-voxel tolerance there.
- hessian sets values <= 0 to 1.  Where frangi's value is within 64 eps of 0 (1 - exp(-s^2 / 2 gamma^2) a few ulp
  from 0: on float32 [0, 1] images with gamma 15 that is much of the image), a one-ulp difference of exp decides between
  a tiny value and 1.  Those voxels are counted and printed; there the result must be 1 or below 64 eps."""
import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter, gaussian_filter1d

import sk_ridges_twin as T

U8, U16, I16, F32, F64 = 0, 1, 2, 3, 4
E_NULL, E_DTYPE, E_SHAPE, E_STRIDE, E_KERNEL, E_BORDER, E_WORKSPACE, E_RANGE, E_UNSUPPORTED, E_ALIGN = \
    -1, -2, -3, -4, -7, -8, -9, -10, -11, -12
FAKE = 0x10000   # 256-byte aligned, never dereferenced: every call with it fails validation or has an empty batch
MODES = ["reflect", "constant", "nearest", "mirror", "wrap"]


def _lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def _S():
    from mie_b200 import skimage_compat as S
    return S


def _image(shape, dtype, seed=0):
    """vessel_volume cropped to `shape` ((D, H, W), or more leading axes: one volume per image)."""
    from mie_b200 import synthetic

    shape = tuple(shape)
    n = int(np.prod(shape[:-3], dtype=np.int64)) if len(shape) > 3 else 1
    vols = [synthetic.vessel_volume(shape[-3:], dtype, seed + i, tubes=6) for i in range(n)]
    return np.stack(vols).reshape(shape)


def _planes(shape, dtype, seed=0):
    """(..., H, W) planes of vessel_volume."""
    h, w = shape[-2:]
    n = int(np.prod(shape[:-2], dtype=np.int64)) if len(shape) > 2 else 1
    from mie_b200 import synthetic

    return synthetic.vessel_volume((n, h, w), dtype, seed, tubes=6).reshape(shape)


# ------------------------------------------------------------------------------------------------ twin (CPU)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_line_loops_equal_scipy(dtype):
    S = _S()
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 5, 9, 40):
        x = (rng.standard_normal((3, n)) * 1000).astype(dtype)
        for sigma in (0.7, 1.0, 3.0, 9.0):
            r, w0, w1 = S._hessian_taps(sigma)
            assert 3 <= r <= 36
            for mode in MODES:
                for cval in ((0.0, 2.5) if mode == "constant" else (0.0,)):
                    kw = dict(mode=mode, cval=cval, truncate=4.0)
                    ref0 = gaussian_filter1d(x, sigma, order=0, **kw)
                    ref1 = gaussian_filter1d(x, sigma, order=1, **kw)
                    got0 = T.sym_line(x, w0, -1, mode, cval)
                    got1 = T.anti_line(x, w1, -1, mode, cval)
                    assert got0.dtype == ref0.dtype and np.array_equal(got0, ref0), (n, sigma, mode, cval)
                    assert got1.dtype == ref1.dtype and np.array_equal(got1, ref1), (n, sigma, mode, cval)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_axis_order_composition_equals_gaussian_filter(dtype):
    S = _S()
    x = (np.random.default_rng(2).standard_normal((7, 9, 11)) * 300).astype(dtype)
    for sigma in (0.7, 2.0):
        _, w0, w1 = S._hessian_taps(sigma)
        for order in [(1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0)]:
            for mode, cval in [("reflect", 0.0), ("constant", -3.0), ("wrap", 0.0), ("mirror", 0.0)]:
                y = x
                for ax, o in enumerate(order):
                    y = (T.anti_line if o else T.sym_line)(y, w1 if o else w0, ax, mode, cval)
                ref = gaussian_filter(x, sigma, order=order, mode=mode, cval=cval, truncate=4.0)
                assert np.array_equal(y, ref), (sigma, order, mode)


def test_package_taps_are_scipys():
    from scipy.ndimage._filters import _gaussian_kernel1d

    S = _S()
    for sigma in (0.3, 0.7, 1.0, 1.5, 3.0, 9.0, 16.0):
        r, w0, w1 = S._hessian_taps(sigma)
        assert r == int(4.0 * sigma + 0.5)
        assert np.array_equal(w0, _gaussian_kernel1d(sigma, 0, r)[::-1])
        assert np.array_equal(w1, _gaussian_kernel1d(sigma, 1, r)[::-1])
        assert np.array_equal(w0, w0[::-1]) and np.array_equal(w1, -w1[::-1])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_twin_2d_closed_form_within_4_ulp_of_eigvalsh(dtype):
    H = T.hessian_matrix(_planes((48, 52), np.int16, 3).astype(dtype), 1.5, mode="reflect")
    e = T.hessian_matrix_eigvals(H)
    m = np.stack([np.stack([H[0], H[1]], -1), np.stack([H[1], H[2]], -1)], -2).astype(np.float64)
    ref = np.moveaxis(np.linalg.eigvalsh(m)[..., ::-1], -1, 0)
    scale = np.abs(ref).max(0)
    assert e.dtype == dtype
    assert np.all(np.abs(e - ref) <= 4 * np.finfo(dtype).eps * scale)


# ------------------------------------------------------------------------------------------------ ABI (CPU)
H, W, D = 40, 48, 9
PAD = W + 24


def _taps(sigma=1.0):
    r, w0, w1 = _S()._hessian_taps(sigma)
    return np.array([sigma]), np.array([r], np.int32), w0, w1


def _call2(n, s=(H * W, W), d=(H * W, W), sd=U16, dd=F64, filt=0, nsc=1, taps=None, mode=4, sp=FAKE, dp=FAKE,
           ws=FAKE, nbytes=1 << 40, h=H, w=W, gamma=-1.0):
    sig, rad, w0, w1 = taps or _taps()
    return _lib().mie_sk_ridge_filter(sp, dp, sd, dd, n, h, w, *s, *d, filt, nsc,
                                      None if sig is None else sig.ctypes.data, None if rad is None else rad.ctypes.data,
                                      w0.ctypes.data, w1.ctypes.data, mode, 0.0, 1, 0.5, 0.5, gamma, ws, nbytes, None)


def _call3(n, s=None, d=None, sd=U16, dd=F64, filt=0, nsc=1, taps=None, mode=4, sp=FAKE, dp=FAKE, ws=FAKE,
           nbytes=1 << 40, gamma=-1.0):
    dense = (D * H * W, H * W, W)
    sig, rad, w0, w1 = taps or _taps()
    return _lib().mie_sk_ridge_filter3d(sp, dp, sd, dd, n, D, H, W, *(s or dense), *(d or dense), filt, nsc,
                                        sig.ctypes.data, rad.ctypes.data, w0.ctypes.data, w1.ctypes.data, mode, 0.0, 1,
                                        0.5, 0.5, gamma, ws, nbytes, None)


def test_workspace_query_does_not_grow_with_n():
    L = _lib()
    for sd, fsz in ((U8, 8), (U16, 8), (I16, 8), (F32, 4)):
        one = L.mie_sk_ridge_filter3d_workspace_bytes(1, 512, 512, 512, sd)
        assert one == 9 * 512 ** 3 * fsz + 2 * 256
        for n in (2, 100, 10 ** 6):
            assert L.mie_sk_ridge_filter3d_workspace_bytes(n, 512, 512, 512, sd) == one
        assert L.mie_sk_hessian_matrix3d_workspace_bytes(10 ** 6, 512, 512, 512, sd) == 5 * 512 ** 3 * fsz
        big = L.mie_sk_ridge_filter_workspace_bytes(10 ** 6, 512, 512, sd)
        # planes keep their running maximum in float64 whatever the image type
        assert big == L.mie_sk_ridge_filter_workspace_bytes(64, 512, 512, sd) == (4 * fsz + 8) * (1 << 24) + 2 * 512
        assert L.mie_sk_ridge_filter_workspace_bytes(1, 512, 512, sd) < big
        assert L.mie_sk_hessian_matrix_workspace_bytes(10 ** 6, 512, 512, sd) == 3 * (1 << 24) * fsz
        small = L.mie_sk_ridge_filter3d_workspace_bytes(10 ** 6, 8, 8, 8, sd)
        assert small == L.mie_sk_ridge_filter3d_workspace_bytes(32768, 8, 8, 8, sd) == 9 * (1 << 24) * fsz + 2 * 32768 * 8
    for bad in [(0, 8, 8, U8), (-1, 8, 8, U8), (1, 0, 8, U8), (1, 8, 0, U8), (1, 8, 8, F64), (1, 8, 8, -1)]:
        assert L.mie_sk_ridge_filter_workspace_bytes(*bad) == 0, bad
        assert L.mie_sk_hessian_matrix_workspace_bytes(*bad) == 0, bad


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_dtype_filter_and_mode_codes(call):
    for sd in (U8, U16, I16, F32):
        for dd in (F64, F32):
            assert call(1, sd=sd, dd=dd, nbytes=16) == E_WORKSPACE, (sd, dd)
        assert call(1, sd=sd, dd=sd if sd != F32 else U8, nbytes=16) == E_DTYPE, sd
    for sd in (F64, 5, -1):
        assert call(1, sd=sd, nbytes=16) == E_DTYPE, sd
    for filt in (0, 1, 2, 3):
        assert call(1, filt=filt, nbytes=16) == E_WORKSPACE, filt
    for filt in (-1, 4):
        assert call(1, filt=filt) == E_UNSUPPORTED, filt
    for mode in range(5):
        assert call(1, mode=mode, nbytes=16) == E_WORKSPACE, mode
    for mode in (-1, 5):
        assert call(1, mode=mode) == E_BORDER, mode


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_scale_codes(call):
    from scipy.ndimage._filters import _gaussian_kernel1d

    sig, rad, w0, w1 = _taps(16.0)
    assert rad[0] == 64 and call(1, taps=(sig, rad, w0, w1), nbytes=16) == E_WORKSPACE
    big = (np.array([16.2]), np.array([65], np.int32), _gaussian_kernel1d(16.2, 0, 65)[::-1].copy(),
           _gaussian_kernel1d(16.2, 1, 65)[::-1].copy())
    assert call(1, taps=big) == E_KERNEL
    sig, rad, w0, w1 = _taps(1.0)
    assert call(1, taps=(sig, np.array([-1], np.int32), w0, w1)) == E_KERNEL
    assert call(1, taps=(sig, rad, w1, w1)) == E_KERNEL          # order-0 taps not symmetric
    assert call(1, taps=(sig, rad, w0, w0)) == E_KERNEL          # order-1 taps not antisymmetric
    lop = w0.copy()
    lop[0] += 1e-3
    assert call(1, taps=(sig, rad, lop, w1)) == E_KERNEL
    for s in (-1.0, float("nan"), float("inf")):
        assert call(1, taps=(np.array([s]), rad, w0, w1)) == E_RANGE, s
    assert call(1, nsc=-1) == E_SHAPE
    assert call(1, nsc=0, nbytes=16) == E_WORKSPACE                # empty sigmas still write the output
    two = (np.array([1.0, 3.0]), np.array([4, 12], np.int32), np.concatenate([w0, _taps(3.0)[2]]),
           np.concatenate([w1, _taps(3.0)[3]]))
    assert call(1, nsc=2, taps=two, nbytes=16) == E_WORKSPACE
    assert call(1, nsc=2, taps=(two[0], two[1], np.concatenate([w0, w0, w0, w0]), two[3])) == E_KERNEL


def test_null_pointers_strides_and_workspace():
    sig, rad, w0, w1 = _taps()
    L = _lib()
    args = (FAKE, FAKE, U16, F64, 1, H, W, H * W, W, H * W, W, 0, 1)
    tail = (rad.ctypes.data, w0.ctypes.data, w1.ctypes.data, 4, 0.0, 1, 0.5, 0.5, -1.0, FAKE, 1 << 40, None)
    assert L.mie_sk_ridge_filter(*args, None, *tail) == E_NULL
    assert _call2(1, sp=None) == E_NULL
    assert _call2(1, dp=None) == E_NULL
    assert _call2(1, ws=None) == E_NULL
    assert _call2(1, ws=FAKE + 8) == E_ALIGN
    assert _call3(1, ws=FAKE + 128) == E_ALIGN
    need = L.mie_sk_ridge_filter_workspace_bytes(2, H, W, U16)
    assert _call2(2, nbytes=need - 1) == E_WORKSPACE
    need3 = L.mie_sk_ridge_filter3d_workspace_bytes(2, D, H, W, F32)
    assert _call3(2, sd=F32, dd=F32, nbytes=need3 - 1) == E_WORKSPACE
    assert _call2(0, sp=None, dp=None, ws=None, nbytes=0) == 0
    assert _call3(0, sp=None, dp=None, ws=None, nbytes=0) == 0
    tight = (H - 1) * PAD + W
    for s in [(H * (W - 1), W - 1), (tight - 1, PAD)]:
        assert _call2(2, s=s, d=(tight, PAD)) == E_STRIDE, s
        assert _call2(2, s=(tight, PAD), d=s) == E_STRIDE, s
    assert _call2(2, s=(tight, PAD), d=(tight, PAD), nbytes=16) == E_WORKSPACE
    slice_ = (H - 1) * PAD + W
    assert _call3(2, s=((D - 1) * slice_ + slice_ - 1, slice_, PAD)) == E_STRIDE
    assert _call3(1, d=(D * slice_, slice_ - 1, PAD)) == E_STRIDE


def test_hessian_matrix_and_eigvals_codes():
    L = _lib()
    r, w0, w1 = _S()._hessian_taps(1.0)
    n = 2
    ext = (n - 1) * H * W + H * W

    def hm(sd=U16, dd=F64, se=ext, rad=r, a=w0, b=w1, mode=0, ws=FAKE, nbytes=1 << 40, sp=FAKE):
        return L.mie_sk_hessian_matrix(sp, FAKE, sd, dd, n, H, W, H * W, W, H * W, W, se, rad, a.ctypes.data,
                                       b.ctypes.data, mode, 0.0, ws, nbytes, None)

    assert hm(nbytes=16) == E_WORKSPACE
    assert hm(sd=F32, dd=F32, nbytes=16) == E_WORKSPACE
    assert hm(dd=F32) == E_DTYPE and hm(sd=F32, dd=F64) == E_DTYPE
    assert hm(se=ext - 1) == E_STRIDE
    assert hm(rad=65) == E_KERNEL
    assert hm(a=w1) == E_KERNEL
    assert hm(mode=7) == E_BORDER
    assert hm(ws=FAKE + 4) == E_ALIGN
    assert hm(sp=None) == E_NULL
    assert hm(nbytes=L.mie_sk_hessian_matrix_workspace_bytes(n, H, W, U16) - 1) == E_WORKSPACE
    d3 = L.mie_sk_hessian_matrix3d(FAKE, FAKE, I16, F64, 1, D, H, W, D * H * W, H * W, W, D * H * W, H * W, W,
                                   D * H * W, r, w0.ctypes.data, w1.ctypes.data, 0, 0.0, FAKE, 16, None)
    assert d3 == E_WORKSPACE
    ev = L.mie_sk_hessian_eigvals
    assert ev(FAKE, FAKE, U16, 2, 10, 10, 10, None) == E_DTYPE
    assert ev(FAKE, FAKE, F64, 4, 10, 10, 10, None) == E_SHAPE
    assert ev(FAKE, FAKE, F64, 3, -1, 10, 10, None) == E_SHAPE
    assert ev(None, FAKE, F64, 3, 10, 10, 10, None) == E_NULL
    assert ev(FAKE, None, F32, 2, 10, 10, 10, None) == E_NULL
    assert ev(FAKE, FAKE, F32, 2, 10, 9, 10, None) == E_STRIDE
    assert ev(FAKE, FAKE, F32, 2, 10, 10, 9, None) == E_STRIDE
    assert ev(None, None, F32, 2, 0, 0, 0, None) == 0


# ------------------------------------------------------------------------------------------------ Python (CPU)
def test_python_argument_errors():
    S = _S()
    x = torch.zeros(16, 16, dtype=torch.uint16)
    for f in (S.frangi, S.hessian, S.sato, S.meijering):
        with pytest.raises(ValueError, match="less than zero"):
            f(x, sigmas=[1, -1])
        with pytest.raises(ValueError, match="mode"):
            f(x, mode="edge")
        with pytest.raises(NotImplementedError):
            f(x, sigmas=[16.5])                      # radius 66
        with pytest.raises(NotImplementedError):
            f(x, sigmas=[0.0])
        with pytest.raises(RuntimeError, match="CUDA tensor"):
            f(x)
        with pytest.raises(ValueError, match="volumetric=True"):
            f(x, volumetric=True)
    with pytest.raises(ValueError, match="less than zero"):
        S.frangi(x, scale_range=(-1, 3), scale_step=2)
    for ugd in (None, False):
        with pytest.raises(NotImplementedError):
            S.hessian_matrix(x, 1.0, use_gaussian_derivatives=ugd)
    with pytest.raises(NotImplementedError):
        S.hessian_matrix(x, 1.0, order="xy", use_gaussian_derivatives=True)
    with pytest.raises(ValueError):
        S.hessian_matrix(x, 1.0, order="ij", use_gaussian_derivatives=True)
    with pytest.raises(ValueError, match="less than zero"):
        S.hessian_matrix(x, -1.0, use_gaussian_derivatives=True)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        S.hessian_matrix(x, 1.0, use_gaussian_derivatives=True)
    with pytest.raises(ValueError, match="3 .2-D. or 6"):
        S.hessian_matrix_eigvals([x.double()] * 4)
    with pytest.raises(TypeError):
        S.hessian_matrix_eigvals([x.double()] * 3)          # host tensors
    for name in ("frangi", "hessian", "sato", "meijering", "hessian_matrix", "hessian_matrix_eigvals"):
        assert name in S.__all__


# ------------------------------------------------------------------------------------------------ GPU helpers
def _eps(dtype):
    return np.finfo(np.float32 if np.dtype(dtype) == np.float32 else np.float64).eps


def _near_ties(img, sigmas, kind, mode="reflect", cval=0, black_ridges=True, alpha=None):
    """Voxels of a 3-D image where, at some sigma, the twin's order by |lambda| (frangi / hessian) or meijering's
    argmax of |.| is decided by a gap below twice the eigenvalue bound."""
    f = img.astype(T._float_type(img.dtype))
    if not black_ridges:
        f = -f
    near = np.zeros(img.shape, bool)
    for sigma in sigmas:
        e = T._hessian_eigvals(f, sigma, mode, cval).astype(np.float64)
        bound = 2 * 64 * _eps(img.dtype) * np.abs(e).max(0)
        if kind == "meijering":
            a = 1 / 4 if alpha is None else alpha
            v = np.abs(np.tensordot(T.linalg.circulant([1, a, a]), e, 1))
            v.sort(0)
            near |= v[-1] - v[-2] <= bound * (1 + 2 * a)
        else:
            a = np.sort(np.abs(e), 0)
            near |= (np.diff(a, axis=0) <= bound).any(0)
    return near


def _compare(got, ref, tol, near=None, what=""):
    """|got - ref| <= tol (a scalar or per voxel) everywhere except at counted near-tie voxels (at most 1e-5 of the
    voxels)."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    bad = ~(np.abs(got - ref) <= tol)
    if near is None:
        assert not bad.any(), f"{what}: {int(bad.sum())} voxels beyond {np.max(tol):.1e}, " \
                              f"max {np.abs(got - ref).max():.3e}"
        return
    assert not (bad & ~near).any(), f"{what}: {int((bad & ~near).sum())} voxels beyond {np.max(tol):.1e} away from " \
                                    f"ties, max {np.abs(got - ref)[~near].max():.3e}"
    ties = int((bad & near).sum())
    print(f"{what}: {ties} near-tie voxels of {bad.size} differ")
    assert ties <= 1e-5 * bad.size, (what, ties)


def _sato_sqrt_tol(img, sigmas, mode, cval, black_ridges):
    """Per voxel: the largest sigma^2 sqrt(E (|e0| + |e1| + E)) over the sigmas, E = 64 eps max|lambda|."""
    f = img.astype(T._float_type(img.dtype))
    if not black_ridges:
        f = -f
    tol = np.zeros(img.shape)
    for sigma in sigmas:
        e = T._hessian_eigvals(f, sigma, mode, cval).astype(np.float64)
        E = 64 * _eps(img.dtype) * np.abs(e).max(0)
        tol = np.maximum(tol, sigma ** 2 * np.sqrt(E * (np.abs(e[0]) + np.abs(e[1]) + E)))
    return tol


def _tol(kind, dtype, ndim, ref):
    if np.dtype(dtype) == np.float32:
        t = 1e-4
    else:
        t = 1e-14 if ndim == 2 else 1e-9
    if kind in ("sato", "meijering"):
        t *= max(float(np.abs(ref).max()), 1e-300)
    return t


def _run(kind, x, dev, volumetric, **kw):
    f = getattr(_S(), kind)
    return f(torch.from_numpy(np.ascontiguousarray(x)).to(dev), volumetric=volumetric, **kw)


def _check_filter(kind, x, dev, volumetric, **kw):
    """Every image (last 2 / 3 axes) of the batch against the twin."""
    out = _run(kind, x, dev, volumetric, **kw)
    per = 3 if volumetric else 2
    assert out.shape == x.shape and out.dtype == (torch.float32 if x.dtype == np.float32 else torch.float64)
    got = out.cpu().numpy().reshape((-1,) + x.shape[-per:])
    xs = x.reshape((-1,) + x.shape[-per:])
    twin_kw = {k: v for k, v in kw.items() if k != "out_dtype"}
    sig = list(kw.get("sigmas", range(1, 10, 2)))
    if "scale_range" in kw:
        sig = list(np.arange(kw["scale_range"][0], kw["scale_range"][1], kw["scale_step"]))
    for i in range(xs.shape[0]):
        ref = getattr(T, kind)(xs[i], **twin_kw)
        tol = _tol(kind, x.dtype, per, ref)
        g = got[i]
        if kind == "hessian":
            pre = T.frangi(xs[i], **{"gamma": 15, **twin_kw})
            cancel = pre <= 64 * _eps(x.dtype)
            assert np.all((g[cancel] == 1) | (np.abs(g[cancel]) <= 64 * _eps(x.dtype))), f"hessian image {i}"
            print(f"hessian image {i}: {int(cancel.sum())} voxels of {cancel.size} within 64 eps of 0 before the "
                  f"replacement, {int((g[cancel] != ref[cancel]).sum())} of them differ")
            g = np.where(cancel, ref, g)
        if volumetric and kind == "sato":
            tol = np.maximum(tol, _sato_sqrt_tol(xs[i], sig, kw.get("mode", "reflect"), kw.get("cval", 0),
                                                 kw.get("black_ridges", True)))
        near = None
        if volumetric and kind in ("frangi", "hessian", "meijering"):
            near = _near_ties(xs[i], sig, kind, kw.get("mode", "reflect"), kw.get("cval", 0),
                              kw.get("black_ridges", True), kw.get("alpha"))
        _compare(g, ref, tol, near, f"{kind} image {i}")
    return out


# ------------------------------------------------------------------------------------------------ GPU: Hessian
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("volumetric", [False, True], ids=["planes", "volumes"])
def test_hessian_elements_and_eigvals_match_the_twin(dev, dtype, volumetric):
    S = _S()
    shape = (2, 11, 17, 14) if volumetric else (2, 37, 29)
    x = _image(shape, dtype, 4) if volumetric else _planes(shape, dtype, 4)
    xt = torch.from_numpy(x).to(dev)
    per = 3 if volumetric else 2
    for sigma in (0.7, 1, 3, 9):
        for mode in MODES:
            for cval in ((0.0, 0.37) if mode == "constant" else (0.0,)):
                H = S.hessian_matrix(xt, sigma, mode=mode, cval=cval, use_gaussian_derivatives=True,
                                     volumetric=volumetric)
                assert len(H) == per * (per + 1) // 2
                got = [h.cpu().numpy() for h in H]
                E = S.hessian_matrix_eigvals(H).cpu().numpy()
                for i in range(shape[0]):
                    ref = T.hessian_matrix(x[i], sigma, mode=mode, cval=cval)
                    for k, (g, r) in enumerate(zip(got, ref)):
                        assert g[i].dtype == r.dtype and np.array_equal(g[i], r), (sigma, mode, cval, i, k)
                    ev = T.hessian_matrix_eigvals(ref)
                    if per == 2:
                        assert np.array_equal(E[:, i], ev), (sigma, mode, i)
                    else:
                        bound = 64 * _eps(dtype) * np.abs(ev.astype(np.float64)).max(0)
                        assert np.all(np.abs(E[:, i].astype(np.float64) - ev) <= bound), (sigma, mode, i)


# ------------------------------------------------------------------------------------------------ GPU: filters
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("kind", ["frangi", "hessian", "sato", "meijering"])
def test_filters_on_planes_match_the_twin(dev, kind, dtype):
    x = _planes((3, 45, 38), dtype, 5)
    _check_filter(kind, x, dev, False)
    _check_filter(kind, x, dev, False, sigmas=[0.7, 2], black_ridges=False, mode="constant", cval=3.0)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("kind", ["frangi", "hessian", "sato", "meijering"])
def test_filters_on_volumes_match_the_twin(dev, kind, dtype):
    x = _image((2, 14, 24, 21), dtype, 6)
    _check_filter(kind, x, dev, True)
    _check_filter(kind, x, dev, True, sigmas=[1, 2.5], black_ridges=False, mode="nearest")


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True], ids=["planes", "volumes"])
def test_filter_options_match_the_twin(dev, volumetric):
    shape = (2, 12, 26, 23) if volumetric else (3, 41, 36)
    for dtype in (np.int16, np.float32):
        x = _image(shape, dtype, 7) if volumetric else _planes(shape, dtype, 7)
        for kind, kw in [("frangi", dict(gamma=30.0)), ("frangi", dict(sigmas=[1, 3])),
                         ("frangi", dict(sigmas=[3, 1])), ("frangi", dict(alpha=0.3, beta=0.8, sigmas=[2])),
                         ("frangi", dict(scale_range=(1, 4), scale_step=1.5)), ("hessian", dict(gamma=None)),
                         ("hessian", dict(sigmas=[1.5], mode="wrap")), ("sato", dict(sigmas=[0.7, 3], mode="mirror")),
                         ("meijering", dict(alpha=0.1, sigmas=[1, 2])),
                         ("frangi", dict(mode="constant", cval=-50.0, black_ridges=False, sigmas=[1, 2]))]:
            _check_filter(kind, x, dev, volumetric, **kw)
        # gamma from the first sigma: the order of the sigmas changes the result
        a = _run("frangi", x, dev, volumetric, sigmas=[1, 3])
        b = _run("frangi", x, dev, volumetric, sigmas=[3, 1])
        assert not torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True], ids=["planes", "volumes"])
def test_constant_empty_and_batched_images(dev, volumetric):
    S = _S()
    shape = (2, 9, 16, 15) if volumetric else (2, 20, 18)
    for dtype in (torch.uint16, torch.float32):
        c = torch.full(shape, 700 if dtype == torch.uint16 else 0.25, dtype=dtype, device=dev)
        for kind in ("frangi", "sato", "meijering"):
            assert bool((getattr(S, kind)(c, volumetric=volumetric) == 0).all()), kind
        assert bool((S.hessian(c, volumetric=volumetric) == 1).all())
        x = torch.from_numpy(_image(shape, np.int16, 8) if volumetric else _planes(shape, np.int16, 8)).to(dev)
        for kind, one in (("frangi", 0), ("sato", 0), ("meijering", 0), ("hessian", 1)):
            e = getattr(S, kind)(x, sigmas=[], volumetric=volumetric)
            assert e.dtype == torch.float64 and bool((e == one).all()), kind
    # per-image gamma and maxima: images of very different contrast in one batch
    x = _image(shape, np.int16, 9) if volumetric else _planes(shape, np.int16, 9)
    x = x.copy()
    x[1] = (x[1].astype(np.int32) // 8).astype(np.int16)
    for kind in ("frangi", "meijering"):
        out = _check_filter(kind, x, dev, volumetric, sigmas=[1, 2])
        alone = getattr(S, kind)(torch.from_numpy(x[1].copy()).to(dev), sigmas=[1, 2], volumetric=volumetric)
        assert torch.equal(out[1], alone)


@pytest.mark.gpu
def test_out_dtype_and_repeatable_bits(dev):
    S = _S()
    x = torch.from_numpy(_image((3, 20, 30, 28), np.uint16, 10)).to(dev)
    a = S.frangi(x, volumetric=True)
    b = S.frangi(x, volumetric=True)
    assert torch.equal(a, b)
    m1, m2 = S.meijering(x, volumetric=True), S.meijering(x, volumetric=True)
    assert torch.equal(m1, m2)
    f = S.frangi(x, volumetric=True, out_dtype=torch.float32)
    assert f.dtype == torch.float32 and torch.equal(f, a.to(torch.float32))
    with pytest.raises(TypeError):
        S.frangi(x, out_dtype=torch.uint16)


def _canvas(t, dev, off, pad_row, pad_slice, volumetric, fill=0):
    shape = t.shape
    h, w = shape[-2:]
    d = shape[1] if volumetric else 1
    sh = w + pad_row
    sd = h * sh + pad_slice
    sn = d * sd + pad_slice if volumetric else sd
    canvas = torch.full((off + shape[0] * sn + 64,), fill, dtype=t.dtype, device=dev)
    strides = (sn, sd, sh, 1) if volumetric else (sn, sh, 1)
    view = canvas.as_strided(shape, strides, off)
    view.copy_(t)
    return canvas, view, ((sn, sd, sh) if volumetric else (sn, sh))


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True], ids=["planes", "volumes"])
@pytest.mark.parametrize("layout", [(0, 16, 0, 8), (0, 8, 40, 0), (1, 3, 7, 3)], ids=["padded-rows", "padded-slices",
                                                                                      "unaligned"])
def test_non_dense_layouts_equal_the_dense_call(dev, volumetric, layout):
    S = _S()
    off, pad_row, pad_slice, doff = layout
    x = torch.from_numpy(_image((2, 9, 23, 21), np.int16, 11) if volumetric else _planes((2, 33, 27), np.int16, 11))
    x = x.to(dev)
    sig = [1.0, 2.0]
    dense = S.frangi(x, sigmas=sig, volumetric=volumetric)
    dense_h = S.hessian_matrix(x, 1.5, mode="constant", cval=0.1, use_gaussian_derivatives=True,
                               volumetric=volumetric)
    _, sv, sstr = _canvas(x, dev, off, pad_row, pad_slice, volumetric)
    dc, dv, dstr = _canvas(torch.zeros(x.shape, dtype=torch.float64, device=dev), dev, doff, pad_row + 1,
                           pad_slice + 2, volumetric, float("nan"))
    dv.fill_(float("nan"))
    L = _lib()
    n, dims = x.shape[0], tuple(x.shape[1:])
    taps = [S._hessian_taps(s) for s in sig]
    sig_a = np.asarray(sig)
    radii = np.asarray([t[0] for t in taps], np.int32)
    t0 = np.concatenate([t[1] for t in taps])
    t1 = np.concatenate([t[2] for t in taps])
    st = torch.cuda.current_stream().cuda_stream
    if volumetric:
        ws = torch.empty(L.mie_sk_ridge_filter3d_workspace_bytes(n, *dims, I16), dtype=torch.uint8, device=dev)
        rc = L.mie_sk_ridge_filter3d(sv.data_ptr(), dv.data_ptr(), I16, F64, n, *dims, *sstr, *dstr, 0, 2,
                                     sig_a.ctypes.data, radii.ctypes.data, t0.ctypes.data, t1.ctypes.data, 4, 0.0, 1,
                                     0.5, 0.5, -1.0, ws.data_ptr(), ws.numel(), st)
    else:
        ws = torch.empty(L.mie_sk_ridge_filter_workspace_bytes(n, *dims, I16), dtype=torch.uint8, device=dev)
        rc = L.mie_sk_ridge_filter(sv.data_ptr(), dv.data_ptr(), I16, F64, n, *dims, *sstr, *dstr, 0, 2,
                                   sig_a.ctypes.data, radii.ctypes.data, t0.ctypes.data, t1.ctypes.data, 4, 0.0, 1,
                                   0.5, 0.5, -1.0, ws.data_ptr(), ws.numel(), st)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(dv, dense)
    outside = torch.ones_like(dc, dtype=torch.bool)
    outside.as_strided(x.shape, dv.stride(), doff).fill_(False)
    assert bool(torch.isnan(dc[outside]).all()), "a store landed outside the output"
    # hessian_matrix through the same non-dense source
    k = len(dense_h)
    he = torch.full((doff + k * x.numel() + 5,), float("nan"), dtype=torch.float64, device=dev)
    r, w0, w1 = S._hessian_taps(1.5)
    if volumetric:
        ws = torch.empty(L.mie_sk_hessian_matrix3d_workspace_bytes(n, *dims, I16), dtype=torch.uint8, device=dev)
        d_, h_, w_ = dims
        rc = L.mie_sk_hessian_matrix3d(sv.data_ptr(), he.data_ptr() + 8 * doff, I16, F64, n, *dims, *sstr,
                                       d_ * h_ * w_, h_ * w_, w_, x.numel(), r, w0.ctypes.data, w1.ctypes.data, 0, 0.1,
                                       ws.data_ptr(), ws.numel(), st)
    else:
        ws = torch.empty(L.mie_sk_hessian_matrix_workspace_bytes(n, *dims, I16), dtype=torch.uint8, device=dev)
        h_, w_ = dims
        rc = L.mie_sk_hessian_matrix(sv.data_ptr(), he.data_ptr() + 8 * doff, I16, F64, n, *dims, *sstr, h_ * w_, w_,
                                     x.numel(), r, w0.ctypes.data, w1.ctypes.data, 0, 0.1, ws.data_ptr(), ws.numel(),
                                     st)
    assert rc == 0
    torch.cuda.synchronize()
    got = he[doff:doff + k * x.numel()].reshape(k, *x.shape)
    assert bool(torch.isnan(he[:doff]).all() and torch.isnan(he[doff + k * x.numel():]).all())
    for e in range(k):
        assert torch.equal(got[e], dense_h[e]), e


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True], ids=["planes", "volumes"])
def test_graph_capture_equals_the_eager_call(dev, volumetric):
    S = _S()
    x = torch.from_numpy(_image((2, 10, 26, 24), np.uint16, 12) if volumetric else _planes((3, 40, 36), np.uint16,
                                                                                           12)).to(dev)
    sig = [1.0, 3.0]
    eager = {k: getattr(S, k)(x, sigmas=sig, volumetric=volumetric) for k in ("frangi", "meijering")}
    L = _lib()
    n, dims = x.shape[0], tuple(x.shape[1:])
    taps = [S._hessian_taps(s) for s in sig]
    sig_a = np.asarray(sig)
    radii = np.asarray([t[0] for t in taps], np.int32)
    t0 = np.concatenate([t[1] for t in taps])
    t1 = np.concatenate([t[2] for t in taps])
    if volumetric:
        need = L.mie_sk_ridge_filter3d_workspace_bytes(n, *dims, U16)
        d, h, w = dims
        layout = (n, d, h, w) + (d * h * w, h * w, w) * 2
        fn = L.mie_sk_ridge_filter3d
    else:
        need = L.mie_sk_ridge_filter_workspace_bytes(n, *dims, U16)
        h, w = dims
        layout = (n, h, w) + (h * w, w) * 2
        fn = L.mie_sk_ridge_filter
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    outs = {k: torch.empty(x.shape, dtype=torch.float64, device=dev) for k in eager}

    def launch():
        for k, code, alpha in (("frangi", 0, 0.5), ("meijering", 3, 1 / (len(dims) + 1))):
            rc = fn(x.data_ptr(), outs[k].data_ptr(), U16, F64, *layout, code, 2, sig_a.ctypes.data, radii.ctypes.data,
                    t0.ctypes.data, t1.ctypes.data, 4, 0.0, 1, alpha, 0.5, -1.0, ws.data_ptr(), ws.numel(),
                    torch.cuda.current_stream().cuda_stream)
            assert rc == 0

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        launch()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for _ in range(2):
        for o in outs.values():
            o.zero_()
        g.replay()
        torch.cuda.synchronize()
        for k in eager:
            assert torch.equal(outs[k], eager[k]), k


@pytest.mark.gpu
def test_batch_beyond_2_pow_31_elements(dev):
    S = _S()
    h, w = 512, 500
    n = 2 ** 31 // (h * w) + 12          # 8400 planes, 2.15e9 elements
    straddle = 2 ** 31 // (h * w)       # plane 8388 holds element 2^31
    assert straddle * h * w < 2 ** 31 < (straddle + 1) * h * w and n * h * w > 2 ** 31
    base = torch.from_numpy(_planes((8, h, w), np.uint8, 13)).to(dev)
    x = base.repeat(n // 8 + 1, 1, 1)[:n].contiguous()
    x[straddle] = torch.flip(x[straddle], (1,))
    out = S.frangi(x, sigmas=[1.5])
    assert out.shape == (n, h, w) and out.dtype == torch.float64
    for i in (0, n // 2, straddle, n - 1):
        one = S.frangi(x[i].clone(), sigmas=[1.5])
        assert torch.equal(out[i], one), i
        ref = T.frangi(x[i].cpu().numpy(), sigmas=[1.5])
        _compare(out[i].cpu().numpy(), ref, 1e-14, None, f"plane {i}")
    assert not torch.equal(out[straddle], out[straddle - 8])


@pytest.mark.gpu
def test_512_cubed_vessel_volume_interior_block(dev):
    from mie_b200 import synthetic

    S = _S()
    vol = synthetic.vessel_volume((512, 512, 512), np.int16, 0)
    sig = [1, 3]
    out = S.frangi(torch.from_numpy(vol).to(dev), sigmas=sig, gamma=40.0, black_ridges=False, volumetric=True)
    assert out.shape == (512, 512, 512) and out.dtype == torch.float64
    got = out.cpu().numpy()
    del out
    r_max = int(4 * max(sig) + 0.5)
    m = 2 * r_max
    # one block centred on the strongest response away from the faces, one at the centre
    inner = got[m:512 - m, m:512 - m, m:512 - m]
    peak = np.clip(np.array(np.unravel_index(np.argmax(inner), inner.shape)) + m - 32, m, 512 - 64 - m)
    for k, (z0, y0, x0) in enumerate([tuple(int(v) for v in peak), (224, 224, 224)]):
        block = vol[z0 - m:z0 + 64 + m, y0 - m:y0 + 64 + m, x0 - m:x0 + 64 + m]
        ref = T.frangi(block, sigmas=sig, gamma=40.0, black_ridges=False)[m:-m, m:-m, m:-m]
        near = _near_ties(block, sig, "frangi", black_ridges=False)[m:-m, m:-m, m:-m]
        _compare(got[z0:z0 + 64, y0:y0 + 64, x0:x0 + 64], ref, 1e-9, near, f"512^3 block at {(z0, y0, x0)}")
        if k == 0:
            assert ref.max() > 0.1   # the block holds a vessel


@pytest.mark.gpu
def test_live_pin_against_skimage(dev):
    filters = pytest.importorskip("skimage.filters")
    feature = pytest.importorskip("skimage.feature")
    x2 = _planes((40, 37), np.uint16, 14)
    x3 = _image((12, 20, 18), np.int16, 15)
    for x, volumetric in ((x2, False), (x3, True)):
        for kind in ("frangi", "hessian", "sato", "meijering"):
            up = getattr(filters, kind)(x, sigmas=[1, 2])
            tw = getattr(T, kind)(x, sigmas=[1, 2])
            got = _run(kind, x, dev, volumetric, sigmas=[1, 2]).cpu().numpy()
            np.testing.assert_allclose(tw, up, rtol=0, atol=1e-12 * max(1.0, np.abs(up).max()))
            np.testing.assert_allclose(got, up, rtol=0, atol=1e-9 * max(1.0, np.abs(up).max()))
        up_h = feature.hessian_matrix(x, 1.5, use_gaussian_derivatives=True)
        tw_h = T.hessian_matrix(x, 1.5)
        got_h = _S().hessian_matrix(torch.from_numpy(x).to(dev), 1.5, use_gaussian_derivatives=True,
                                    volumetric=volumetric)
        for u, t, g in zip(up_h, tw_h, got_h):
            assert np.array_equal(t, u) and np.array_equal(g.cpu().numpy(), u)
        up_e = feature.hessian_matrix_eigvals(up_h)
        np.testing.assert_allclose(T.hessian_matrix_eigvals(tw_h), up_e, rtol=0, atol=1e-12 * np.abs(up_e).max())
