"""Median with any footprint (filters.median / skimage_compat.median with a footprint, every scipy mode and cval;
mie_sk_median / mie_sk_median3d).

The reference is scipy.ndimage.median_filter itself: skimage.filters.median calls it (behavior='ndimage'), and a median
is pure selection, so every GPU output is compared value for value (np.array_equal) against scipy.

CPU: the cval casts and the rank / origin / border rules, pinned against the installed scipy through a numpy twin of the
kernel (ordered keys, MSB-first radix counting); disk / ball; the ABI's host validation with fake pointers; the Python
argument errors.  GPU: every dtype and mode over disk, ball, random sparse, even-extent, one-cell, line and box
footprints up to both bounds, cval casts, degenerate shapes, float specials, the dispatch to the 3x3(x3) kernels,
`out=`, non-dense layouts and batches, repeatable bits, graph capture, a batch beyond 2^31 elements, a 512^3 volume and a
live pin against scikit-image."""
import math
import warnings

import numpy as np
import pytest
import torch
from scipy import ndimage as ndi

U8, U16, I16, F32 = 0, 1, 2, 3
E_NULL, E_DTYPE, E_SHAPE, E_STRIDE, E_KERNEL, E_BORDER, E_RANGE = -1, -2, -3, -4, -7, -8, -10
FAKE = 0x10000   # never dereferenced: every call with it fails validation or has an empty batch
MODES = ["reflect", "mirror", "nearest", "wrap", "constant"]
BORDER = {"constant": 0, "mirror": 1, "nearest": 2, "wrap": 3, "reflect": 4}
DTYPES = [np.uint8, np.uint16, np.int16, np.float32]
CODE = {np.uint8: U8, np.uint16: U16, np.int16: I16, np.float32: F32}
TORCH = {np.uint8: torch.uint8, np.uint16: torch.uint16, np.int16: torch.int16, np.float32: torch.float32}


def _lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def _S():
    from mie_b200 import skimage_compat as S
    return S


def _F():
    from mie_b200 import filters as F
    return F


def _rand(dtype, shape, seed, lo=None, hi=None):
    r = np.random.default_rng(seed)
    if dtype == np.float32:
        return (r.standard_normal(shape) * 100).astype(np.float32)
    info = np.iinfo(dtype)
    return r.integers(info.min if lo is None else lo, (info.max if hi is None else hi) + 1, shape).astype(dtype)


def _scipy(x, fp, mode, cval=0.0):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return ndi.median_filter(x, footprint=np.asarray(fp, bool), mode=mode, cval=cval)


def _sparse(shape, seed, p=0.4):
    r = np.random.default_rng(seed)
    fp = r.random(shape) < p
    fp.flat[r.integers(fp.size)] = True
    return fp


# ------------------------------------------------------------------------------------------------ twin (CPU)
_PAD = {"reflect": "symmetric", "mirror": "reflect", "nearest": "edge", "wrap": "wrap", "constant": "constant"}


def _to_key(x):
    if x.dtype == np.float32:
        u = x.view(np.uint32).astype(np.uint64)
        return np.where(u >> 31, ~u & 0xFFFFFFFF, u | 0x80000000), 32
    if x.dtype == np.int16:
        return (x.view(np.uint16) ^ 0x8000).astype(np.uint64), 16
    return x.astype(np.uint64), 8 * x.itemsize


def _from_key(k, dtype):
    if dtype == np.float32:
        k = k.astype(np.uint64)
        return np.where(k >> 31, k ^ 0x80000000, ~k & 0xFFFFFFFF).astype(np.uint32).view(np.float32)
    if dtype == np.int16:
        return (k.astype(np.uint16) ^ 0x8000).view(np.int16)
    return k.astype(dtype)


def twin_median(x, fp, mode, cast_cval=0):
    """What the kernel computes, in numpy: pad by extent // 2 before and extent - 1 - extent // 2 after (the cast cval
    in 'constant'), ordered keys, and per output the largest key with at most count // 2 samples below it."""
    fp = np.asarray(fp, bool)
    pads = [(e // 2, e - 1 - e // 2) for e in fp.shape]
    if mode == "constant":
        xp = np.pad(x, pads, mode="constant", constant_values=np.array(cast_cval).astype(x.dtype))
    else:
        xp = np.pad(x, pads, mode=_PAD[mode])
    keys, bits = _to_key(xp)
    cells = np.argwhere(fp)
    samples = np.stack([keys[tuple(slice(c, c + s) for c, s in zip(cell, x.shape))] for cell in cells])
    rank = len(cells) // 2
    res = np.zeros(x.shape, np.uint64)
    for b in range(bits - 1, -1, -1):
        piv = res | np.uint64(1 << b)
        cnt = (samples < piv).sum(axis=0)
        res = np.where(cnt <= rank, piv, res)
    return _from_key(res, x.dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_twin_equals_scipy_in_every_mode(dtype):
    fps2 = [np.ones((3, 3)), _S().disk(2), _sparse((2, 4), 1), _sparse((5, 3), 2), np.ones((1, 4)), np.ones((1, 2)),
            [[0, 0, 1]], np.ones((7, 7))]
    fps3 = [_S().ball(1), _sparse((4, 4, 2), 3), np.ones((2, 1, 1))]
    for mode in MODES:
        for k, fp in enumerate(fps2):
            for shape in [(9, 11), (2, 3), (1, 5), (4, 1)]:
                x = _rand(dtype, shape, k)
                cv = _F().median_cval(TORCH[dtype], 3.0 if dtype != np.float32 else -2.5,
                                      np.asarray(fp, bool).sum() == 2 and np.asarray(fp, bool).all())
                c = 3.0 if dtype != np.float32 else -2.5
                assert np.array_equal(twin_median(x, fp, mode, cv), _scipy(x, fp, mode, c)), (mode, k, shape)
        for k, fp in enumerate(fps3):
            x = _rand(dtype, (5, 3, 6), 10 + k)
            assert np.array_equal(twin_median(x, fp, mode, 0), _scipy(x, fp, mode)), (mode, k)


def test_scipy_rank_and_fold_rules():
    """The rules include/mie.h states, as scipy 1.18.1 behaves."""
    assert np.array_equal(_scipy(np.array([1, 2, 3, 4], np.uint8), np.ones(4), "nearest"), [1, 2, 3, 4])
    x = np.array([[1, 2, 3], [4, 5, 6]], np.uint8)
    for mode in ("reflect", "mirror", "wrap"):
        assert _scipy(x, np.ones((7, 7)), mode).tolist() == [[4, 4, 4], [3, 3, 3]], mode
    assert _scipy(x, np.ones((7, 7)), "nearest").tolist() == [[3, 3, 3], [4, 4, 4]]
    # the cval is cast before selection: with 300 -> 44 the top-middle window holds 44 x3, 50 x2 and 200 x4
    col = np.array([[50, 200, 200]] * 3, np.uint8)
    assert _scipy(col, np.ones((3, 3)), "constant", 300)[0, 1] == 50
    with pytest.raises(RuntimeError, match="rank not within filter footprint size"):
        _scipy(x, np.zeros((3, 3)), "nearest")
    with pytest.raises(RuntimeError, match=r"footprint.ndim \(3\) must match len\(axes\) \(2\)"):
        _scipy(x, np.ones((3, 3, 3)), "nearest")


def test_scipy_reflect_reads_outside_the_image_far_beyond_short_axes():
    """At offset -2 n m (m >= 2) of an axis of length n > 1, scipy's 'reflect' reads neither the image nor the cval:
    the previous row's last sample here.  filters.median refuses footprints that reach that far in 'reflect'."""
    img = np.array([[5, 6], [7, 8], [9, 10]], np.int16)
    fp = np.zeros((1, 17), bool)
    fp[0, 0] = True   # offset -8 = -4 n
    out = _scipy(img, fp, "reflect", -7)
    assert out[1:, 0].tolist() == [6, 8]                          # the sample before each row: not cval, not the row
    assert _undefined_in_scipy((3, 2), fp, "reflect") and not _undefined_in_scipy((3, 3), fp, "reflect")
    fp[0, 0], fp[0, 1] = False, True                                # offset -7: an ordinary fold
    assert np.array_equal(_scipy(img, fp, "reflect"), twin_median(img, fp, "reflect"))


CVALS_INT = [300, -1, -2, 0.7, -0.7, 1000.7, -300.5, 255.9, 70000, -70000.5, -32769.0, 40000.7, 2.0 ** 31 - 1,
             -2.0 ** 31]


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16])
def test_cval_casts_equal_scipys(dtype):
    """An isolated cell at offset -1 puts the cast cval itself into the output at x = 0 (rank 0 of 1)."""
    F = _F()
    fp = np.array([[1, 0, 0]], bool)
    img = np.full((1, 3), 7, dtype)
    for c in CVALS_INT:
        want = int(_scipy(img, fp, "constant", c)[0, 0])
        assert F.median_cval(TORCH[dtype], c) == want, c
    # uint8: 300 -> 44, -1 -> 255, 0.7 -> 0; int16: -2.5 -> -2
    assert [F.median_cval(torch.uint8, c) for c in (300, -1, 0.7)] == [44, 255, 0]
    assert F.median_cval(torch.int16, -2.5) == -2
    for c in (float("inf"), float("-inf"), float("nan"), 2.0 ** 31, 1e10, -2.0 ** 31 - 1):
        with pytest.raises(NotImplementedError):
            F.median_cval(TORCH[dtype], c)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16])
def test_two_cell_box_compares_before_the_cast(dtype):
    """A two-cell all-ones footprint runs scipy's separable maximum filter: the double cval is compared first."""
    F = _F()
    info = np.iinfo(dtype)
    img = _rand(dtype, (3, 5), 4)
    for shape in [(1, 2), (2, 1)]:
        fp = np.ones(shape, bool)
        for c in (-1, -300.5, -70000.5, 0.7, float(info.min) - 0.5, 5.5):
            cv = F.median_cval(TORCH[dtype], c, True)
            assert np.array_equal(twin_median(img, fp, "constant", cv), _scipy(img, fp, "constant", c)), (shape, c)
        with pytest.raises(NotImplementedError):
            F.median_cval(TORCH[dtype], float(info.max) + 1, True)


def test_float32_cval_casts():
    F = _F()
    assert F.median_cval(torch.float32, 0.1) == float(np.float32(0.1))
    assert F.median_cval(torch.float32, 1e300) == math.inf and F.median_cval(torch.float32, -1e300) == -math.inf
    img = np.full((1, 3), -5, np.float32)
    for c in (0.1, 1e300, -1e300, 1e-46, -2.5):
        assert F.median_cval(torch.float32, c) == float(_scipy(img, [[1, 0, 0]], "constant", c)[0, 0]), c


def test_disk_and_ball():
    S = _S()
    assert [int(S.disk(r).sum()) for r in (1, 2, 3)] == [5, 13, 29]
    assert [int(S.ball(r).sum()) for r in (1, 2, 3)] == [7, 33, 123]
    assert int(S.ball(8).sum()) == 2109 and S.disk(32).shape == (65, 65) and S.ball(8).shape == (17, 17, 17)
    for r in (0, 1, 4, 7):
        g = np.arange(-r, r + 1)
        d = S.disk(r)
        assert d.dtype == np.uint8 and d.shape == (2 * r + 1,) * 2
        assert np.array_equal(d, (g[:, None] ** 2 + g[None, :] ** 2 <= r * r).astype(np.uint8))
        b = S.ball(r)
        assert b.dtype == np.uint8 and b.shape == (2 * r + 1,) * 3
        for z in range(2 * r + 1):
            assert np.array_equal(b[z], (g[:, None] ** 2 + g[None, :] ** 2 + g[z] ** 2 <= r * r).astype(np.uint8))


# ------------------------------------------------------------------------------------------------ ABI (CPU)
H, W, D = 20, 24, 6


def _fp(shape):
    a = np.ones(shape, np.uint8)
    return a, a.ctypes.data


def _c2(n=0, dtype=U16, s=(H * W, W), d=(H * W, W), fshape=(3, 3), fptr=None, mode=2, cval=0.0, sp=FAKE, dp=FAKE,
        h=H, w=W):
    a, p = _fp(fshape)
    return _lib().mie_sk_median(sp, dp, dtype, n, h, w, *s, *d, p if fptr is None else fptr, *fshape, mode, cval, None)


def _c3(n=0, dtype=U16, s=(D * H * W, H * W, W), d=(D * H * W, H * W, W), fshape=(3, 3, 3), fptr=None, mode=2,
        cval=0.0, sp=FAKE, dp=FAKE):
    a, p = _fp(fshape)
    return _lib().mie_sk_median3d(sp, dp, dtype, n, D, H, W, *s, *d, p if fptr is None else fptr, *fshape, mode, cval,
                                  None)


@pytest.mark.parametrize("call", [_c2, _c3], ids=["planes", "volumes"])
def test_abi_validation(call):
    nd = 2 if call is _c2 else 3
    bound = 65 if nd == 2 else 17
    assert call() == 0                                          # empty batch: a no-op after the checks
    for dt in (U8, U16, I16, F32):
        assert call(dtype=dt) == 0
    for dt in (-1, 4, 5):
        assert call(dtype=dt) == E_DTYPE
    assert call(fshape=(bound,) * nd) == 0
    for bad in [(bound + 1,) + (1,) * (nd - 1), (1,) * (nd - 1) + (bound + 1,), (0,) + (3,) * (nd - 1)]:
        assert call(fshape=bad) == E_KERNEL, bad
    empty = np.zeros((3,) * nd, np.uint8)
    assert call(fptr=empty.ctypes.data) == E_KERNEL
    for m in (-1, 5):
        assert call(mode=m) == E_BORDER
    for m in range(5):
        assert call(mode=m) == 0
    assert call(dtype=U8, cval=255.0) == 0 and call(dtype=U8, cval=256.0) == E_RANGE
    assert call(dtype=U8, cval=-1.0) == E_RANGE and call(dtype=U8, cval=0.5) == E_RANGE
    assert call(dtype=I16, cval=-32768.0) == 0 and call(dtype=I16, cval=32768.0) == E_RANGE
    assert call(dtype=U16, cval=65535.0) == 0 and call(dtype=U16, cval=float("nan")) == E_RANGE
    assert call(dtype=F32, cval=0.1) == E_RANGE and call(dtype=F32, cval=float(np.float32(0.1))) == 0
    assert call(dtype=F32, cval=float("inf")) == 0 and call(dtype=F32, cval=1e300) == E_RANGE
    assert call(n=1, sp=None) == E_NULL and call(n=1, dp=None) == E_NULL


def test_abi_null_footprint_and_strides():
    L = _lib()
    assert L.mie_sk_median(FAKE, FAKE, U8, 0, H, W, H * W, W, H * W, W, None, 3, 3, 2, 0.0, None) == E_NULL
    assert L.mie_sk_median3d(FAKE, FAKE, U8, 0, D, H, W, D * H * W, H * W, W, D * H * W, H * W, W, None, 3, 3, 3, 2,
                             0.0, None) == E_NULL
    assert _c2(n=2, s=(H * W, W - 1)) == E_STRIDE
    assert _c2(n=2, d=(H * W - 1, W)) == E_STRIDE
    assert _c2(n=2, s=(H * W + 7, W + 3), d=(H * W + 80, W + 4)) == E_STRIDE    # plane stride below (h-1) sh + w
    assert _c3(n=2, s=(D * H * W, H * W - 1, W)) == E_STRIDE
    assert _c3(n=2, d=(D * H * W - 1, H * W, W)) == E_STRIDE
    assert _c2(h=0) == E_SHAPE and _c2(w=0) == E_SHAPE and _c2(n=-1) == E_SHAPE


def test_host_tensors_are_refused():
    with pytest.raises(RuntimeError, match="CUDA"):
        _F().median(torch.zeros((4, 4), dtype=torch.uint8), np.ones((3, 3)), mode="reflect")


@pytest.mark.gpu
def test_python_argument_errors(dev):
    F = _F()
    x = torch.zeros((9, 9), dtype=torch.uint8, device=dev)
    v = torch.zeros((5, 9, 9), dtype=torch.uint8, device=dev)
    with pytest.raises(RuntimeError, match="rank not within filter footprint size"):
        F.median(x, np.zeros((3, 3)))
    with pytest.raises(RuntimeError, match=r"footprint.ndim \(3\) must match len\(axes\) \(2\)"):
        F.median(x, np.ones((3, 3, 3)))
    with pytest.raises(RuntimeError, match=r"footprint.ndim \(2\) must match len\(axes\) \(3\)"):
        F.median(v, np.ones((3, 3)))
    for mode in ("grid-wrap", "grid-mirror", "grid-constant", "foo"):
        with pytest.raises(NotImplementedError):
            F.median(x, np.ones((3, 3)), mode=mode)
    with pytest.raises(NotImplementedError):
        F.median(x, behavior="rank")
    with pytest.raises(NotImplementedError):
        F.median(x, np.ones((66, 1)))
    with pytest.raises(NotImplementedError):
        F.median(v, np.ones((18, 1, 1)))
    for c in (float("inf"), float("nan"), 1e10):
        with pytest.raises(NotImplementedError):
            F.median(x, np.ones((3, 3)), mode="constant", cval=c)
    F.median(x, np.ones((3, 3)), mode="reflect", cval=float("inf"))       # cval only matters in 'constant'
    with pytest.raises(NotImplementedError):
        F.median(v, _S().ball(1), halo_lo=v[0].contiguous())
    with pytest.raises(ValueError):
        F.median(x, _S().disk(1), out=x)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu(x, dev):
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def _undefined_in_scipy(shape, fp, mode):
    """scipy's 'reflect' reads outside the image at offsets -2 n m (m >= 2) of an axis of length n > 1."""
    return mode == "reflect" and any(1 < n <= e // 8 for n, e in zip(shape, np.asarray(fp).shape))


def _check(dev, x, fp, mode, cval=0.0, what=""):
    F = _F()
    if _undefined_in_scipy(x.shape, fp, mode):
        with pytest.raises(NotImplementedError):
            F.median(_gpu(x, dev), fp, mode=mode, cval=cval)
        return
    got = F.median(_gpu(x, dev), fp, mode=mode, cval=cval).cpu().numpy()
    ref = _scipy(x, fp, mode, cval)
    assert np.array_equal(got, ref), (what, mode, cval, x.dtype, np.asarray(fp).shape, int(np.sum(got != ref)))


FP2 = {"disk1": lambda: _S().disk(1), "disk2": lambda: _S().disk(2), "disk3": lambda: _S().disk(3),
       "disk4": lambda: _S().disk(4), "disk5": lambda: _S().disk(5), "sparse2x4": lambda: _sparse((2, 4), 5),
       "sparse7x6": lambda: _sparse((7, 6), 6, 0.3), "sparse4x4": lambda: _sparse((4, 4), 7, 0.5),
       "one-cell": lambda: np.ones((1, 1)), "corner": lambda: [[0, 0, 0], [0, 0, 0], [0, 0, 1]],
       "line1x7": lambda: np.ones((1, 7)), "line6x1": lambda: np.ones((6, 1)), "box3": lambda: np.ones((3, 3)),
       "box5": lambda: np.ones((5, 5)), "box2x4": lambda: np.ones((2, 4)), "pair1x2": lambda: np.ones((1, 2))}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", MODES)
def test_planes_match_scipy(dev, dtype, mode):
    for k, (name, make) in enumerate(FP2.items()):
        for shape in [(37, 45), (8, 70)]:
            _check(dev, _rand(dtype, shape, k), make(), mode, 0.0, name)


FP3 = {"ball1": lambda: _S().ball(1), "ball2": lambda: _S().ball(2), "ball3": lambda: _S().ball(3),
       "sparse4x4x2": lambda: _sparse((4, 4, 2), 8), "sparse3x5x4": lambda: _sparse((3, 5, 4), 9, 0.3),
       "one-cell": lambda: np.ones((1, 1, 1)), "line1x1x5": lambda: np.ones((1, 1, 5)),
       "line4x1x1": lambda: np.ones((4, 1, 1)), "box3": lambda: np.ones((3, 3, 3)), "box5": lambda: np.ones((5, 5, 5)),
       "box2x2x2": lambda: np.ones((2, 2, 2))}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode", MODES)
def test_volumes_match_scipy(dev, dtype, mode):
    for k, (name, make) in enumerate(FP3.items()):
        for shape in [(11, 13, 35), (3, 9, 40)]:
            _check(dev, _rand(dtype, shape, 20 + k), make(), mode, 0.0, name)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_footprints_at_the_bounds(dev, dtype):
    S = _S()
    for mode in MODES:
        x = _rand(dtype, (70, 75), 30)
        _check(dev, x, np.ones((65, 65)), mode, 0.0, "65x65")
        _check(dev, x, S.disk(32), mode, 0.0, "disk32")
        _check(dev, x, np.ones((65, 1)), mode, 0.0, "65x1")
        v = _rand(dtype, (19, 21, 34), 31)
        _check(dev, v, S.ball(8), mode, 0.0, "ball8")
        if mode in ("reflect", "constant"):
            _check(dev, v, np.ones((17, 17, 17)), mode, 0.0, "17^3")
            _check(dev, v, _sparse((17, 16, 17), 32, 0.2), mode, 0.0, "sparse17")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_constant_mode_cvals(dev, dtype):
    S = _S()
    if dtype == np.float32:
        cvals = [0.1, -2.5, 1e300, -1e300, float("inf"), 3.0, 1e-46]
    else:
        cvals = CVALS_INT + [0, 7]
    x = _rand(dtype, (23, 29), 40)
    v = _rand(dtype, (7, 9, 12), 41)
    for c in cvals:
        _check(dev, x, S.disk(2), "constant", c, "disk2")
        _check(dev, x, np.ones((3, 3)), "constant", c, "box3")
        _check(dev, x, _sparse((2, 4), 42), "constant", c, "sparse2x4")
        _check(dev, v, S.ball(1), "constant", c, "ball1")
        _check(dev, v, np.ones((3, 3, 3)), "constant", c, "box3^3")
    # two-cell boxes: scipy's separable maximum filter compares the double cval first
    for c in ([-1, -300.5, 5.5, 0.0] if dtype != np.float32 else [-1e300, 0.1, 1e300]):
        _check(dev, x, np.ones((1, 2)), "constant", c, "pair")
        _check(dev, v, np.ones((2, 1, 1)), "constant", c, "pair3d")
    col = np.array([[50, 200, 200]] * 3, np.uint8)
    if dtype == np.uint8:
        got = _F().median(_gpu(col, dev), np.ones((3, 3)), mode="constant", cval=300).cpu().numpy()
        assert got[0, 1] == 50


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
def test_small_and_degenerate_shapes(dev, dtype):
    S = _S()
    for mode in MODES:
        for shape in [(1, 1), (1, 9), (9, 1), (2, 3), (3, 33), (5, 65), (2, 97)]:
            x = _rand(dtype, shape, 50)
            for fp in (S.disk(3), np.ones((7, 7)), _sparse((5, 4), 51), np.ones((1, 2)), np.ones((65, 3))):
                _check(dev, x, fp, mode, 0.0, f"plane {shape}")
        for shape in [(1, 1, 1), (2, 1, 2), (1, 3, 5), (3, 2, 33), (2, 5, 1)]:
            v = _rand(dtype, shape, 52)
            for fp in (S.ball(2), np.ones((5, 5, 5)), _sparse((4, 4, 2), 53), np.ones((17, 1, 3))):
                _check(dev, v, fp, mode, 0.0, f"volume {shape}")


@pytest.mark.gpu
def test_float_specials(dev):
    S = _S()
    r = np.random.default_rng(60)
    specials = np.array([np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, 1.0, -1.0, 3.4e38, -3.4e38],
                        np.float32)
    x = r.choice(specials, (31, 40)).astype(np.float32)
    v = r.choice(specials, (6, 9, 33)).astype(np.float32)
    for mode in MODES:
        for fp in (S.disk(2), np.ones((2, 4)), np.ones((3, 3)), _sparse((3, 6), 61)):
            _check(dev, x, fp, mode, 0.0, "specials")
        for fp in (S.ball(1), np.ones((2, 2, 2))):
            _check(dev, v, fp, mode, 0.0, "specials 3d")
    _check(dev, x, S.disk(1), "constant", -np.inf, "specials cval")


@pytest.mark.gpu
def test_default_footprint_runs_the_3x3_kernels_and_the_new_kernel_agrees(dev, monkeypatch):
    F = _F()
    seen = []
    real = F.call

    def spy(device, name, *args):
        seen.append(name)
        return real(device, name, *args)

    monkeypatch.setattr(F, "call", spy)
    x2 = _gpu(_rand(np.uint16, (40, 50), 70), dev)
    x3 = _gpu(_rand(np.int16, (9, 20, 37), 71), dev)
    cases = [(x2, None, "nearest", 0.0, "mie_median2d"), (x2, np.ones((3, 3)), "nearest", 0.0, "mie_median2d"),
             (x2, torch.ones(3, 3), "constant", 0.0, "mie_median2d"), (x2, [[1] * 3] * 3, "constant", 0.4, "mie_median2d"),
             (x3, None, "nearest", 0.0, "mie_median3d"), (x3, np.ones((3, 3, 3)), "constant", 0.0, "mie_median3d"),
             (x2, None, "reflect", 0.0, "mie_sk_median"), (x2, None, "constant", 5.0, "mie_sk_median"),
             (x2, _S().disk(1), "nearest", 0.0, "mie_sk_median"), (x3, None, "wrap", 0.0, "mie_sk_median3d"),
             (x3, _S().ball(1), "nearest", 0.0, "mie_sk_median3d")]
    for x, fp, mode, cval, name in cases:
        seen.clear()
        out = F.median(x, fp, mode=mode, cval=cval)
        assert seen == [name], (name, seen)
        ref = _scipy(x.cpu().numpy(), np.ones((3,) * x.dim()) if fp is None else np.asarray(fp), mode, cval)
        assert np.array_equal(out.cpu().numpy(), ref)
    monkeypatch.undo()
    # the new kernel on the default footprint equals the old one bit for bit (float32 included)
    L = _lib()
    st = torch.cuda.current_stream().cuda_stream
    for dtype in DTYPES:
        for mode in ("nearest", "constant"):
            p = _gpu(_rand(dtype, (3, 33, 70), 72), dev)
            fp = np.ones((3, 3), np.uint8)
            new = torch.empty_like(p)
            assert L.mie_sk_median(p.data_ptr(), new.data_ptr(), CODE[dtype], 3, 33, 70, 33 * 70, 70, 33 * 70, 70,
                                   fp.ctypes.data, 3, 3, BORDER[mode], 0.0, st) == 0
            for i in range(3):
                assert torch.equal(new[i], F.median(p[i], mode=mode)), (dtype, mode, i)
            fp3 = np.ones((3, 3, 3), np.uint8)
            new3 = torch.empty_like(p)
            assert L.mie_sk_median3d(p.data_ptr(), new3.data_ptr(), CODE[dtype], 1, 3, 33, 70, 3 * 33 * 70, 33 * 70, 70,
                                     3 * 33 * 70, 33 * 70, 70, fp3.ctypes.data, 3, 3, 3, BORDER[mode], 0.0, st) == 0
            assert torch.equal(new3, F.median(p, mode=mode)), (dtype, mode)


@pytest.mark.gpu
def test_out_argument(dev):
    F = _F()
    x = _gpu(_rand(np.int16, (30, 41), 80), dev)
    out = torch.empty_like(x)
    assert F.median(x, _S().disk(3), out=out, mode="mirror") is out
    assert np.array_equal(out.cpu().numpy(), _scipy(x.cpu().numpy(), _S().disk(3), "mirror"))
    with pytest.raises(ValueError):
        F.median(x, _S().disk(3), out=torch.empty((30, 40), dtype=torch.int16, device=dev))
    with pytest.raises(ValueError):
        F.median(x, _S().disk(3), out=torch.empty_like(x, dtype=torch.uint16))
    big = torch.empty((2, 30, 41), dtype=torch.int16, device=dev)
    big[0].copy_(x)
    with pytest.raises(ValueError):
        F.median(big[0], _S().disk(3), out=big[0])
    F.median(big[0], _S().disk(3), out=big[1], mode="mirror")     # same storage, no overlap
    assert torch.equal(big[1], out)


def _canvas(shape, dtype, dev, off, pads, fill):
    """A strided view of `shape` at element offset `off` with each non-innermost stride grown by pads[i]."""
    strides = [1]
    for i in range(len(shape) - 1, 0, -1):
        strides.insert(0, strides[0] * shape[i] + pads[i - 1])
    size = off + sum((s - 1) * st for s, st in zip(shape, strides)) + 1 + 64
    canvas = torch.full((size,), fill, dtype=dtype, device=dev)
    return canvas, canvas.as_strided(shape, strides, off), strides


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
@pytest.mark.parametrize("layout", [(0, (7, 5)), (1, (0, 3)), (3, (13, 1))], ids=["padded", "unaligned", "odd"])
def test_non_dense_layouts_and_batches(dev, dtype, layout):
    L = _lib()
    off, pads = layout
    st = torch.cuda.current_stream().cuda_stream
    fill = 77 if dtype == np.uint8 else 77.0
    # planes: n = 3
    x = _rand(dtype, (3, 19, 43), 90)
    fp = _sparse((5, 6), 91).astype(np.uint8)
    _, sv, ss = _canvas(x.shape, TORCH[dtype], dev, off, pads, fill)
    sv.copy_(_gpu(x, dev))
    dc, dv, ds = _canvas(x.shape, TORCH[dtype], dev, off + 2, (pads[1] + 1, pads[0] + 2), fill)
    assert L.mie_sk_median(sv.data_ptr(), dv.data_ptr(), CODE[dtype], 3, 19, 43, ss[0], ss[1], ds[0], ds[1],
                           fp.ctypes.data, 5, 6, BORDER["wrap"], 0.0, st) == 0
    torch.cuda.synchronize()
    for i in range(3):   # every image is filtered on its own
        assert np.array_equal(dv[i].cpu().numpy(), _scipy(x[i], fp, "wrap")), i
    inside = torch.zeros_like(dc, dtype=torch.bool)
    inside.as_strided(x.shape, dv.stride(), dv.storage_offset()).fill_(True)
    assert bool((dc[~inside] == fill).all()), "a store landed outside the output"
    # volumes: n = 2
    v = _rand(dtype, (2, 5, 11, 37), 92)
    fp3 = _S().ball(2)
    _, sv, ss = _canvas(v.shape, TORCH[dtype], dev, off, (pads[0], pads[1], pads[1]), fill)
    sv.copy_(_gpu(v, dev))
    dc, dv, ds = _canvas(v.shape, TORCH[dtype], dev, off + 1, (pads[1] + 3, pads[0], pads[1] + 1), fill)
    cv = 9.0
    assert L.mie_sk_median3d(sv.data_ptr(), dv.data_ptr(), CODE[dtype], 2, 5, 11, 37, *ss[:3], *ds[:3], fp3.ctypes.data,
                             5, 5, 5, BORDER["constant"], cv, st) == 0
    torch.cuda.synchronize()
    for i in range(2):
        assert np.array_equal(dv[i].cpu().numpy(), _scipy(v[i], fp3, "constant", cv)), i
    inside = torch.zeros_like(dc, dtype=torch.bool)
    inside.as_strided(v.shape, dv.stride(), dv.storage_offset()).fill_(True)
    assert bool((dc[~inside] == fill).all())


@pytest.mark.gpu
def test_repeatable_bits_and_graph_capture(dev):
    F = _F()
    S = _S()
    x = _gpu(_rand(np.float32, (64, 96), 100), dev)
    v = _gpu(_rand(np.uint16, (12, 40, 50), 101), dev)
    a = F.median(x, S.disk(4), mode="reflect")
    b = F.median(v, S.ball(2), mode="wrap")
    for _ in range(3):
        assert torch.equal(F.median(x, S.disk(4), mode="reflect"), a)
        assert torch.equal(F.median(v, S.ball(2), mode="wrap"), b)
    oa, ob = torch.empty_like(x), torch.empty_like(v)

    def launch():
        F.median(x, S.disk(4), mode="reflect", out=oa)
        F.median(v, S.ball(2), mode="wrap", out=ob)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        launch()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for _ in range(2):
        oa.zero_()
        ob.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(oa, a) and torch.equal(ob, b)


@pytest.mark.gpu
def test_batch_beyond_2_pow_31_elements(dev):
    L = _lib()
    h, w = 512, 500
    n = 2 ** 31 // (h * w) + 12
    straddle = 2 ** 31 // (h * w)
    assert straddle * h * w < 2 ** 31 < (straddle + 1) * h * w
    base = _gpu(_rand(np.uint8, (8, h, w), 110), dev)
    x = base.repeat(n // 8 + 1, 1, 1)[:n].contiguous()
    x[straddle] = torch.flip(x[straddle], (1,))
    out = torch.empty_like(x)
    fp = _S().disk(2)
    assert L.mie_sk_median(x.data_ptr(), out.data_ptr(), U8, n, h, w, h * w, w, h * w, w, fp.ctypes.data, 5, 5,
                           BORDER["reflect"], 0.0, torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    for i in (0, n // 2, straddle, n - 1):
        assert np.array_equal(out[i].cpu().numpy(), _scipy(x[i].cpu().numpy(), fp, "reflect")), i
    assert not torch.equal(out[straddle], out[straddle - 8])


@pytest.mark.gpu
def test_512_cubed_int16_ball2(dev):
    from mie_b200 import synthetic

    F = _F()
    fp = _S().ball(2)
    m = 2   # extent // 2
    vol = synthetic.phantom_volume((512, 512, 512), np.int16, seed=5)
    xt = _gpu(vol, dev)
    for mode in MODES:
        got = F.median(xt, fp, mode=mode, cval=-1000.0).cpu().numpy()
        blocks = [(0, 0, 0), (512 - 24, 512 - 24, 512 - 24), (0, 250, 512 - 24), (200, 300, 100), (256, 128, 384)]
        for z0, y0, x0 in blocks if mode != "wrap" else blocks[3:]:   # wrap reads the opposite face
            lo = [max(0, c - m) for c in (z0, y0, x0)]
            hi = [min(512, c + 24 + m) for c in (z0, y0, x0)]
            crop = vol[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]]
            ref = _scipy(crop, fp, mode, -1000.0)
            sl = tuple(slice(c - l, c - l + 24) for c, l in zip((z0, y0, x0), lo))
            assert np.array_equal(got[z0:z0 + 24, y0:y0 + 24, x0:x0 + 24], ref[sl]), (mode, (z0, y0, x0))


@pytest.mark.gpu
def test_live_pin_against_skimage(dev):
    filters = pytest.importorskip("skimage.filters")
    morphology = pytest.importorskip("skimage.morphology")
    S = _S()
    for r in (1, 2, 3, 5):
        assert np.array_equal(S.disk(r), morphology.disk(r))
    for r in (1, 2, 3):
        assert np.array_equal(S.ball(r), morphology.ball(r))
    x = _rand(np.uint16, (40, 37), 120)
    v = _rand(np.int16, (12, 20, 18), 121)
    for mode in MODES:
        assert np.array_equal(S.median(_gpu(x, dev), S.disk(3), mode=mode, cval=7).cpu().numpy(),
                              filters.median(x, morphology.disk(3), mode=mode, cval=7))
        assert np.array_equal(S.median(_gpu(v, dev), S.ball(2), mode=mode, cval=-7).cpu().numpy(),
                              filters.median(v, morphology.ball(2), mode=mode, cval=-7))
