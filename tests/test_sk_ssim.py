"""skimage.metrics.structural_similarity on planes and whole volumes (skimage_compat.structural_similarity,
mie_sk_structural_similarity / mie_sk_structural_similarity3d).

CPU: scipy.ndimage's line arithmetic as the twin (tests/sk_ssim_twin.py) transcribes it, pinned against the installed
scipy; the twin's exact S == 1 on identical images; the ABI's host validation; the Python argument errors.  GPU: the map
bit for bit and mssim within 1e-12 against the twin (only the mean's summation order differs), repeatable bits, every
window kind and dtype, non-dense layouts, a 512^3 volume, a batch beyond 2^31 elements and graph capture."""
import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter, gaussian_filter1d, uniform_filter, uniform_filter1d

import sk_ssim_twin as T

U8, U16, I16, F32, F64 = 0, 1, 2, 3, 4
E_NULL, E_DTYPE, E_SHAPE, E_STRIDE, E_KERNEL, E_WORKSPACE, E_ALIGN = -1, -2, -3, -4, -7, -9, -12
FAKE = 0x10000   # 256-byte aligned, never dereferenced: every call with it fails validation or has an empty batch
TAPS11 = T.gaussian_weights(1.5)


def _lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def _pair(shape, dtype, seed=0):
    """A phantom-like image and a noisy, blurred copy of it (float32 on [0, 1))."""
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    x = rng.integers(0, 4096, size=shape).astype(np.float64)
    x = uniform_filter(x, 3) + rng.normal(0, 200, size=shape) * (rng.random(shape) < 0.5)
    y = gaussian_filter(x, 1.0) + rng.normal(0, 80, size=shape)
    out = []
    for v in (x, y):
        v = np.clip(v, 0, 4095)
        if dt == np.uint8:
            out.append((v // 16).astype(np.uint8))
        elif dt == np.uint16:
            out.append(v.astype(np.uint16))
        elif dt == np.int16:
            out.append((v - 1024).astype(np.int16))
        else:
            out.append((v / 4096.0).astype(np.float32))
    return out


# ------------------------------------------------------------------------------------------------ twin (CPU)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_line_loops_equal_scipy(dtype):
    rng = np.random.default_rng(1)
    for n in (1, 2, 3, 7, 12, 61):
        x = (rng.standard_normal((4, n)) * 1000).astype(dtype)
        for size in (1, 3, 7, 11, 33):
            got, ref = T.uniform_line(x, size), uniform_filter1d(x, size, axis=-1)
            assert got.dtype == ref.dtype and np.array_equal(got, ref), (n, size)
        for sigma in (0.3, 1.5, 2.2, 4.5):
            got = T.gaussian_line(x, T.gaussian_weights(sigma))
            assert np.array_equal(got, gaussian_filter1d(x, sigma, truncate=3.5, mode="reflect")), (n, sigma)


@pytest.mark.parametrize("shape", [(12, 9), (9, 10, 11), (3, 8, 7)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_axis_order_composition_equals_the_nd_filters(shape, dtype):
    x = (np.random.default_rng(2).standard_normal(shape) * 300).astype(dtype)
    assert np.array_equal(T.filter_axes(x, T.uniform_line, 7), uniform_filter(x, 7))
    assert np.array_equal(T.filter_axes(x, T.uniform_line, 3), uniform_filter(x, 3))
    w = T.gaussian_weights(1.5)
    assert np.array_equal(T.filter_axes(x, T.gaussian_line, w), gaussian_filter(x, 1.5, truncate=3.5, mode="reflect"))


def test_package_taps_are_scipys():
    from mie_b200 import skimage_compat as S

    x = np.random.default_rng(3).standard_normal((3, 40))
    for sigma in (0.5, 1.5, 2.0, 4.6):
        w = S._ssim_taps(sigma, 3.5)
        assert np.array_equal(w, T.gaussian_weights(sigma))
        assert np.array_equal(T.gaussian_line(x, w), gaussian_filter1d(x, sigma, truncate=3.5, mode="reflect"))
    assert np.array_equal(S._ssim_taps(0.0, 3.5), [1.0])


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("gaussian", [False, True])
def test_twin_identical_images_give_one_exactly(dtype, gaussian):
    for shape in [(23, 19), (11, 13, 12)]:
        x, _ = _pair(shape, dtype, 4)
        kw = dict(data_range=1.0) if dtype == np.float32 else {}
        m, s = T.structural_similarity(x, x, gaussian_weights=gaussian, full=True, **kw)
        assert np.all(s == 1) and m == 1.0


# ------------------------------------------------------------------------------------------------ ABI (CPU)
H, W, D = 64, 64, 9
PAD = W + 48


def _call2(n, a=(H * W, W), b=(H * W, W), m=(H * W, W), sd=U16, md=F64, win=7, taps=None, ntaps=0, ap=FAKE, bp=FAKE,
           mp=FAKE, mssim=FAKE, ws=FAKE, nbytes=1 << 40, h=H, w=W):
    return _lib().mie_sk_structural_similarity(ap, bp, mp, sd, md, n, h, w, *a, *b, *m, win, taps, ntaps, 343 / 342,
                                               6.5025, 58.5225, mssim, ws, nbytes, None)


def _call3(n, a=None, b=None, m=None, sd=U16, md=F64, win=7, taps=None, ntaps=0, ap=FAKE, bp=FAKE, mp=FAKE,
           mssim=FAKE, ws=FAKE, nbytes=1 << 40, d=D, h=H, w=W):
    dense = (d * h * w, h * w, w)
    return _lib().mie_sk_structural_similarity3d(ap, bp, mp, sd, md, n, d, h, w, *(a or dense), *(b or dense),
                                                 *(m or dense), win, taps, ntaps, 343 / 342, 6.5025, 58.5225, mssim, ws,
                                                 nbytes, None)


def test_workspace_query_is_bounded_in_batch_and_depth():
    L = _lib()
    for sd in (U8, U16, I16, F32):
        small = L.mie_sk_structural_similarity_workspace_bytes(1, 37, 53, sd)
        assert 0 < small < 1 << 20
        for n in (1, 256, 10 ** 6):
            assert L.mie_sk_structural_similarity_workspace_bytes(n, 512, 512, sd) < 1 << 30
        for n, d in [(1, 512), (1, 10 ** 6), (10 ** 4, 512), (10 ** 6, 7)]:
            assert L.mie_sk_structural_similarity3d_workspace_bytes(n, d, 512, 512, sd) < 1 << 30, (n, d, sd)
    assert L.mie_sk_structural_similarity3d_workspace_bytes(1, 10 ** 6, 512, 512, I16) == \
        L.mie_sk_structural_similarity3d_workspace_bytes(7, 512, 512, 512, I16)
    for bad in [(0, 8, 8, U8), (-1, 8, 8, U8), (1, 0, 8, U8), (1, 8, 0, U8), (1, 8, 8, F64), (1, 8, 8, -1)]:
        assert L.mie_sk_structural_similarity_workspace_bytes(*bad) == 0, bad
    assert L.mie_sk_structural_similarity3d_workspace_bytes(1, 0, 8, 8, U8) == 0


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_dtype_codes(call):
    for sd, md in [(U8, F64), (U16, F64), (I16, F64), (F32, F32)]:
        assert call(1, sd=sd, md=md, nbytes=16) == E_WORKSPACE, (sd, md)
        assert call(1, sd=sd, md=F32 if md == F64 else F64, nbytes=16) == E_DTYPE, sd
        assert call(1, sd=sd, md=sd, mp=None, nbytes=16) == E_WORKSPACE, sd   # no map: its dtype is not read
    for sd in (F64, 5, -1):
        assert call(1, sd=sd, nbytes=16) == E_DTYPE, sd


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_window_and_shape_codes(call):
    for win in (0, -1, 2, 8, 35, 34):
        assert call(1, win=win) == E_KERNEL, win
    t = TAPS11.ctypes.data
    for ntaps in (0, -1, 2, 12, 35):
        assert call(1, taps=t, ntaps=ntaps) == E_KERNEL, ntaps
    assert call(1, taps=t, ntaps=11, win=3, nbytes=16) == E_WORKSPACE   # taps wider than the window: legal
    assert call(1, win=33, nbytes=16, **({} if call is _call2 else dict(d=33))) == E_WORKSPACE
    kw = dict(h=9, w=W) if call is _call2 else dict(d=9, h=H, w=W)
    assert call(1, win=9, nbytes=16, **kw) == E_WORKSPACE               # an axis exactly win_size long
    assert call(1, win=11, **kw) == E_SHAPE
    if call is _call3:
        assert call(1, win=11, d=10, h=H, w=W) == E_SHAPE
        assert call(1, win=7, d=1, h=H, w=W) == E_SHAPE                  # a (1, h, w) volume is not a plane
    assert call(1, win=11, h=H, w=10) == E_SHAPE


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_null_pointers_and_workspace(call):
    assert call(1, ap=None) == E_NULL
    assert call(1, bp=None) == E_NULL
    assert call(1, mssim=None) == E_NULL
    assert call(1, ws=None) == E_NULL
    assert call(1, ws=FAKE + 8) == E_ALIGN
    assert call(1, mp=None, ws=FAKE + 8) == E_ALIGN   # a NULL map is legal
    L = _lib()
    need = (L.mie_sk_structural_similarity_workspace_bytes(2, H, W, U16) if call is _call2 else
            L.mie_sk_structural_similarity3d_workspace_bytes(2, D, H, W, U16))
    assert call(2, nbytes=need - 1) == E_WORKSPACE
    assert call(0, ap=None, bp=None, mp=None, mssim=None, ws=None, nbytes=0) == 0   # empty batch: no pointers needed


def _tight(ssh):
    return (H - 1) * ssh + W


def test_plane_strides_too_small_are_refused():
    ok = (_tight(PAD), PAD)
    bad = [("row stride w - 1", 1, (H * (W - 1), W - 1)), ("plane stride one short of the last row", 2, (_tight(PAD) - 1, PAD)),
           ("plane stride one short, dense rows", 2, (_tight(W) - 1, W))]
    for what, n, s in bad:
        assert _call2(n, a=s, b=ok, m=ok) == E_STRIDE, "a " + what
        assert _call2(n, a=ok, b=s, m=ok) == E_STRIDE, "b " + what
        assert _call2(n, a=ok, b=ok, m=s) == E_STRIDE, "map " + what
        assert _call2(n, a=ok, b=ok, m=s, mp=None, nbytes=16) == E_WORKSPACE, "no map " + what
    assert _call2(0, a=((H + 3) * PAD, PAD), b=(_tight(W + 1) + 3, W + 1), m=ok) == 0


def _vol(ssh, ssd=None, ssn=None):
    ssd = (H - 1) * ssh + W if ssd is None else ssd
    ssn = (D - 1) * ssd + (H - 1) * ssh + W if ssn is None else ssn
    return ssn, ssd, ssh


def test_volume_strides_too_small_are_refused():
    ok = _vol(PAD)
    tight_d = (H - 1) * PAD + W
    bad = [("row stride w - 1", 1, _vol(W - 1)),
           ("slice stride one short of the last row", 1, _vol(PAD, ssd=tight_d - 1, ssn=D * tight_d)),
           ("volume stride one short", 2, _vol(PAD, ssn=(D - 1) * tight_d + (H - 1) * PAD + W - 1))]
    for what, n, s in bad:
        assert _call3(n, a=s, b=ok, m=ok) == E_STRIDE, "a " + what
        assert _call3(n, a=ok, b=s, m=ok) == E_STRIDE, "b " + what
        assert _call3(n, a=ok, b=ok, m=s) == E_STRIDE, "map " + what


# ------------------------------------------------------------------------------------------------ Python (CPU)
def test_python_argument_errors():
    from mie_b200 import skimage_compat as S

    x = torch.zeros(16, 16, dtype=torch.uint16)
    f = torch.zeros(16, 16, dtype=torch.float32)
    with pytest.raises(ValueError, match="same dimensions"):
        S.structural_similarity(x, torch.zeros(16, 15, dtype=torch.uint16))
    with pytest.raises(ValueError, match="data_range"):
        S.structural_similarity(f, f)
    with pytest.raises(ValueError, match="odd"):
        S.structural_similarity(x, x, win_size=6)
    with pytest.raises(ValueError, match="exceeds"):
        S.structural_similarity(x, x, win_size=17)
    v = torch.zeros(5, 16, 16, dtype=torch.uint16)
    with pytest.raises(ValueError, match="exceeds"):   # 7x7x7 windows on a 5-slice volume
        S.structural_similarity(v, v, volumetric=True)
    with pytest.raises(ValueError, match="volumetric=True"):
        S.structural_similarity(x, x, volumetric=True)
    for k in ("K1", "K2", "sigma"):
        with pytest.raises(ValueError, match=k):
            S.structural_similarity(x, x, **{k: -0.1})
    with pytest.raises(NotImplementedError):
        S.structural_similarity(x, x, gradient=True)
    with pytest.raises(NotImplementedError):
        S.structural_similarity(x, x, channel_axis=0)
    with pytest.raises(NotImplementedError):
        S.structural_similarity(x, x.to(torch.int16))
    with pytest.raises(NotImplementedError):
        S.structural_similarity(torch.zeros(40, 40, dtype=torch.uint8), torch.zeros(40, 40, dtype=torch.uint8), win_size=35)
    with pytest.raises(NotImplementedError):   # sigma 5 needs 2 * int(17.5 + 0.5) + 1 = 37 taps
        S.structural_similarity(torch.zeros(40, 40, dtype=torch.uint8), torch.zeros(40, 40, dtype=torch.uint8),
                                gaussian_weights=True, sigma=5.0, win_size=11)
    with pytest.raises(ZeroDivisionError):
        S.structural_similarity(x, x, win_size=1)
    with pytest.raises(TypeError):
        S.structural_similarity(x, x, K3=0.1)
    with pytest.raises(TypeError):
        S.structural_similarity(np.zeros((16, 16), np.uint16), x)
    with pytest.raises(TypeError):
        S.structural_similarity(x.double(), x.double(), data_range=1.0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        S.structural_similarity(x, x)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        S.structural_similarity(x, x, win_size=1, use_sample_covariance=False)
    assert "structural_similarity" in S.__all__


# ------------------------------------------------------------------------------------------------ GPU
def _gpu(x, y, dev, volumetric=False, **kw):
    """-> (mssim as a float64 array of the leading shape, S as numpy) through the public path."""
    from mie_b200 import skimage_compat as S

    xt = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    yt = torch.from_numpy(np.ascontiguousarray(y)).to(dev)
    m, s = S.structural_similarity(xt, yt, full=True, volumetric=volumetric, **kw)
    m2 = S.structural_similarity(xt, yt, full=False, volumetric=volumetric, **kw)
    m = np.asarray(m.numpy() if isinstance(m, torch.Tensor) else m)
    m2 = np.asarray(m2.numpy() if isinstance(m2, torch.Tensor) else m2)
    assert np.array_equal(m, m2), "full=False gave another mssim"
    return m, s.cpu().numpy()


def _check(x, y, dev, volumetric=False, **kw):
    """Every image of the batch (the last 2 / 3 axes) against the twin: map bit for bit, mssim within 1e-12."""
    if x.dtype == np.float32:
        kw.setdefault("data_range", 1.0)
    m, s = _gpu(x, y, dev, volumetric, **kw)
    per = 3 if volumetric else 2
    lead = x.shape[:-per]
    xs, ys = x.reshape((-1,) + x.shape[-per:]), y.reshape((-1,) + x.shape[-per:])
    ms, ss = m.reshape(-1), s.reshape(xs.shape)
    assert s.dtype == (np.float32 if x.dtype == np.float32 else np.float64) and s.shape == x.shape
    assert m.shape == lead
    for i in range(xs.shape[0]):
        ref_m, ref_s = T.structural_similarity(xs[i], ys[i], full=True, **kw)
        assert np.array_equal(ss[i], ref_s), f"image {i}: {int((ss[i] != ref_s).sum())} differing of {ref_s.size}; " \
                                             f"max |diff| {np.abs(ss[i].astype(np.float64) - ref_s).max():.3e}"
        assert abs(ms[i] - ref_m) <= 1e-12, (i, ms[i], ref_m)
    return m, s


WINDOWS = [dict(win_size=3), dict(), dict(win_size=11), dict(win_size=33), dict(gaussian_weights=True),
           dict(gaussian_weights=True, sigma=0.8), dict(gaussian_weights=True, win_size=3)]
WIN_IDS = ["box3", "box7", "box11", "box33", "gauss1.5", "gauss0.8", "gauss1.5-win3"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("win", WINDOWS, ids=WIN_IDS)
def test_planes_match_the_twin(dev, dtype, win):
    side = max(win.get("win_size", 7), 11)
    for shape in [(side, side + 4), (2, 3, 37, 45), (61, 34)]:
        x, y = _pair(shape, dtype, 5)
        _check(x, y, dev, **win)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("win", WINDOWS, ids=WIN_IDS)
def test_volumes_match_the_twin(dev, dtype, win):
    k = win.get("win_size", 11 if win.get("gaussian_weights") and "sigma" not in win else 7)
    shapes = [(k, k, k + 2), (2, k + 2, k + 5, k + 3)] if k >= 11 else [(k, k, k), (2, 1, 13, 17, 15), (9, 31, 20)]
    for shape in shapes:
        x, y = _pair(shape, dtype, 6)
        _check(x, y, dev, volumetric=True, **win)


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True])
def test_arguments_match_the_twin(dev, volumetric):
    shape = (2, 11, 24, 19) if volumetric else (3, 40, 33)
    for dtype in (np.uint16, np.float32):
        x, y = _pair(shape, dtype, 7)
        for kw in [dict(use_sample_covariance=False), dict(K1=0.05, K2=0.1), dict(data_range=4095),
                   dict(gaussian_weights=True, use_sample_covariance=False, K1=0.0),
                   dict(win_size=1, use_sample_covariance=False)]:
            if dtype == np.float32 and "data_range" in kw:
                kw = dict(data_range=0.5)
            _check(x, y, dev, volumetric, **kw)


@pytest.mark.gpu
def test_identical_images_score_one_and_runs_repeat(dev):
    from mie_b200 import skimage_compat as S

    for dtype in (torch.uint8, torch.uint16, torch.int16):
        x = torch.from_numpy(_pair((20, 24, 28), np.dtype(str(dtype).split(".")[1]), 8)[0]).to(dev)
        for kw in (dict(), dict(gaussian_weights=True)):
            assert S.structural_similarity(x, x, volumetric=True, **kw) == 1.0
            m, s = S.structural_similarity(x, x, volumetric=True, full=True, **kw)
            assert m == 1.0 and bool((s == 1).all())
    x, y = (torch.from_numpy(v).to(dev) for v in _pair((3, 30, 40, 50), np.int16, 9))
    a = S.structural_similarity(x, y, volumetric=True, full=True)
    b = S.structural_similarity(x, y, volumetric=True, full=True)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def _canvas(t, dev, off, pad_row, pad_slice, volumetric, fill=0):
    """`t` placed at element offset `off` of a canvas with rows padded by pad_row and slices / planes by pad_slice;
    -> (canvas, view, (strides of the ABI))."""
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
@pytest.mark.parametrize("volumetric", [False, True])
@pytest.mark.parametrize("layout", [(0, 0, 0, 0, 0), (0, 16, 0, 8, 0), (0, 8, 40, 0, 24), (1, 3, 7, 3, 5)],
                         ids=["dense", "padded-rows", "padded-slices", "unaligned"])
def test_non_dense_layouts_equal_the_dense_call(dev, volumetric, layout):
    from mie_b200 import skimage_compat as S

    off, pad_row, pad_slice, boff, moff = layout
    x, y = (torch.from_numpy(v).to(dev) for v in _pair((2, 9, 37, 45) if volumetric else (2, 37, 45), np.int16, 10))
    dense_m, dense_s = S.structural_similarity(x, y, full=True, volumetric=volumetric)
    _, av, astr = _canvas(x, dev, off, pad_row, pad_slice, volumetric)
    _, bv, bstr = _canvas(y, dev, boff, pad_row + 5, pad_slice, volumetric)
    mc, mv, mstr = _canvas(torch.zeros(x.shape, dtype=torch.float64, device=dev), dev, moff, pad_row + 1, pad_slice + 2,
                           volumetric, float("nan"))
    mv.fill_(float("nan"))
    L = _lib()
    n = x.shape[0]
    mssim = torch.empty(n, dtype=torch.float64, device=dev)
    if volumetric:
        ws = torch.empty(L.mie_sk_structural_similarity3d_workspace_bytes(n, *x.shape[1:], I16), dtype=torch.uint8,
                         device=dev)
        rc = L.mie_sk_structural_similarity3d(av.data_ptr(), bv.data_ptr(), mv.data_ptr(), I16, F64, n, *x.shape[1:],
                                              *astr, *bstr, *mstr, 7, None, 0, 343 / 342, (0.01 * 65535) ** 2,
                                              (0.03 * 65535) ** 2, mssim.data_ptr(), ws.data_ptr(), ws.numel(),
                                              torch.cuda.current_stream().cuda_stream)
    else:
        ws = torch.empty(L.mie_sk_structural_similarity_workspace_bytes(n, *x.shape[1:], I16), dtype=torch.uint8,
                         device=dev)
        rc = L.mie_sk_structural_similarity(av.data_ptr(), bv.data_ptr(), mv.data_ptr(), I16, F64, n, *x.shape[1:],
                                            *astr, *bstr, *mstr, 7, None, 0, 49 / 48, (0.01 * 65535) ** 2,
                                            (0.03 * 65535) ** 2, mssim.data_ptr(), ws.data_ptr(), ws.numel(),
                                            torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(mv, dense_s)
    assert torch.equal(mssim.cpu(), dense_m)
    outside = torch.ones_like(mc, dtype=torch.bool)
    outside.as_strided(x.shape, mv.stride(), moff).fill_(False)
    assert bool(torch.isnan(mc[outside]).all()), "a store landed outside the map"


@pytest.mark.gpu
def test_512_cubed_volume_against_its_gaussian(dev):
    from mie_b200 import skimage_compat as S, synthetic

    x = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, 0)).to(dev)
    y = S.gaussian(x, 1.0, volumetric=True)
    m, s = S.structural_similarity(x, y, volumetric=True, full=True)
    assert S.structural_similarity(x, y, volumetric=True) == m
    xn, yn = x.cpu().numpy(), y.cpu().numpy()
    del x, y
    ref_m, ref_s = T.structural_similarity(xn, yn, full=True)
    assert abs(m - ref_m) <= 1e-12, (m, ref_m)
    assert 0.0 < m < 1.0
    assert np.array_equal(s.cpu().numpy(), ref_s)


@pytest.mark.gpu
def test_batch_beyond_2_pow_31_elements(dev):
    from mie_b200 import skimage_compat as S

    h, w = 512, 500
    n = 2 ** 31 // (h * w) + 12          # 8400 planes, 2.15e9 elements
    straddle = 2 ** 31 // (h * w)       # plane 8388 holds element 2^31
    assert straddle * h * w < 2 ** 31 < (straddle + 1) * h * w and n * h * w > 2 ** 31
    bx, by = (torch.from_numpy(v).to(dev) for v in _pair((8, h, w), np.uint8, 11))
    x = bx.repeat(n // 8 + 1, 1, 1)[:n].contiguous()
    y = by.repeat(n // 8 + 1, 1, 1)[:n].contiguous()
    y[straddle] = torch.flip(y[straddle], (1,))
    m = S.structural_similarity(x, y)
    assert m.shape == (n,) and m.dtype == torch.float64
    for i in (0, straddle, n - 1):
        assert m[i].item() == S.structural_similarity(x[i].clone(), y[i].clone()), i
        ref = T.structural_similarity(x[i].cpu().numpy(), y[i].cpu().numpy())
        assert abs(m[i].item() - ref) <= 1e-12, i
    assert m[straddle].item() != m[straddle - 8].item()


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True])
def test_graph_capture_equals_the_eager_call(dev, volumetric):
    from mie_b200 import skimage_compat as S

    x, y = (torch.from_numpy(v).to(dev) for v in _pair((2, 12, 40, 36) if volumetric else (3, 64, 72), np.uint16, 12))
    eager_m, eager_s = S.structural_similarity(x, y, volumetric=volumetric, full=True, gaussian_weights=True)
    L = _lib()
    n, dims = x.shape[0], tuple(x.shape[1:])
    taps = T.gaussian_weights(1.5)
    nd = len(dims)
    npts = 11 ** nd
    if volumetric:
        need = L.mie_sk_structural_similarity3d_workspace_bytes(n, *dims, U16)
        d, h, w = dims
        layout = (n, d, h, w) + (d * h * w, h * w, w) * 3
        fn = L.mie_sk_structural_similarity3d
    else:
        need = L.mie_sk_structural_similarity_workspace_bytes(n, *dims, U16)
        h, w = dims
        layout = (n, h, w) + (h * w, w) * 3
        fn = L.mie_sk_structural_similarity
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    mssim = torch.empty(n, dtype=torch.float64, device=dev)
    smap = torch.empty(x.shape, dtype=torch.float64, device=dev)

    def launch():
        rc = fn(x.data_ptr(), y.data_ptr(), smap.data_ptr(), U16, F64, *layout, 11, taps.ctypes.data, taps.size,
                npts / (npts - 1), (0.01 * 65535) ** 2, (0.03 * 65535) ** 2, mssim.data_ptr(), ws.data_ptr(), ws.numel(),
                torch.cuda.current_stream().cuda_stream)
        assert rc == 0

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        launch()   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    for _ in range(2):
        mssim.zero_()
        smap.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(mssim.cpu(), eager_m) and torch.equal(smap, eager_s)


@pytest.mark.gpu
def test_live_pin_against_skimage(dev):
    metrics = pytest.importorskip("skimage.metrics")
    for (x, y), volumetric, kw in [(_pair((40, 33), np.uint16, 13), False, {}),
                                   (_pair((11, 24, 19), np.int16, 14), True, {}),
                                   (_pair((11, 24, 19), np.float32, 15), True, dict(data_range=1.0, gaussian_weights=True))]:
        up_m, up_s = metrics.structural_similarity(x, y, full=True, **kw)
        tw_m, tw_s = T.structural_similarity(x, y, full=True, **kw)
        got_m, got_s = _gpu(x, y, dev, volumetric, **kw)
        assert np.array_equal(tw_s, up_s) and tw_m == up_m
        assert np.array_equal(got_s, up_s) and abs(float(got_m) - up_m) <= 1e-12
