"""skimage.restoration.denoise_tv_chambolle on planes and whole volumes (skimage_compat.denoise_tv_chambolle,
mie_sk_denoise_tv_chambolle / mie_sk_denoise_tv_chambolle3d).

CPU: properties of the numpy twin (tests/sk_tv_chambolle_twin.py), the ABI's host-side validation and the Python
argument errors.  GPU: the CUDA path against the twin bit for bit with equal iteration counts — every case first
asserts that the twin's closest stopping test is far from a tie, since only the energy sums' order differs — plus
per-image stopping in a batch, non-dense layouts, a 512^3 volume, a batch beyond 2^31 elements and graph capture."""
import ctypes as C

import numpy as np
import pytest
import torch

import sk_tv_chambolle_twin as T

U8, U16, I16, F32, F64 = 0, 1, 2, 3, 4
E_NULL, E_DTYPE, E_SHAPE, E_STRIDE, E_WORKSPACE, E_RANGE, E_ALIGN = -1, -2, -3, -4, -9, -10, -12
FAKE = 0x10000   # 256-byte aligned, never dereferenced: every call with it fails validation or has an empty batch
NP = {U8: np.uint8, U16: np.uint16, I16: np.int16, F32: np.float32}
MARGIN = 1e-4


def _lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def _img(shape, dtype, seed=0):
    """Phantom planes / volumes where both sides are large enough, seeded noise otherwise; float32 on [0, 1)."""
    from mie_b200 import synthetic

    dt = np.dtype(dtype)
    h, w = shape[-2:]
    if h >= 16 and w >= 16:
        if len(shape) == 3 and shape[0] > 1:
            x = synthetic.phantom_volume(shape, np.int16 if dt == np.int16 else np.uint16, seed)
        else:
            x = synthetic.phantom(shape, np.int16 if dt == np.int16 else np.uint16, seed)
        x = x.astype(np.int64)
    else:
        x = np.random.default_rng(seed).integers(0, 4096, size=shape)
        x = x - 1024 if dt == np.int16 else x
    if dt == np.uint8:
        return (np.clip(x, 0, 4095) // 16).astype(np.uint8)
    if dt == np.float32:
        return (x.astype(np.float32) + 1024.0) / 8192.0
    return x.astype(dt)


def _twin(x, **kw):
    out, iters, margin = T.denoise_tv_chambolle(x, **kw)
    assert margin > MARGIN, f"case within {margin:.2e} of a stopping tie: pick another"
    return out, iters


# ------------------------------------------------------------------------------------------------ twin (CPU)
def test_twin_constant_image_runs_every_pass_and_comes_back_unchanged():
    x = np.full((12, 9), 77, np.uint8)
    out, iters, margin = T.denoise_tv_chambolle(x, max_num_iter=37)
    assert iters == 37 and margin == np.inf
    assert np.array_equal(out, T.img_as_float(x))
    v = np.full((3, 5, 4), 0.25, np.float32)
    out, iters, _ = T.denoise_tv_chambolle(v)
    assert iters == 200 and out.dtype == np.float32 and np.array_equal(out, v)


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
def test_twin_one_pass_returns_the_float_image(dtype):
    x = _img((21, 17), dtype, 3)
    out, iters, _ = T.denoise_tv_chambolle(x, max_num_iter=1)
    assert iters == 1 and np.array_equal(out, T.img_as_float(x))
    assert out.dtype == (np.float32 if dtype == np.float32 else np.float64)


@pytest.mark.parametrize("shape", [(40, 33), (7, 19, 23)])
def test_twin_preserves_the_mean(shape):
    # sum(div p) = 0 under upstream's boundary rules: p_a is 0 on the last index of axis a
    x = _img(shape, np.uint16, 4)
    out, iters, _ = T.denoise_tv_chambolle(x, weight=0.2)
    assert iters > 2
    assert abs(out.mean() - T.img_as_float(x).mean()) <= 1e-12


def test_twin_is_deterministic_and_smooths():
    x = _img((64, 64), np.uint16, 5)
    a, ia, _ = T.denoise_tv_chambolle(x)
    b, ib, _ = T.denoise_tv_chambolle(x)
    assert ia == ib and np.array_equal(a, b)
    f = T.img_as_float(x)
    assert np.abs(np.diff(a, axis=1)).sum() < np.abs(np.diff(f, axis=1)).sum()


# ------------------------------------------------------------------------------------------------ ABI (CPU)
H, W, D = 64, 64, 5
PAD = W + 48


def _call2(n, s=(H * W, W), d=(H * W, W), sd=U16, dd=F64, weight=0.1, max_iter=200, src=FAKE, dst=FAKE, ws=FAKE,
           nbytes=1 << 40, h=H, w=W):
    return _lib().mie_sk_denoise_tv_chambolle(src, dst, sd, dd, n, h, w, *s, *d, weight, 2e-4, max_iter, None, ws, nbytes,
                                              None)


def _call3(n, s=None, d=None, sd=U16, dd=F64, weight=0.1, max_iter=200, src=FAKE, dst=FAKE, ws=FAKE, nbytes=1 << 40):
    dense = (D * H * W, H * W, W)
    return _lib().mie_sk_denoise_tv_chambolle3d(src, dst, sd, dd, n, D, H, W, *(s or dense), *(d or dense), weight, 2e-4,
                                                max_iter, None, ws, nbytes, None)


def test_workspace_query():
    L = _lib()
    for n, h, w in [(1, 1, 1), (3, 37, 53), (2, 512, 512)]:
        for sd, fsz in [(U8, 8), (U16, 8), (I16, 8), (F32, 4)]:
            got = L.mie_sk_tv_chambolle_workspace_bytes(n, h, w, sd)
            base = 2 * 2 * n * h * w * fsz   # two float copies of p (2 components)
            assert base < got <= base + 512 + n * (32 + 16 * h * w), (n, h, w, sd)
    for n, d, h, w in [(1, 1, 1, 1), (2, 33, 47, 61)]:
        for sd, fsz in [(I16, 8), (F32, 4)]:
            got = L.mie_sk_tv_chambolle3d_workspace_bytes(n, d, h, w, sd)
            base = 2 * 3 * n * d * h * w * fsz
            assert base < got <= base + 512 + n * (32 + 16 * d * h * w), (n, d, h, w, sd)
    # one (1, h, w) volume holds three components, one plane two
    assert L.mie_sk_tv_chambolle3d_workspace_bytes(1, 1, 64, 64, U8) > L.mie_sk_tv_chambolle_workspace_bytes(1, 64, 64, U8)
    for bad in [(0, 8, 8, U8), (-1, 8, 8, U8), (1, 0, 8, U8), (1, 8, 0, U8), (1, 8, 8, F64), (1, 8, 8, -1)]:
        assert L.mie_sk_tv_chambolle_workspace_bytes(*bad) == 0, bad
    assert L.mie_sk_tv_chambolle3d_workspace_bytes(1, 0, 8, 8, U8) == 0


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_dtype_combinations(call):
    for sd in (U8, U16, I16, F32):
        for dd in (F32, F64):   # valid: validation goes on to the workspace size
            assert call(1, sd=sd, dd=dd, nbytes=16) == E_WORKSPACE, (sd, dd)
        for dd in (U8, U16, I16, 5, -1):
            assert call(1, sd=sd, dd=dd, nbytes=16) == E_DTYPE, (sd, dd)
    for sd in (F64, 5, -1):
        assert call(1, sd=sd, dd=F64, nbytes=16) == E_DTYPE, sd


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_weight_and_iteration_codes(call):
    for weight in (0.0, -0.1, float("nan"), float("inf"), -float("inf")):
        assert call(1, weight=weight) == E_RANGE, weight
    for it in (0, -1, -200):
        assert call(1, max_iter=it) == E_SHAPE, it
    assert call(1, weight=1e-300, max_iter=1, nbytes=16) == E_WORKSPACE   # tiny but positive weight is legal


@pytest.mark.parametrize("call", [_call2, _call3], ids=["planes", "volumes"])
def test_null_pointers_and_workspace(call):
    assert call(1, src=None) == E_NULL
    assert call(1, dst=None) == E_NULL
    assert call(1, ws=None) == E_NULL
    assert call(1, ws=FAKE + 8) == E_ALIGN
    L = _lib()
    need = (L.mie_sk_tv_chambolle_workspace_bytes(2, H, W, U16) if call is _call2 else
            L.mie_sk_tv_chambolle3d_workspace_bytes(2, D, H, W, U16))
    s2 = (H * W, W) if call is _call2 else None
    assert call(2, s=s2, d=s2, nbytes=need - 1) == E_WORKSPACE
    # an empty batch needs no pointer and no workspace
    assert call(0, src=None, dst=None, ws=None, nbytes=0) == 0


def _tight(ssh):
    return (H - 1) * ssh + W


def test_plane_strides_too_small_are_refused():
    ok = (_tight(PAD), PAD)
    bad = [
        ("row stride w - 1", 1, (H * (W - 1), W - 1), ok),
        ("plane stride one short of the last row", 2, (_tight(PAD) - 1, PAD), ok),
        ("plane stride one short, dense rows", 2, (_tight(W) - 1, W), ok),
    ]
    bad += [(f"destination {what}", n, d, s) for what, n, s, d in bad]
    for what, n, s, d in bad:
        assert _call2(n, s, d) == E_STRIDE, what
    assert _call2(0, ((H + 3) * PAD, PAD), (_tight(PAD), PAD)) == 0
    assert _call2(0, (_tight(W + 1) + 3, W + 1), ((H + 3) * PAD, PAD)) == 0


def _vol(ssh, ssd=None, ssn=None):
    ssd = (H - 1) * ssh + W if ssd is None else ssd
    ssn = (D - 1) * ssd + (H - 1) * ssh + W if ssn is None else ssn
    return ssn, ssd, ssh


def test_volume_strides_too_small_are_refused():
    ok = _vol(PAD)
    tight_d = (H - 1) * PAD + W
    bad = [
        ("row stride w - 1", 1, _vol(W - 1), ok),
        ("slice stride one short of the last row", 1, _vol(PAD, ssd=tight_d - 1, ssn=D * tight_d), ok),
        ("volume stride one short of the last slice's last row", 2,
         _vol(PAD, ssn=(D - 1) * tight_d + (H - 1) * PAD + W - 1), ok),
        ("volume stride ignoring the padded slices", 2, _vol(PAD, ssd=(H + 3) * PAD, ssn=D * H * W), ok),
    ]
    bad += [(f"destination {what}", n, d, s) for what, n, s, d in bad]
    for what, n, s, d in bad:
        assert _call3(n, s, d) == E_STRIDE, what
    padded = _vol(PAD, ssd=(H + 3) * PAD, ssn=(D + 1) * (H + 3) * PAD)
    assert _call3(0, padded, _vol(W + 1, ssd=H * (W + 1) + 3, ssn=D * (H * (W + 1) + 3) + 5)) == 0


# ------------------------------------------------------------------------------------------------ Python (CPU)
def test_python_argument_errors():
    from mie_b200 import skimage_compat as S

    x = torch.zeros(8, 8, dtype=torch.uint16)
    with pytest.raises(NotImplementedError):
        S.denoise_tv_chambolle(x, channel_axis=0)
    for weight in (0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            S.denoise_tv_chambolle(x, weight=weight)
    with pytest.raises(ValueError):
        S.denoise_tv_chambolle(x, max_num_iter=0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        S.denoise_tv_chambolle(x)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        S.denoise_tv_chambolle(torch.zeros(2, 8, 8, dtype=torch.int16), volumetric=True)
    with pytest.raises(ValueError):
        S.denoise_tv_chambolle(x, volumetric=True)   # a volume needs (D, H, W)
    with pytest.raises(TypeError):
        S.denoise_tv_chambolle(np.zeros((8, 8), np.uint16))
    assert "denoise_tv_chambolle" in S.__all__


# ------------------------------------------------------------------------------------------------ GPU
def _gpu(x, dev, volumetric=False, out_dtype=None, **kw):
    """-> (output as numpy, passes run per image) through the public path."""
    from mie_b200 import skimage_compat as S

    xt = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    per = 3 if volumetric else 2
    n = int(np.prod(x.shape[:-per], dtype=np.int64)) if x.ndim > per else 1
    iters = torch.zeros(n, dtype=torch.int32, device=dev)
    out = S._denoise_tv_chambolle(xt, kw.get("weight", 0.1), kw.get("eps", 2e-4), kw.get("max_num_iter", 200), None,
                                  out_dtype, volumetric, iters)
    torch.cuda.synchronize()
    return out.cpu().numpy(), iters.cpu().numpy()


def _same(got, ref):
    assert got.dtype == ref.dtype and got.shape == ref.shape
    assert np.array_equal(got, ref), f"{int((got != ref).sum())} differing of {got.size}; max |diff| " \
                                     f"{np.abs(got.astype(np.float64) - ref).max():.3e}"


PLANE_SHAPES = [(1, 1), (1, 37), (29, 1), (37, 53), (512, 512)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("shape", PLANE_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_planes_match_the_twin(dev, dtype, shape):
    x = _img(shape, dtype, 7)
    ref, it = _twin(x)
    got, its = _gpu(x, dev)
    _same(got, ref)
    assert its.tolist() == [it]


VOLUMES = [((1, 37, 53), np.uint16), ((2, 31, 40), np.uint8), ((33, 47, 61), np.int16), ((33, 47, 61), np.float32),
           ((64, 128, 128), np.int16)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,dtype", VOLUMES, ids=lambda v: str(v))
def test_volumes_match_the_twin(dev, shape, dtype):
    x = _img(shape, dtype, 8)
    ref, it = _twin(x)
    got, its = _gpu(x, dev, volumetric=True)
    _same(got, ref)
    assert its.tolist() == [it]
    if shape[0] == 1:   # tau = 1/6 and a third component: not the 2-D result
        flat, _ = _gpu(x[0], dev)
        assert not np.array_equal(got[0], flat)


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True])
def test_arguments_match_the_twin(dev, volumetric):
    shape = (9, 40, 44) if volumetric else (96, 80)
    for dtype in (np.uint16, np.float32):
        x = _img(shape, dtype, 9)
        for kw in [dict(weight=0.05), dict(weight=0.3), dict(eps=0.0, max_num_iter=7), dict(max_num_iter=1),
                   dict(weight=0.02, eps=1e-3, max_num_iter=30)]:
            ref, it = _twin(x, **kw)
            got, its = _gpu(x, dev, volumetric, **kw)
            _same(got, ref)
            assert its.tolist() == [it], kw
        if dtype == np.uint16:
            got32, _ = _gpu(x, dev, volumetric, out_dtype=torch.float32)
            _same(got32, _twin(x)[0].astype(np.float32))


@pytest.mark.gpu
def test_images_of_a_batch_stop_independently(dev):
    planes = np.stack([np.full((128, 96), 1500, np.uint16), _img((128, 96), np.uint16, 10), _img((128, 96), np.uint16, 11)])
    refs = [_twin(p) for p in planes]
    assert refs[0][1] == 200 and refs[1][1] < 100 and refs[2][1] < 100
    got, its = _gpu(planes.reshape(3, 1, 128, 96), dev)
    for i, (ref, it) in enumerate(refs):
        _same(got[i, 0], ref)
        assert its[i] == it
    vols = np.stack([np.full((6, 40, 36), -200, np.int16), _img((6, 40, 36), np.int16, 12)])
    got, its = _gpu(vols, dev, volumetric=True)
    for i in range(2):
        ref, it = _twin(vols[i])
        _same(got[i], ref)
        assert its[i] == it


def _canvas_call(x, dev, volumetric, off, pad_row, pad_slice, dst_off):
    """Run the ABI on `x` (n, [d,] h, w) placed at element offset `off` of a canvas with rows padded by `pad_row` and
    slices / planes by `pad_slice`; the float64 destination likewise at `dst_off`.  Returns the destination region."""
    from mie_b200 import _ffi

    L = _lib()
    xt = torch.from_numpy(x).to(dev)
    shape = x.shape
    h, w = shape[-2:]
    d = shape[1] if volumetric else 1
    sh = w + pad_row
    sd = h * sh + pad_slice
    sn = d * sd + pad_slice if volumetric else sd

    def place(dtype, o, fill):
        size = o + shape[0] * sn + 64
        canvas = torch.full((size,), fill, dtype=dtype, device=dev)
        strides = (sn, sd, sh, 1) if volumetric else (sn, sh, 1)
        return canvas, canvas.as_strided(shape, strides, o)

    src_c, src_v = place(xt.dtype, off, 0)
    src_v.copy_(xt)
    dst_c, dst_v = place(torch.float64, dst_off, float("nan"))
    n = shape[0]
    code = _ffi.DTYPE_CODE[xt.dtype]
    if volumetric:
        ws = torch.empty(L.mie_sk_tv_chambolle3d_workspace_bytes(n, d, h, w, code), dtype=torch.uint8, device=dev)
        rc = L.mie_sk_denoise_tv_chambolle3d(src_v.data_ptr(), dst_v.data_ptr(), code, F64, n, d, h, w, sn, sd, sh, sn, sd,
                                             sh, 0.1, 2e-4, 200, None, ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream)
    else:
        ws = torch.empty(L.mie_sk_tv_chambolle_workspace_bytes(n, h, w, code), dtype=torch.uint8, device=dev)
        rc = L.mie_sk_denoise_tv_chambolle(src_v.data_ptr(), dst_v.data_ptr(), code, F64, n, h, w, sn, sh, sn, sh, 0.1,
                                           2e-4, 200, None, ws.data_ptr(), ws.numel(),
                                           torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    outside = torch.ones_like(dst_c, dtype=torch.bool)
    outside.as_strided(shape, dst_v.stride(), dst_off).fill_(False)
    assert bool(torch.isnan(dst_c[outside]).all()), "a store landed outside the destination region"
    return dst_v.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True])
@pytest.mark.parametrize("layout", [(0, 0, 0, 0), (0, 16, 0, 0), (0, 8, 40, 0), (1, 3, 7, 3)],
                         ids=["dense", "padded-rows", "padded-slices", "unaligned"])
def test_non_dense_layouts_equal_the_dense_call(dev, volumetric, layout):
    off, pad_row, pad_slice, dst_off = layout
    x = np.stack([_img((5, 37, 45) if volumetric else (37, 45), np.int16, s) for s in (13, 14)])
    dense, _ = _gpu(x, dev, volumetric)
    got = _canvas_call(x, dev, volumetric, off, pad_row, pad_slice, dst_off)
    _same(got, dense)


@pytest.mark.gpu
def test_512_cubed_volume(dev):
    from mie_b200 import skimage_compat as S

    x = _img((512, 512, 512), np.int16, 0)
    ref, it = _twin(x, eps=0.0, max_num_iter=3)
    got, its = _gpu(x, dev, True, eps=0.0, max_num_iter=3)
    _same(got, ref)
    assert its.tolist() == [3]
    del ref, got
    xt = torch.from_numpy(x).to(dev)
    runs = []
    for _ in range(2):
        iters = torch.zeros(1, dtype=torch.int32, device=dev)
        out = S._denoise_tv_chambolle(xt, 0.1, 2e-4, 200, None, None, True, iters)
        runs.append((out, int(iters.item())))
    assert runs[0][1] == runs[1][1] and 1 < runs[0][1] < 200
    assert torch.equal(runs[0][0], runs[1][0])
    f = (xt.to(torch.float64) * 2.0 + 1.0) / 65535.0
    assert abs(float(runs[0][0].mean()) - float(f.mean())) <= 1e-12


@pytest.mark.gpu
def test_batch_beyond_2_pow_31_elements(dev):
    from mie_b200 import skimage_compat as S

    h, w = 512, 500
    n = 2 ** 31 // (h * w) + 12          # 8400 planes, 2.15e9 elements
    straddle = 2 ** 31 // (h * w)       # plane 8388 holds element 2^31
    assert straddle * h * w < 2 ** 31 < (straddle + 1) * h * w and n * h * w > 2 ** 31
    base = torch.from_numpy(_img((8, h, w), np.float32, 15)).to(dev)
    x = base.repeat(n // 8 + 1, 1, 1)[:n].contiguous()
    x[straddle] = torch.flip(x[straddle], (1,))
    out = S.denoise_tv_chambolle(x, max_num_iter=2)
    for i in (0, straddle, n - 1):
        alone = S.denoise_tv_chambolle(x[i].clone(), max_num_iter=2)
        assert torch.equal(out[i], alone), i
    assert not torch.equal(out[straddle], out[straddle - 8])


@pytest.mark.gpu
@pytest.mark.parametrize("volumetric", [False, True])
def test_graph_capture_equals_the_eager_call(dev, volumetric):
    from mie_b200 import skimage_compat as S

    x = torch.from_numpy(_img((6, 48, 40) if volumetric else (3, 64, 72), np.uint16, 16)).to(dev)
    eager = S.denoise_tv_chambolle(x, volumetric=volumetric)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        S.denoise_tv_chambolle(x, volumetric=volumetric)   # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = S.denoise_tv_chambolle(x, volumetric=volumetric)
    for _ in range(2):
        captured.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(captured, eager)


@pytest.mark.gpu
def test_live_pin_against_skimage(dev):
    restoration = pytest.importorskip("skimage.restoration")
    for x, volumetric in [(_img((96, 80), np.uint16, 17), False), (_img((9, 40, 44), np.int16, 18), True)]:
        up = restoration.denoise_tv_chambolle(x)
        twin, _ = _twin(x)
        got, _ = _gpu(x, dev, volumetric)
        assert np.abs(twin - up).max() <= 1e-12
        assert np.abs(got - up).max() <= 1e-12
