"""skimage.filters.gaussian / unsharp_mask on whole 3-D volumes (skimage_compat.gaussian(..., volumetric=True),
skimage_compat.unsharp_mask(..., volumetric=True), mie_gaussian3d / mie_unsharp3d).

CPU: the per-voxel oracle (orc_gaussian3d_ex in tests/gaussian3d_oracle.c, built on oracle/mie_oracle.c) against scipy.ndimage.gaussian_filter in float64
on all five border modes, and with kz = 1 against the 2-D oracle bit for bit.  GPU: the CUDA kernel against the
oracle bit for bit (float32 compared as bits), and against the existing per-plane kernels when sigma_z = 0."""

import numpy as np
import pytest
import torch

MODES = ["nearest", "reflect", "mirror", "constant", "wrap"]

# Largest |oracle - scipy float64| on [0, 1] data measured over the cases below on the CPU: 2.7e-7 (gaussian) and
# 3.0e-7 (unsharp, amount <= 1.7).  The 2-D pin (tests/test_skimage_compat.py) uses 5e-7.
TOL = 5e-7


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _scipy_cases():
    return [
        ((9, 17, 23), 1.0, 4.0),
        ((9, 17, 23), (2.0, 0.7, 1.3), 4.0),      # anisotropic
        ((8, 33, 31), (0, 1.5, 1.0), 4.0),        # z not filtered
        ((5, 6, 7), (1.2, 0, 0.8), 3.0),          # y not filtered, truncate != 4
        ((6, 12, 10), 0.6, 2.5),
        ((1, 10, 12), 2.0, 4.0),                  # one slice, rz = 8
        ((3, 8, 8), (2.0, 2.0, 2.0), 4.0),        # thinner than the z radius on every axis
        ((2, 2, 2), 2.0, 4.0),
    ]


@pytest.mark.parametrize("mode", MODES)
def test_oracle_gaussian3d_matches_scipy(mode):
    import scipy.ndimage as ndi

    import gaussian3d_oracle as G

    rng = np.random.default_rng(0)
    for shape, sigma, truncate in _scipy_cases():
        x = rng.random(shape).astype(np.float32)
        got = G.skimage_gaussian3d(x, sigma, mode, truncate)
        ref = ndi.gaussian_filter(x.astype(np.float64), sigma, mode=mode, truncate=truncate, cval=0.0)
        assert got.dtype == np.float32 and got.shape == x.shape
        assert np.abs(got - ref).max() <= TOL, (shape, sigma, truncate)


@pytest.mark.parametrize("preserve_range", [False, True])
def test_oracle_unsharp3d_matches_scipy(preserve_range):
    import scipy.ndimage as ndi

    import gaussian3d_oracle as G

    rng = np.random.default_rng(1)
    for shape in [(9, 17, 23), (2, 5, 40)]:
        x = rng.random(shape).astype(np.float32)
        for radius, amount in [(1.0, 1.0), (2.0, 1.7), ((0.5, 1.0, 1.5), 0.5)]:
            got = G.skimage_unsharp_mask3d(x, radius, amount, preserve_range)
            x64 = x.astype(np.float64)
            ref = x64 + amount * (x64 - ndi.gaussian_filter(x64, radius, mode="reflect"))
            if not preserve_range:
                ref = np.clip(ref, 0.0, 1.0)
            assert np.abs(got - ref).max() <= TOL, (shape, radius, amount)


@pytest.mark.parametrize("mode", MODES)
def test_oracle_kz1_is_the_2d_oracle_per_plane(mode):
    import gaussian3d_oracle as G
    import oracle as O

    rng = np.random.default_rng(2)
    x = rng.random((4, 20, 30)).astype(np.float32)
    wz, wy, wx = G.gaussian_taps3d((0, 1.3, 0.8))
    assert wz.tolist() == [1.0]
    got = G.sep3d(x, wz, wy, wx, O.SCIPY_MODES[mode])
    ref = O.gaussian_blur2d(x, (wy.size, wx.size), (1.3, 0.8), O.SCIPY_MODES[mode])
    assert np.array_equal(_bits(got), _bits(ref))
    for amount, clip in [(1.0, 0), (1.7, 1)]:
        got = G.sep3d(x, wz, wy, wx, "symmetric", 1, amount, clip)
        ref = np.empty_like(x)
        O._check(O.lib().orc_gaussian2d_ex(O._ptr(x), O._ptr(ref), 4, 20, 30, O._ptr(wx), wx.size, O._ptr(wy), wy.size,
                                           O.BORDERS["symmetric"], 1, amount, clip))
        assert np.array_equal(_bits(got), _bits(ref))


def test_gaussian3d_abi_rejects_bad_arguments_before_any_launch():
    from mie_b200 import _ffi

    L = _ffi.lib()
    fake = 0x10000
    w9 = np.full(33, 1.0 / 9, np.float32)
    wp = w9.ctypes.data

    def call(fn="g", src=fake, dst=fake, sd=1, dd=1, n=1, d=8, h=8, w=8, ss=(512, 64, 8), ds=(512, 64, 8),
             k=(9, 9, 9), wts=(wp, wp, wp), border=2, lo=0.0, hi=65535.0):
        taps = (wts[0], k[0], wts[1], k[1], wts[2], k[2])
        if fn == "g":
            return L.mie_gaussian3d(src, dst, sd, dd, n, d, h, w, *ss, *ds, *taps, border, lo, hi, None)
        return L.mie_unsharp3d(src, dst, sd, dd, n, d, h, w, *ss, *ds, *taps, border, 1.5, 1, lo, hi, None)

    for fn in ("g", "u"):
        assert call(fn, k=(8, 9, 9)) == -7 and call(fn, k=(9, 0, 9)) == -7 and call(fn, k=(9, 9, 35)) == -7
        assert call(fn, k=(9, 9, -1)) == -7                                    # MIE_E_KERNEL
        assert call(fn, border=5) == -8 and call(fn, border=-1) == -8          # MIE_E_BORDER: unknown mode only
        assert call(fn, d=0) == -3 and call(fn, w=-1) == -3 and call(fn, n=-1) == -3   # MIE_E_SHAPE
        assert call(fn, src=None) == -1 and call(fn, dst=None) == -1           # MIE_E_NULL
        assert call(fn, wts=(wp, None, wp)) == -1
        assert call(fn, sd=7) == -2 and call(fn, dd=0) == -2                   # MIE_E_DTYPE: dst is src or F32
        assert call(fn, lo=1.0, hi=1.0) == -10                                 # MIE_E_RANGE
        assert call(fn, ss=(512, 64, 7)) == -4 and call(fn, ds=(512, 63, 8)) == -4   # MIE_E_STRIDE
        assert call(fn, n=2, ss=(511, 64, 8)) == -4
        assert call(fn, src=None, dst=None, n=0) == 0                          # empty batch: nothing to do
        # radius beyond the axis is legal for every mode (no F.pad limit): still n == 0, so nothing runs
        assert call(fn, n=0, d=1, h=2, w=3, ss=(6, 6, 3), ds=(6, 6, 3), k=(33, 33, 33), border=1) == 0


def test_python_argument_errors_before_the_device_check():
    from mie_b200 import skimage_compat as K

    vol = torch.zeros(4, 8, 8, dtype=torch.uint16)   # CPU tensor: every error below comes before require_cuda
    with pytest.raises(ValueError, match="volumetric=True expects"):
        K.gaussian(torch.zeros(8, 8), 1.0, volumetric=True)
    with pytest.raises(ValueError, match="volumetric=True expects"):
        K.unsharp_mask(torch.zeros(1, 1, 1, 1, 8, 8), volumetric=True)
    with pytest.raises(TypeError):
        K.gaussian(np.zeros((4, 8, 8)), volumetric=True)
    with pytest.raises(ValueError, match="non-negative"):
        K.gaussian(vol, (1.0, -1.0, 1.0), volumetric=True)
    with pytest.raises(ValueError, match="sigma_z"):
        K.gaussian(vol, (1.0, 1.0), volumetric=True)
    with pytest.raises(ValueError, match="taps"):
        K.gaussian(vol, (4.2, 1.0, 1.0), volumetric=True)
    with pytest.raises(ValueError, match="taps"):
        K.unsharp_mask(vol, 5.0, volumetric=True)
    with pytest.raises(ValueError, match="mode"):
        K.gaussian(vol, 1.0, mode="edge", volumetric=True)
    with pytest.raises(NotImplementedError):
        K.gaussian(vol, 1.0, mode="constant", cval=1, volumetric=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        K.gaussian(vol, (0, 1.0, 1.0), volumetric=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        K.unsharp_mask(vol, 1.0, 1.5, volumetric=True)


# ---------------------------------------------------------------------------------------------------- GPU parity
def _ref(x, sigma, mode="nearest", truncate=4.0, value_range=None, out_f32=False, unsharp=None):
    """Oracle result in the dtype the CUDA path returns: to01 -> orc_gaussian3d_ex -> from01."""
    import gaussian3d_oracle as G
    import oracle as O

    x01 = O.to01(x, value_range)
    if unsharp is None:
        y = G.skimage_gaussian3d(x01, sigma, mode, truncate)
    else:
        y = G.skimage_unsharp_mask3d(x01, sigma, *unsharp)
    return y if out_f32 or x.dtype == np.float32 else O.from01(y, x.dtype, value_range)


def _data(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == np.float32:
        return rng.random(shape).astype(np.float32)
    info = np.iinfo(dtype)
    return rng.integers(info.min, info.max + 1, shape).astype(dtype)


def _gpu_cases():
    u8, u16, i16, f32 = np.uint8, np.uint16, np.int16, np.float32
    cases = [
        # name, shape, dtype, sigma, mode, truncate, value_range, out_f32
        ("u8 sigma 1", (19, 37, 45), u8, 1.0, "nearest", 4.0, None, False),
        ("u16 anisotropic", (23, 50, 70), u16, (2.0, 0.7, 1.3), "reflect", 4.0, None, False),
        ("i16 zero z sigma", (11, 40, 33), i16, (0, 1.5, 1.0), "mirror", 4.0, None, False),
        ("f32 truncate 3", (9, 66, 97), f32, 1.2, "constant", 3.0, None, False),
        ("u16 -> f32", (13, 29, 41), u16, (1.0, 2.0, 0.5), "wrap", 4.0, None, True),
        ("i16 -> f32 zero y sigma", (12, 31, 40), i16, (1.0, 0, 1.0), "nearest", 4.0, None, True),
        ("33 taps on every axis", (40, 45, 70), u16, 4.0, "nearest", 4.0, None, False),
        ("x 33 taps, y 1, z 3", (10, 20, 80), u8, (0.25, 0, 4.0), "reflect", 4.0, None, False),
        ("d = 1", (1, 64, 64), i16, 1.0, "reflect", 4.0, None, False),
        ("d < rz", (3, 40, 40), u16, 2.0, "mirror", 4.0, None, False),
        ("ragged 2 x 17 taps", (70, 67, 131), u16, 2.0, "reflect", 4.0, None, False),
        ("HU window on int16", (17, 48, 52), i16, 1.0, "nearest", 4.0, (-1024.0, 3071.0), False),
        ("HU window -> f32", (17, 48, 52), i16, 1.0, "reflect", 4.0, (-1024.0, 3071.0), True),
    ]
    for mode in MODES:   # every axis shorter than its radius
        cases.append((f"thin {mode}", (2, 3, 5), u16, 2.0, mode, 4.0, None, False))
        cases.append((f"thin f32 {mode}", (5, 7, 2), f32, (2.0, 1.0, 3.0), mode, 4.0, None, False))
    # 1 .. 33 taps on each axis: radius r -> sigma r / 4 at truncate 4 (r = 0: sigma 0, one tap)
    for r in range(17):
        rz, ry, rx = r, (r + 5) % 17, (r + 11) % 17
        cases.append((f"taps {2 * rz + 1}/{2 * ry + 1}/{2 * rx + 1}", (21, 27, 38), u16, (rz / 4, ry / 4, rx / 4),
                      MODES[r % 5], 4.0, None, False))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("case", _gpu_cases(), ids=lambda c: c[0])
def test_gpu_gaussian3d_matches_oracle(dev, case):
    from mie_b200 import skimage_compat as K

    name, shape, dtype, sigma, mode, truncate, vr, out_f32 = case
    x = _data(shape, dtype, len(name))
    got = K.gaussian(torch.from_numpy(x).to(dev), sigma, mode=mode, truncate=truncate, value_range=vr,
                     out_dtype=torch.float32 if out_f32 else None, volumetric=True).cpu().numpy()
    ref = _ref(x, sigma, mode, truncate, vr, out_f32)
    assert got.dtype == ref.dtype and got.shape == ref.shape
    assert np.array_equal(_bits(got), _bits(ref)), int((got != ref).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.uint16, np.int16, np.float32])
@pytest.mark.parametrize("amount", [1.0, 1.7])
@pytest.mark.parametrize("preserve_range", [False, True])
def test_gpu_unsharp3d_matches_oracle(dev, dtype, amount, preserve_range):
    from mie_b200 import skimage_compat as K

    for shape, radius in [((14, 37, 45), 1.0), ((9, 30, 70), (0.5, 2.0, 1.0)), ((3, 20, 20), 2.0)]:
        x = _data(shape, dtype, 3)
        got = K.unsharp_mask(torch.from_numpy(x).to(dev), radius, amount, preserve_range, volumetric=True).cpu().numpy()
        ref = _ref(x, radius, unsharp=(amount, preserve_range))
        assert np.array_equal(_bits(got), _bits(ref)), (shape, radius, int((got != ref).sum()))
    if dtype != np.float32:
        got = K.unsharp_mask(torch.from_numpy(x).to(dev), radius, amount, preserve_range, out_dtype=torch.float32,
                             volumetric=True).cpu().numpy()
        assert np.array_equal(_bits(got), _bits(_ref(x, radius, out_f32=True, unsharp=(amount, preserve_range))))


@pytest.mark.gpu
def test_gpu_gaussian3d_batches_are_per_volume(dev):
    from mie_b200 import skimage_compat as K, synthetic

    x = np.stack([synthetic.phantom_volume((24, 40, 36), np.int16, s) for s in range(6)]).reshape(2, 3, 24, 40, 36)
    xd = torch.from_numpy(x).to(dev)
    got5 = K.gaussian(xd, (1.0, 1.5, 0.8), mode="mirror", volumetric=True).cpu().numpy()
    got4 = K.gaussian(xd.reshape(6, 24, 40, 36), (1.0, 1.5, 0.8), mode="mirror", volumetric=True).cpu().numpy()
    assert got5.shape == x.shape and np.array_equal(got5.reshape(got4.shape), got4)
    for i in range(6):
        one = K.gaussian(xd.reshape(6, 24, 40, 36)[i], (1.0, 1.5, 0.8), mode="mirror", volumetric=True).cpu().numpy()
        assert np.array_equal(got4[i], one)
    assert np.array_equal(got4[5], _ref(x.reshape(6, 24, 40, 36)[5], (1.0, 1.5, 0.8), "mirror"))
    u5 = K.unsharp_mask(xd, 1.0, 1.5, volumetric=True).cpu().numpy()
    for i in range(2):
        for c in range(3):
            assert np.array_equal(u5[i, c], K.unsharp_mask(xd[i, c], 1.0, 1.5, volumetric=True).cpu().numpy())


@pytest.mark.gpu
def test_gpu_zero_z_sigma_equals_the_per_plane_kernels(dev):
    """sigma (0, s, s) is the existing per-slice gaussian and radius (0, r, r) the existing unsharp_mask, bit for bit.
    (5, 128, 256) with 9 taps is the geometry of the 2-D marching kernel, the others run the 2-D tile kernels."""
    from mie_b200 import skimage_compat as K, synthetic

    cases = [
        (synthetic.phantom((1, 5, 128, 256), np.uint16, 0)[0], 1.0, "nearest"),
        (synthetic.phantom((1, 5, 128, 256), np.uint16, 1)[0], 1.0, "mirror"),
        (synthetic.phantom((1, 5, 128, 256), np.uint16, 2)[0], 1.0, "constant"),
        (_data((4, 37, 53), np.int16, 4), 1.3, "reflect"),
        (_data((3, 70, 90), np.uint8, 5), 2.0, "wrap"),
        (_data((3, 40, 44), np.float32, 6), 0.7, "nearest"),
    ]
    for x, s, mode in cases:
        xd = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
        two_d = K.gaussian(xd, s, mode=mode).cpu().numpy()
        three_d = K.gaussian(xd, (0, s, s), mode=mode, volumetric=True).cpu().numpy()
        assert np.array_equal(_bits(three_d), _bits(two_d)), (x.shape, s, mode)
        for amount, pr in [(1.0, True), (1.0, False), (1.7, False)]:
            two_d = K.unsharp_mask(xd, s, amount, pr).cpu().numpy()
            three_d = K.unsharp_mask(xd, (0, s, s), amount, pr, volumetric=True).cpu().numpy()
            assert np.array_equal(_bits(three_d), _bits(two_d)), (x.shape, s, amount, pr)


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [1.0, 2.0])
def test_gpu_gaussian3d_512_cube_phantom(dev, sigma):
    from mie_b200 import skimage_compat as K, synthetic

    x = synthetic.phantom_volume((512, 512, 512), np.int16, 3)
    got = K.gaussian(torch.from_numpy(x).to(dev), sigma, volumetric=True).cpu().numpy()
    ref = _ref(x, sigma)
    assert np.array_equal(got, ref), int((got != ref).sum())


@pytest.mark.gpu
def test_gpu_gaussian3d_batch_beyond_2_31_elements(dev):
    """17 x 512^3 uint8 = 2.28e9 elements: the last volume starts beyond 2^31, so 32-bit offsets would wrap."""
    from mie_b200 import skimage_compat as K, synthetic

    last = (synthetic.phantom_volume((512, 512, 512), np.uint16, 9) >> 4).astype(np.uint8)
    x = torch.empty((17, 512, 512, 512), dtype=torch.uint8, device=dev)
    x[:16] = 7
    x[16] = torch.from_numpy(last).to(dev)
    got = K.gaussian(x, 1.0, mode="reflect", volumetric=True)
    assert int(got[:16].min()) == 7 and int(got[:16].max()) == 7
    tail = got[16].cpu().numpy()
    del got, x
    ref = _ref(last, 1.0, "reflect")
    assert np.array_equal(tail, ref), int((tail != ref).sum())


@pytest.mark.gpu
def test_gpu_volume_against_real_skimage(dev):
    pytest.importorskip("skimage")
    from skimage import filters

    from mie_b200 import skimage_compat as K, synthetic

    v = synthetic.phantom_volume((32, 48, 40), np.uint16, 0)
    got = K.gaussian(torch.from_numpy(v).to(dev), 1.5, out_dtype=torch.float32, volumetric=True).cpu().numpy()
    assert np.abs(got - filters.gaussian(v, sigma=1.5)).max() < 1e-6
    u = np.random.default_rng(0).random((20, 30, 28)).astype(np.float32)
    got = K.unsharp_mask(torch.from_numpy(u).to(dev), 1.0, 1.5, volumetric=True).cpu().numpy()
    assert np.abs(got - filters.unsharp_mask(u.astype(np.float64), 1.0, 1.5)).max() < 1e-6
