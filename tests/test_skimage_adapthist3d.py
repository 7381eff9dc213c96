"""skimage.exposure.equalize_adapthist on whole 3-D volumes (skimage_compat.equalize_adapthist(..., volumetric=True),
mie_sk_equalize_adapthist3d).  RECALLED semantics like the 2-D path (tests/test_skimage_exposure.py).

CPU: the array-level numpy twin (oracle/skimage_twin.py, n-dimensional) and the per-voxel C restatement
(tests/sk_adapthist3d_oracle.c, built on oracle/mie_oracle.c) must agree BIT FOR BIT, stage by stage; a one-slice
volume with kd = 1 must give the 2-D oracle's result.  GPU: the CUDA path must reproduce the oracle bit for bit (float64 compared as bits)."""
import numpy as np
import pytest
import torch


def _vol_cases():
    from mie_b200 import synthetic

    rng = np.random.default_rng(7)
    ahe = rng.integers(0, 4096, (48, 48, 48)).astype(np.uint16)
    ahe[:30] = 0   # 30 * 48 * 48 = 69 120 voxels in one bin: above the 65 535 limit that clip_limit = 0 stands for
    return [
        ("phantom_volume 64^3 i16 default", synthetic.phantom_volume((64, 64, 64), np.int16, 0), None, 0.01, 256),
        ("uniform u16 (37, 50, 45) ragged", rng.integers(0, 65536, (37, 50, 45)).astype(np.uint16), None, 0.01, 256),
        ("anisotropic kernel (5, 7, 6) nbins 128", rng.integers(0, 65536, (23, 30, 29)).astype(np.uint16), (5, 7, 6), 0.03,
         128),
        ("u8 int kernel 8", rng.integers(0, 256, (20, 33, 27)).astype(np.uint8), 8, 0.02, 256),
        ("constant volume", np.full((16, 20, 18), 1000, np.uint16), None, 0.01, 256),
        ("clip_limit 0, 48^3 kernel, one bin above 65535", ahe, 48, 0.0, 256),
        ("float32 volume", rng.random((24, 30, 28)).astype(np.float32), None, 0.01, 256),
        ("volume smaller than one region (reflect pad longer than the axis)",
         rng.integers(0, 65536, (3, 5, 4)).astype(np.uint16), (7, 9, 10), 0.5, 64),
        ("two grey levels", (rng.integers(0, 2, (20, 24, 22)) * 3000).astype(np.uint16), None, 0.01, 256),
    ]


@pytest.mark.parametrize("case", _vol_cases(), ids=lambda c: c[0])
def test_adapthist3d_twin_and_per_voxel_restatement_agree(case):
    import sk_adapthist3d_oracle as V
    import skimage_twin as S

    _, x, ks, cl, nb = case
    a, sa = S.equalize_adapthist(x, ks, cl, nb, return_stages=True)
    b, sb = V.sk_equalize_adapthist3d(x, ks, cl, nb, return_stages=True)
    assert np.array_equal(sa["grey"], sb["grey"])
    assert np.array_equal(sa["clahe"], sb["clahe"])
    assert a.dtype == b.dtype and a.shape == x.shape and np.array_equal(a, b)
    assert a.min() >= 0.0 and a.max() <= 1.0


def test_clip_limit_zero_case_clips_at_65535():
    """The ASSUMED 'no clipping' limit of 65 535 takes effect in 3-D: the region's biggest bin exceeds it."""
    import sk_adapthist3d_oracle as V

    _, x, ks, cl, nb = [c for c in _vol_cases() if c[0].startswith("clip_limit 0")][0]
    _, st = V.sk_equalize_adapthist3d(x, ks, cl, nb, return_stages=True)
    assert st["maps"].shape == (1, 1, 1, nb)
    assert np.bincount((st["grey"] // (1 + 16384 // nb)).ravel()).max() > 65535
    # unclipped, the first bin alone would map to int(69 120 * 16383 / 110 592) = 10 238; clipped it maps lower
    assert st["maps"][0, 0, 0, 0] < 10238


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.float32])
@pytest.mark.parametrize("ks", [None, (17, 23), (4, 3)])
def test_single_slice_volume_equals_the_2d_image(dtype, ks):
    import oracle as O
    import sk_adapthist3d_oracle as V

    rng = np.random.default_rng(11)
    if dtype == np.float32:
        x = rng.random((100, 130)).astype(np.float32)
    else:
        x = rng.integers(0, np.iinfo(dtype).max + 1, (100, 130)).astype(dtype)
    ks3 = None if ks is None else (1,) + ks
    ref, sr = O.sk_equalize_adapthist(x, ks, 0.01, 256, return_stages=True)
    got, sg = V.sk_equalize_adapthist3d(x[None], ks3, 0.01, 256, return_stages=True)
    assert np.array_equal(sg["clahe"][0], sr["clahe"])
    assert got.dtype == ref.dtype and np.array_equal(got[0], ref)


def test_volumetric_argument_errors_need_no_gpu():
    from mie_b200 import skimage_compat as K

    v = torch.zeros(8, 8, 8, dtype=torch.uint16)
    with pytest.raises(ValueError):
        K.equalize_adapthist(torch.zeros(8, 8, dtype=torch.uint16), volumetric=True)
    with pytest.raises(ValueError):
        K.equalize_adapthist(torch.zeros(1, 1, 1, 8, 8, 8, dtype=torch.uint16), volumetric=True)
    with pytest.raises(ValueError):
        K.equalize_adapthist(v, kernel_size=(4, 4), volumetric=True)
    with pytest.raises(ValueError):
        K.equalize_adapthist(v, kernel_size=(4, 0, 4), volumetric=True)
    with pytest.raises(NotImplementedError):
        K.equalize_adapthist(v, nbins=5000, volumetric=True)
    with pytest.raises(TypeError):
        K.equalize_adapthist(np.zeros((8, 8, 8), np.uint16), volumetric=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        K.equalize_adapthist(v, volumetric=True)


def _align256(v):
    return (v + 255) // 256 * 256


def test_adapthist3d_workspace_query():
    from mie_b200 import _ffi

    L = _ffi.lib()
    # input ranges + result ranges, a 65 536-entry code -> bin table per volume, the region mappings, the uint16 volume
    assert L.mie_sk_adapthist3d_workspace_bytes(2, 64, 64, 64, 8, 8, 8, 256) == (
        256 + 2 * 65536 * 2 + 2 * 512 * 256 * 2 + 2 * 64 ** 3 * 2)
    assert L.mie_sk_adapthist3d_workspace_bytes(1, 37, 50, 45, 4, 6, 5, 128) == (
        256 + 65536 * 2 + _align256(10 * 9 * 9 * 128 * 2) + _align256(37 * 50 * 45 * 2))
    assert L.mie_sk_adapthist3d_workspace_bytes(0, 8, 8, 8, 2, 2, 2, 256) == 0
    assert L.mie_sk_adapthist3d_workspace_bytes(1, 8, 8, 8, 0, 2, 2, 256) == 0


def test_adapthist3d_abi_rejects_bad_arguments_before_any_launch():
    from mie_b200 import _ffi

    L = _ffi.lib()
    fake = 0x10000
    need = L.mie_sk_adapthist3d_workspace_bytes(1, 8, 8, 8, 4, 4, 4, 256)

    def call(src=fake, dst=fake, sd=1, dd=4, n=1, d=8, h=8, w=8, ss=(512, 64, 8), ds=(512, 64, 8), k=(4, 4, 4), nbins=256,
             ws=fake, wsb=need):
        return L.mie_sk_equalize_adapthist3d(src, dst, sd, dd, n, d, h, w, *ss, *ds, *k, 0.01, nbins, ws, wsb, None)

    assert call(k=(0, 4, 4)) == -7 and call(k=(4, 4, -1)) == -7            # MIE_E_KERNEL
    assert call(nbins=0) == -11 and call(nbins=4097) == -11                 # MIE_E_UNSUPPORTED
    assert call(k=(2000, 2000, 2000)) == -3                                 # kd * kr * kc > 2^31 - 1
    assert call(d=0) == -3 and call(n=-1) == -3 and call(n=65536) == -3      # MIE_E_SHAPE
    assert call(src=None) == -1 and call(ws=None) == -1                     # MIE_E_NULL
    assert call(ws=fake + 8) == -12                                         # MIE_E_ALIGN
    assert call(wsb=need - 1) == -9                                         # MIE_E_WORKSPACE
    assert call(sd=7) == -2 and call(dd=1) == -2                            # MIE_E_DTYPE
    assert call(ss=(512, 64, 7)) == -4 and call(ds=(512, 63, 8)) == -4      # MIE_E_STRIDE
    assert call(n=2, ss=(511, 64, 8)) == -4
    assert call(src=None, dst=None, n=0, ws=None, wsb=0) == 0               # empty batch: nothing to do


# ---------------------------------------------------------------------------------------------------- GPU parity
def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", _vol_cases(), ids=lambda c: c[0])
def test_gpu_equalize_adapthist3d_matches_oracle(dev, case):
    import sk_adapthist3d_oracle as V
    from mie_b200 import skimage_compat as K

    _, x, ks, cl, nb = case
    ref = V.sk_equalize_adapthist3d(x, ks, cl, nb)
    got = K.equalize_adapthist(torch.from_numpy(x).to(dev), ks, cl, nb, volumetric=True).cpu().numpy()
    assert got.dtype == ref.dtype and got.shape == ref.shape
    assert np.array_equal(_bits(got), _bits(ref)), int((got != ref).sum())
    if ref.dtype == np.float64:
        got32 = K.equalize_adapthist(torch.from_numpy(x).to(dev), ks, cl, nb, out_dtype=torch.float32,
                                     volumetric=True).cpu().numpy()
        assert np.array_equal(got32, ref.astype(np.float32))


@pytest.mark.gpu
def test_gpu_adapthist3d_batch_is_per_volume(dev):
    import sk_adapthist3d_oracle as V
    from mie_b200 import skimage_compat as K, synthetic

    x = np.stack([synthetic.phantom_volume((40, 56, 48), np.int16, s) for s in (1, 2)])
    x[1] //= 3
    xd = torch.from_numpy(x).to(dev)
    got = K.equalize_adapthist(xd, volumetric=True).cpu().numpy()
    for i in range(2):
        assert np.array_equal(_bits(got[i]), _bits(V.sk_equalize_adapthist3d(x[i])))
    # (B, C, D, H, W): the same volumes
    got5 = K.equalize_adapthist(xd[:, None], volumetric=True).cpu().numpy()
    assert got5.shape == (2, 1, 40, 56, 48) and np.array_equal(_bits(got5[:, 0]), _bits(got))


@pytest.mark.gpu
def test_gpu_adapthist3d_512_cube_phantom(dev):
    """A 512^3 int16 volume with the default 64^3 kernel: d * h = 262 144 rows (beyond a 65 535 grid dimension) and
    regions of 262 144 voxels counted by a cluster of CTAs."""
    import sk_adapthist3d_oracle as V
    from mie_b200 import skimage_compat as K, synthetic

    x = synthetic.phantom_volume((512, 512, 512), np.int16, 3)
    got = K.equalize_adapthist(torch.from_numpy(x).to(dev), volumetric=True).cpu().numpy()
    ref = V.sk_equalize_adapthist3d(x)
    assert np.array_equal(_bits(got), _bits(ref)), int((got != ref).sum())


@pytest.mark.gpu
def test_gpu_single_slice_volume_equals_the_2d_kernels(dev):
    from mie_b200 import skimage_compat as K, synthetic

    rng = np.random.default_rng(5)
    cases = [
        (synthetic.phantom((1, 1, 512, 512), np.uint16, 0)[0, 0], (64, 64)),
        (rng.integers(0, 65536, (100, 130)).astype(np.uint16), (17, 23)),
        (rng.integers(0, 256, (64, 61)).astype(np.uint8), (8, 8)),
        (rng.random((80, 72)).astype(np.float32), (10, 9)),
        (rng.integers(0, 65536, (5, 7)).astype(np.uint16), (4, 3)),
    ]
    for x, (kr, kc) in cases:
        xd = torch.from_numpy(x).to(dev)
        two_d = K.equalize_adapthist(xd, (kr, kc)).cpu().numpy()
        three_d = K.equalize_adapthist(xd[None], kernel_size=(1, kr, kc), volumetric=True)[0].cpu().numpy()
        assert np.array_equal(_bits(three_d), _bits(two_d))


def test_twins_against_real_skimage_volume():
    pytest.importorskip("skimage")
    from skimage import exposure

    import sk_adapthist3d_oracle as V
    import skimage_twin as S
    from mie_b200 import synthetic

    v = synthetic.phantom_volume((64, 64, 64), np.int16, 0)
    ref = exposure.equalize_adapthist(v)
    assert np.array_equal(S.equalize_adapthist(v), ref)
    assert np.array_equal(V.sk_equalize_adapthist3d(v), ref)


@pytest.mark.gpu
def test_cuda_volume_against_real_skimage(dev):
    pytest.importorskip("skimage")
    from skimage import exposure

    from mie_b200 import skimage_compat as K, synthetic

    v = synthetic.phantom_volume((64, 64, 64), np.int16, 0)
    got = K.equalize_adapthist(torch.from_numpy(v).to(dev), volumetric=True).cpu().numpy()
    assert np.array_equal(got, exposure.equalize_adapthist(v))
