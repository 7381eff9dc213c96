"""Every C-ABI entry point on non-dense layouts (include/mie.h: plane i at base + i*stride_n, row y at + y*stride_h,
strides in elements, for the source and the destination separately).

The Python layer always hands the library dense tensors, so a kernel that indexes with `w` instead of its row stride,
with `h*w` instead of its plane stride, or that addresses the destination with the source strides, computes the right
pixels there.  Here every image lives in a canvas: one flat byte buffer in which the region of interest (ROI) starts at
a chosen byte offset from a 256-byte aligned base and is laid out with chosen strides.  Source gaps are poisoned (NaN
for float32, alternating min / max codes for integers) so that a kernel reading padding changes its result;
destination gaps hold 0xA5 and must still do after the call; the source canvas must come back byte for byte.

The result read back from the ROI must equal, bit for bit, the same call on a dense copy of the ROI (layout D, which
is what the Python functions pass); one case per entry point is also compared directly with the CPU oracle.  Where the
tuned kernel is a separate kernel, the launched kernel names (torch.profiler, CUDA activity) show which variant ran."""
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENT = 0xA5
TAIL = 64   # canvas bytes behind the last ROI element (a store past the ROI lands there)
CODE = {np.uint8: 0, np.uint16: 1, np.int16: 2, np.float32: 3, np.float64: 4}
RANGE = {np.uint8: (0.0, 255.0), np.uint16: (0.0, 65535.0), np.int16: (-32768.0, 32767.0), np.float32: (0.0, 1.0)}
BITS = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}   # same-width integer view of a dtype
SENT_BITS = {1: SENT, 2: -23131, 4: -1515870811, 8: -6510615555426900571}   # 0xA5 in every byte, as signed integers
U8, U16, I16, F32 = np.uint8, np.uint16, np.int16, np.float32
INTS = (U8, U16, I16)
ALL = (U8, U16, I16, F32)


# ------------------------------------------------------------------------------------------------------------ layouts
def plane_strides(layout, e, h, w):
    """(byte offset of the ROI, row stride, plane stride) of a 2-D layout for elements of e bytes."""
    if layout == "D":
        return 0, w, h * w
    if layout == "P":       # padded rows, still 16-byte aligned
        return 16, w + 48, (h + 3) * (w + 48)
    if layout == "T":       # the tightest plane stride the ABI accepts: next plane right after the last row's pixels
        return 16, w + 48, (h - 1) * (w + 48) + w
    if layout == "U":       # every alignment guard must refuse
        return e, w + 1, h * (w + 1) + 3
    if layout == "H":       # 8-byte but not 16-byte aligned rows
        return 8, w + max(8 // e, 1), h * (w + max(8 // e, 1))
    if layout == "S":       # one plane, plane stride 0 (not checked for n == 1)
        return 16, w + 48, 0
    if layout == "G":       # plane offsets beyond 32 bits
        return 16, w + 48, (1 << 31) + 48
    raise ValueError(layout)


def layout_strides(layout, e, shape):
    """(byte offset, strides in ABI order) for a (n, h, w) or (n, d, h, w) ROI."""
    if len(shape) == 3:
        off, ssh, ssn = plane_strides(layout, e, shape[1], shape[2])
        return off, (ssn, ssh)
    n, d, h, w = shape
    off, ssh, ssd = plane_strides(layout, e, h, w)
    if layout == "D":
        return off, (d * ssd, ssd, ssh)
    if layout == "P":
        return off, ((d + 1) * ssd, ssd, ssh)
    if layout == "T":
        return off, ((d - 1) * ssd + (h - 1) * ssh + w, ssd, ssh)
    if layout == "U":
        return off, (d * ssd + 5, ssd, ssh)
    if layout == "H":
        return off, (d * ssd, ssd, ssh)
    if layout == "S":
        return off, (0, (h + 3) * ssh, ssh)
    if layout == "G":
        return off, ((1 << 31) + 48, (h + 3) * ssh, ssh)
    raise ValueError(layout)


class Canvas:
    """One ROI of `shape` elements of `dtype` inside a flat byte buffer on `dev`, laid out as `layout`."""

    def __init__(self, dev, dtype, shape, layout, role):
        self.dtype = np.dtype(dtype)
        self.e = self.dtype.itemsize
        self.shape = tuple(int(s) for s in shape)
        self.layout, self.role = layout, role
        self.off, self.strides = layout_strides(layout, self.e, self.shape)
        estr = self.strides + (1,)
        span = sum((s - 1) * st for s, st in zip(self.shape, estr)) + 1
        body = -(-(span * self.e + TAIL) // 8) * 8
        self.buf = torch.empty(self.off + body, dtype=torch.uint8, device=dev)
        assert self.buf.data_ptr() % 256 == 0 or not self.buf.is_cuda
        self.ptr = self.buf.data_ptr() + self.off
        self.estr = estr
        bits = self._bits()
        if role == "src":
            if self.dtype == np.float32:
                self.buf[self.off:].view(torch.float32).fill_(float("nan"))
                self.buf[:self.off].fill_(0xFF)     # a NaN pattern too, should a kernel read before the ROI
            else:
                info = np.iinfo(self.dtype)
                lo, hi = (np.array([info.min, info.max], self.dtype).view(f"i{self.e}") if self.e > 1
                          else np.array([info.min, info.max], self.dtype))
                bits.fill_(int(lo))
                bits[1::2] = int(hi)
                self.buf[:self.off].fill_(int(hi) & 0xFF)
        else:
            self.buf.fill_(SENT)

    def _bits(self):
        return self.buf[self.off:].view(BITS[self.e])

    def _roi(self):
        return torch.as_strided(self._bits(), self.shape, self.estr)

    def write(self, x):
        x = np.ascontiguousarray(x, self.dtype)
        assert x.shape == self.shape
        self._roi().copy_(torch.from_numpy(x.view(f"i{self.e}") if self.e > 1 else x).to(self.buf.device))
        torch.cuda.synchronize()
        self.snapshot = self.buf.clone()

    def read(self):
        torch.cuda.synchronize()
        return self._roi().contiguous().cpu().numpy().view(self.dtype).copy()

    def check_source_unchanged(self, what):
        torch.cuda.synchronize()
        assert torch.equal(self.buf, self.snapshot), f"{what}: the source canvas was written"

    def check_gaps(self, what):
        """Every byte outside the ROI still holds the sentinel (restores the ROI to the sentinel to test at once)."""
        torch.cuda.synchronize()
        self._roi().fill_(SENT_BITS[self.e])
        bad = (self.buf != SENT).nonzero()
        assert bad.numel() == 0, (f"{what}: {bad.numel()} gap bytes of the {self.layout} destination written, "
                                  f"first at byte {int(bad[0]) - self.off} from the ROI base")


class Dense:
    """A dense device output (histograms, LUTs, metric sums: their layout is fixed by the ABI) with sentinels."""

    def __init__(self, dev, dtype, shape):
        self.dtype, self.shape = np.dtype(dtype), tuple(shape)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.buf = torch.full((self.nbytes + 512,), SENT, dtype=torch.uint8, device=dev)
        self.ptr = self.buf.data_ptr() + 256

    def read(self, what):
        torch.cuda.synchronize()
        assert bool((self.buf[:256] == SENT).all()) and bool((self.buf[256 + self.nbytes:] == SENT).all()), \
            f"{what}: wrote outside the dense output"
        raw = self.buf[256:256 + self.nbytes].cpu().numpy()
        return raw.view(self.dtype).reshape(self.shape).copy()


def workspace(dev, nbytes):
    return torch.empty(max(int(nbytes), 1) + 256, dtype=torch.uint8, device=dev)


def stream():
    return torch.cuda.current_stream().cuda_stream


def rand(dtype, shape, seed):
    rng = np.random.default_rng(seed)
    if dtype == F32:
        return rng.random(shape, dtype=np.float32)
    info = np.iinfo(dtype)
    return rng.integers(info.min, int(info.max) + 1, shape).astype(dtype)


def launched_kernels(fn):
    """Names of the CUDA kernels `fn` launches (torch.profiler with CUDA activity only)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def ran(names, kernel):
    return any(re.search(rf"\b{kernel}\b", s) for s in names)


def lib():
    from mie_b200 import _ffi
    return _ffi.lib()


def check(rc):
    from mie_b200 import _ffi
    _ffi.check(rc)


def taps(k, sigma=1.0):
    from mie_b200.filters import get_gaussian_kernel1d
    return np.ascontiguousarray(get_gaussian_kernel1d(k, sigma), np.float32)


# ------------------------------------------------------------------------------------------------ entry-point table
class Op:
    """One entry point with fixed parameters.  call(dev, srcs, dst, dtype, shape) launches it; srcs are Canvas
    objects (two for the metrics), dst a Canvas, or None when out_shape() names a dense output."""

    def __init__(self, name, dtypes, shape, call, out_dtype=None, out_shape=None, nsrc=1, oracle=None, tol=None,
                 policy=()):
        self.name, self.dtypes, self.shape, self.call = name, dtypes, shape, call
        self.out_dtype = out_dtype or (lambda dt: dt)
        self.out_shape, self.nsrc, self.oracle, self.tol, self.policy = out_shape, nsrc, oracle, tol, policy


def _lohi(dt):
    return RANGE[dt]


def _gauss(fn, kx, ky, border, amount=None):
    def call(dev, s, d, dt, shape):
        wx, wy = taps(kx), taps(ky)
        lo, hi = _lohi(dt)
        n, h, w = shape
        args = (s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides,
                wx.ctypes.data, kx, wy.ctypes.data, ky, border)
        if amount is None:
            return getattr(lib(), fn)(*args, lo, hi, stream())
        return lib().mie_unsharp_amount(*args, amount, 1, lo, hi, stream())
    return call


def _o_sep(kx, ky, border, unsharp, amount=None):
    def oracle(x, dt):
        import oracle as O
        x01 = O.to01(x)
        if amount is not None:
            return O.from01(O.skimage_unsharp_mask(x01, 1.0, amount), dt)
        f = O.unsharp_mask if unsharp else O.gaussian_blur2d
        return O.from01(f(x01, (ky, kx), 1.0, border), dt)
    return oracle


def _clahe_hist(grid):
    def call(dev, s, out, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        return lib().mie_clahe_hist(s[0].ptr, CODE[dt], n, h, w, *s[0].strides, grid[0], grid[1], 0, lo, hi, out.ptr,
                                    stream())
    return call


def _clahe_luts(grid, sem):
    def call(dev, s, out, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        if sem == 16:
            return lib().mie_clahe16_luts(s[0].ptr, n, h, w, *s[0].strides, grid[0], grid[1], 2.0, out.ptr, stream())
        return lib().mie_clahe_luts(s[0].ptr, CODE[dt], n, h, w, *s[0].strides, grid[0], grid[1], 2.0, sem, lo, hi,
                                    out.ptr, stream())
    return call


def _clahe_apply(grid):
    def call(dev, s, d, dt, shape):
        import oracle as O
        lo, hi = _lohi(dt)
        n, h, w = shape
        # LUTs of the dense input from the oracle: the stage is tested on its own
        luts = torch.from_numpy(O.clahe_luts(O.to01(call.x), 2.0, grid).reshape(-1)).to(dev)
        return lib().mie_clahe_apply(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides,
                                     grid[0], grid[1], 0, lo, hi, luts.data_ptr(), stream())
    return call


def _clahe(grid, sem):
    def call(dev, s, d, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        if sem == 1 and dt == U16:
            need = lib().mie_clahe16_lut_bytes(grid[0], grid[1]) * n + 256
        else:
            need = lib().mie_clahe_workspace_bytes(n, h, w, grid[0], grid[1])
        ws = workspace(dev, need)
        return lib().mie_clahe(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides,
                               grid[0], grid[1], 2.0, sem, lo, hi, ws.data_ptr(), need, stream())
    return call


def _o_clahe(grid, sem):
    def oracle(x, dt):
        import oracle as O
        if sem == 1:
            return O.opencv_clahe(x, 2.0, grid)
        return O.from01(O.equalize_clahe(O.to01(x), 2.0, grid), dt)
    return oracle


def _equalize(dev, s, d, dt, shape):
    lo, hi = _lohi(dt)
    n, h, w = shape
    need = lib().mie_equalize_workspace_bytes(n)
    ws = workspace(dev, need)
    return lib().mie_equalize(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides, lo, hi,
                              ws.data_ptr(), need, stream())


def _median2d(ky, kx, border):
    def call(dev, s, d, dt, shape):
        n, h, w = shape
        return lib().mie_median2d(s[0].ptr, d.ptr, CODE[dt], n, h, w, *s[0].strides, *d.strides, ky, kx, border,
                                  stream())
    return call


def _median3d(border, halos):
    def call(dev, s, d, dt, shape):
        dd, h, w = shape
        lo = hi = None
        if halos:
            call.halo = [torch.from_numpy(rand(dt, (h, w), 90 + i).view(f"i{np.dtype(dt).itemsize}")
                                          if np.dtype(dt).itemsize > 1 else rand(dt, (h, w), 90 + i)).to(dev)
                         for i in range(2)]
            lo, hi = call.halo[0].data_ptr(), call.halo[1].data_ptr()
        return lib().mie_median3d(s[0].ptr, d.ptr, CODE[dt], dd, h, w, *s[0].strides, *d.strides, lo, hi, border,
                                  stream())
    return call


def _o_median3d(border, halos):
    def oracle(x, dt):
        import oracle as O
        h, w = x.shape[1:]
        hl = (rand(dt, (h, w), 90), rand(dt, (h, w), 91)) if halos else (None, None)
        return O.median3d(x, {2: "nearest", 0: "constant"}[border], *hl)
    return oracle


def _wsp(k, s=1.5):
    k1 = taps(k, s)
    return np.ascontiguousarray((k1[:, None] * k1[None, :]).astype(np.float32))


def _bilateral(k):
    def call(dev, s, d, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        wsp = _wsp(k)
        return lib().mie_bilateral(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides,
                                   wsp.ctypes.data, k, k, 0.1, 1, lo, hi, stream())
    return call


def _o_bilateral(k):
    def oracle(x, dt):
        import oracle as O
        return O.from01(O.bilateral_blur(O.to01(x), k, 0.1, (1.5, 1.5), "reflect"), dt)
    return oracle


def _nlm(dev, s, d, dt, shape):
    lo, hi = _lohi(dt)
    n, h, w = shape
    return lib().mie_nlm(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides, 5, 6, 0.1,
                         0.0, lo, hi, stream())


def _nlm_slow(dev, s, d, dt, shape):
    lo, hi = _lohi(dt)
    n, h, w = shape
    return lib().mie_nlm_slow(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides, *d.strides, 5, 4,
                              0.1, 0.0, lo, hi, stream())


def _o_nlm(slow):
    def oracle(x, dt):
        import oracle as O
        x01 = O.to01(x).astype(np.float64)
        if slow:
            return O.denoise_nl_means_slow(x01, 5, 4, 0.1, 0.0)
        return O.denoise_nl_means(x01, 5, 6, 0.1, 0.0)
    return oracle


def _sqdiff(dev, s, out, dt, shape):
    n, h, w = shape
    need = lib().mie_metric_workspace_bytes(n, h, w, 0)
    ws = workspace(dev, need)
    return lib().mie_sqdiff_sums(s[0].ptr, s[1].ptr, CODE[dt], n, h, w, *s[0].strides, *s[1].strides, out.ptr,
                                 ws.data_ptr(), need, stream())


def _ssim(dev, s, out, dt, shape):
    n, h, w = shape
    need = lib().mie_metric_workspace_bytes(n, h, w, 7)
    ws = workspace(dev, need)
    return lib().mie_ssim_sums(s[0].ptr, s[1].ptr, CODE[dt], n, h, w, *s[0].strides, *s[1].strides, 7, 6.5, 58.5,
                               out.ptr, ws.data_ptr(), need, stream())


def _o_sqdiff(a, b, dt):
    d = a.astype(np.float64) - b.astype(np.float64)
    return np.stack([(d * d).sum(axis=(1, 2)), np.abs(d).sum(axis=(1, 2))], axis=1)


def _o_ssim(a, b, dt):
    from scipy.signal import convolve2d
    ws = 7
    out = []
    for g, p in zip(a.astype(np.float64), b.astype(np.float64)):
        f = lambda x: convolve2d(x, np.ones((ws, ws)) / ws ** 2, mode="valid")  # noqa: E731
        m1, m2 = f(g), f(p)
        s1, s2, s12 = f(g * g) - m1 * m1, f(p * p) - m2 * m2, f(g * p) - m1 * m2
        ssim = ((2 * m1 * m2 + 6.5) * (2 * s12 + 58.5)) / ((m1 * m1 + m2 * m2 + 6.5) * (s1 + s2 + 58.5))
        cs = (2 * s12 + 58.5) / (s1 + s2 + 58.5)
        out.append([ssim.sum(), cs.sum()])
    return np.array(out)


def _chain(grid, stages):
    def call(dev, s, d, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        t = taps(9)
        need = lib().mie_chain_workspace_bytes(n, h, w, grid[0], grid[1])
        ws = workspace(dev, need)
        return lib().mie_chain_gauss_clahe_unsharp(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides,
                                                   *d.strides, t.ctypes.data, 9, t.ctypes.data, 9, grid[0], grid[1], 2.0,
                                                   t.ctypes.data, 9, t.ctypes.data, 9, 1, lo, hi, stages, ws.data_ptr(),
                                                   need, stream())
    return call


def _o_chain(grid):
    def oracle(x, dt):
        import oracle as O
        return O.chain_gauss_clahe_unsharp(x, grid_size=grid)
    return oracle


def _bilateral_clahe(grid):
    def call(dev, s, d, dt, shape):
        lo, hi = _lohi(dt)
        n, h, w = shape
        wsp = _wsp(9)
        need = lib().mie_bilateral_clahe_workspace_bytes(n, h, w, grid[0], grid[1])
        ws = workspace(dev, need)
        return lib().mie_bilateral_clahe(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides,
                                         *d.strides, wsp.ctypes.data, 9, 0.1, 1, grid[0], grid[1], 2.0, lo, hi, 7,
                                         ws.data_ptr(), need, stream())
    return call


def _o_bilateral_clahe(grid):
    def oracle(x, dt):
        import oracle as O
        return O.from01(O.equalize_clahe(O.bilateral_blur(O.to01(x), 9, 0.1, (1.5, 1.5), "reflect"), 2.0, grid), dt)
    return oracle


def _sk_out(dt):
    return F32 if dt == F32 else np.float64


def _sk_adapthist(k):
    def call(dev, s, d, dt, shape):
        n, h, w = shape
        need = lib().mie_sk_adapthist_workspace_bytes(n, h, w, k[0], k[1], 256)
        ws = workspace(dev, need)
        return lib().mie_sk_equalize_adapthist(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides,
                                               *d.strides, k[0], k[1], 0.01, 256, ws.data_ptr(), need, stream())
    return call


def _sk_eqhist(dev, s, d, dt, shape):
    n, h, w = shape
    need = lib().mie_sk_equalize_hist_workspace_bytes(n, CODE[dt])
    ws = workspace(dev, need)
    return lib().mie_sk_equalize_hist(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides,
                                      *d.strides, ws.data_ptr(), need, stream())


def sk_bilateral_tables(x, dt, win, sigma_color, sigma_spatial, bins):
    """The host tables of skimage_compat.denoise_bilateral (per-plane colour LUT, spatial LUT, (min, max) codes)."""
    flat = x.reshape(x.shape[0], -1).astype(np.int64)
    ranges = np.stack([flat.min(axis=1), flat.max(axis=1)], axis=1).astype(np.int32)
    f = ranges.astype(np.float64)
    f = f / 255.0 if dt == U8 else (f / 65535.0 if dt == U16 else (f * 2.0 + 1.0) / 65535.0)
    max_value = np.where(f[:, 0] < 0, f[:, 1] - f[:, 0], f[:, 1])
    luts = np.ones((x.shape[0], bins), np.float64)
    for i in range(x.shape[0]):
        if ranges[i, 0] != ranges[i, 1]:
            values = np.linspace(0, max_value[i], bins, endpoint=False)
            luts[i] = np.exp(-0.5 * (values ** 2 / sigma_color ** 2))
    ext = (win - 1) // 2
    g = np.arange(-ext, ext + 1)
    rr, cc = np.meshgrid(g, g, indexing="ij")
    spatial = np.exp(-0.5 * (np.hypot(rr, cc) ** 2 / float(sigma_spatial) ** 2)).ravel()
    return luts, spatial, ranges


def _sk_bilateral(dev, s, d, dt, shape):
    n, h, w = shape
    luts, spatial, ranges = sk_bilateral_tables(_sk_bilateral.x, dt, 5, 0.1, 1.0, 1000)
    dl, dsp, dr = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (luts, spatial, ranges))
    _sk_bilateral.keep = (dl, dsp, dr)
    return lib().mie_sk_denoise_bilateral(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, h, w, *s[0].strides,
                                          *d.strides, 5, 1000, 2, 0.0, dl.data_ptr(), dsp.data_ptr(), dr.data_ptr(),
                                          stream())


def _per_plane(f):
    def oracle(x, dt):
        return np.stack([f(p) for p in x])
    return oracle


def _gauss3d(unsharp, kz):
    def call(dev, s, d, dt, shape):
        lo, hi = _lohi(dt)
        n, dd, h, w = shape
        wx, wy, wz = taps(9), taps(7, 0.8), (taps(kz, 1.2) if kz > 1 else np.ones(1, np.float32))
        args = (s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, dd, h, w, *s[0].strides, *d.strides,
                wx.ctypes.data, 9, wy.ctypes.data, 7, wz.ctypes.data, wz.size, 4)
        if unsharp:
            return lib().mie_unsharp3d(*args, 1.5, 1, lo, hi, stream())
        return lib().mie_gaussian3d(*args, lo, hi, stream())
    return call


def _o_gauss3d(unsharp, kz):
    def oracle(x, dt):
        import oracle as O
        from gaussian3d_oracle import sep3d
        wz = taps(kz, 1.2) if kz > 1 else np.ones(1, np.float32)
        y = sep3d(O.to01(x), wz, taps(7, 0.8), taps(9), "symmetric", int(unsharp), 1.5 if unsharp else 1.0,
                  int(unsharp))
        return O.from01(y, dt)
    return oracle


def _adapthist3d(dev, s, d, dt, shape):
    n, dd, h, w = shape
    k = (2, 8, 16)
    need = lib().mie_sk_adapthist3d_workspace_bytes(n, dd, h, w, *k, 128)
    ws = workspace(dev, need)
    return lib().mie_sk_equalize_adapthist3d(s[0].ptr, d.ptr, CODE[dt], CODE[d.dtype.type], n, dd, h, w, *s[0].strides,
                                             *d.strides, *k, 0.02, 128, ws.data_ptr(), need, stream())


def _o_adapthist3d(x, dt):
    from sk_adapthist3d_oracle import sk_equalize_adapthist3d
    return np.stack([sk_equalize_adapthist3d(v, (2, 8, 16), 0.02, 128) for v in x])


def _o_sk(which):
    def oracle(x, dt):
        import oracle as O
        if which == "adapthist":
            return np.stack([O.sk_equalize_adapthist(p, (16, 32), 0.01, 256) for p in x])
        if which == "eqhist":
            return np.stack([O.sk_equalize_hist(p) for p in x])
        return np.stack([O.sk_denoise_bilateral(p, 5, 0.1, 1.0, 1000, "symmetric") for p in x])
    return oracle


# shapes: the tuned Gaussian needs W % 128 == 0, H % 64 == 0 and 9 taps; the tuned chain 64 x 64 tiles; the tuned CLAHE
# tiles of a multiple of 8 (16 for uint8) pixels; the packed medians W % 8 == 0
S2 = (2, 64, 128)
OPS = [
    Op("gaussian9", ALL, S2, _gauss("mie_gaussian2d", 9, 9, 1), oracle=_o_sep(9, 9, "reflect", 0)),
    Op("gaussian9_f32out", INTS, S2, _gauss("mie_gaussian2d", 9, 9, 1), out_dtype=lambda dt: F32),
    Op("gaussian5_symmetric", ALL, (2, 40, 72), _gauss("mie_gaussian2d", 5, 5, 4), oracle=_o_sep(5, 5, "symmetric", 0)),
    Op("gaussian11x7", ALL, (2, 40, 72), _gauss("mie_gaussian2d", 11, 7, 2), oracle=_o_sep(11, 7, "replicate", 0)),
    Op("unsharp9", ALL, S2, _gauss("mie_unsharp", 9, 9, 1), oracle=_o_sep(9, 9, "reflect", 1)),
    Op("unsharp_amount", ALL, (2, 40, 72), _gauss("mie_unsharp_amount", 9, 9, 4, amount=1.5),
       oracle=_o_sep(9, 9, "symmetric", 1, amount=1.5)),
    Op("clahe_hist", ALL, (2, 128, 128), _clahe_hist((4, 4)), out_shape=lambda n: (n, 4, 4, 256),
       out_dtype=lambda dt: np.uint32),
    Op("clahe_luts", ALL, (2, 128, 128), _clahe_luts((4, 4), 0), out_shape=lambda n: (n, 4, 4, 256),
       out_dtype=lambda dt: np.uint8),
    Op("clahe_luts_opencv", (U8,), (2, 128, 128), _clahe_luts((4, 4), 1), out_shape=lambda n: (n, 4, 4, 256),
       out_dtype=lambda dt: np.uint8),
    Op("clahe16_luts", (U16,), (2, 128, 128), _clahe_luts((2, 2), 16), out_shape=lambda n: (n, 2, 2, 65536),
       out_dtype=lambda dt: np.uint16),
    Op("clahe_apply", ALL, (2, 128, 128), _clahe_apply((4, 4))),
    Op("clahe", ALL, (2, 128, 128), _clahe((4, 4), 0), oracle=_o_clahe((4, 4), 0)),
    Op("clahe_opencv", (U8, U16), (2, 128, 128), _clahe((4, 4), 1), oracle=_o_clahe((4, 4), 1)),
    Op("equalize", ALL, S2, _equalize, oracle=lambda x, dt: __import__("oracle").from01(
        __import__("oracle").equalize(__import__("oracle").to01(x)), dt)),
    Op("equalize_slab", ALL, S2, _equalize, policy=("equalize_slab",)),
    Op("equalize_three_pass", ALL, S2, _equalize, policy=("equalize_three_pass",)),
    Op("median3", ALL, (2, 40, 64), _median2d(3, 3, 0), oracle=lambda x, dt: __import__("oracle").median_blur(x, 3)),
    Op("median5", ALL, (2, 40, 64), _median2d(5, 5, 2)),
    Op("median7", ALL, (2, 40, 64), _median2d(7, 7, 4)),
    Op("median3x5", ALL, (2, 40, 64), _median2d(3, 5, 1)),
    Op("median3d", ALL, (6, 24, 64), _median3d(2, False), oracle=_o_median3d(2, False)),
    Op("median3d_halos", ALL, (6, 24, 64), _median3d(0, True), oracle=_o_median3d(0, True)),
    Op("bilateral", ALL, (2, 40, 72), _bilateral(9), oracle=_o_bilateral(9), tol="tolerance"),
    Op("bilateral15_exact", ALL, (2, 40, 72), _bilateral(15), policy=("bilateral_exact_exp",)),
    Op("bilateral_exact", ALL, (2, 40, 72), _bilateral(9), oracle=_o_bilateral(9), policy=("bilateral_exact_exp",)),
    Op("nlm", ALL, (2, 24, 40), _nlm, out_dtype=lambda dt: F32, oracle=_o_nlm(False), tol="tolerance"),
    Op("nlm_slow", ALL, (2, 16, 24), _nlm_slow, out_dtype=lambda dt: np.float64, oracle=_o_nlm(True),
       tol=1e-13),
    Op("sqdiff_sums", ALL, (2, 40, 64), _sqdiff, nsrc=2, out_shape=lambda n: (n, 2), out_dtype=lambda dt: np.float64,
       oracle=_o_sqdiff),
    Op("ssim_sums", ALL, (2, 40, 64), _ssim, nsrc=2, out_shape=lambda n: (n, 2), out_dtype=lambda dt: np.float64,
       oracle=_o_ssim, tol=1e-9),
    Op("chain", ALL, (2, 128, 256), _chain((2, 4), 3), oracle=_o_chain((2, 4))),
    Op("chain_march", ALL, (2, 128, 256), _chain((2, 4), 3 | 4)),
    Op("chain_tiles", ALL, (2, 128, 256), _chain((2, 4), 3 | 8)),
    Op("chain_unfused", ALL, (2, 100, 72), _chain((2, 3), 3), oracle=_o_chain((2, 3))),
    Op("bilateral_clahe", ALL, (2, 128, 128), _bilateral_clahe((4, 4))),
    Op("bilateral_clahe_exact", ALL, (2, 128, 128), _bilateral_clahe((4, 4)), oracle=_o_bilateral_clahe((4, 4)),
       policy=("bilateral_exact_exp",)),
    Op("sk_equalize_adapthist", ALL, (2, 64, 96), _sk_adapthist((16, 32)), out_dtype=_sk_out,
       oracle=_o_sk("adapthist")),
    Op("sk_equalize_hist", INTS, (2, 40, 72), _sk_eqhist, out_dtype=lambda dt: np.float64, oracle=_o_sk("eqhist")),
    Op("sk_denoise_bilateral", INTS, (2, 40, 72), _sk_bilateral, out_dtype=lambda dt: np.float64,
       oracle=_o_sk("bilateral")),
    Op("gaussian3d", ALL, (2, 6, 24, 48), _gauss3d(False, 5), oracle=_o_gauss3d(False, 5)),
    Op("unsharp3d", ALL, (2, 6, 24, 48), _gauss3d(True, 3), oracle=_o_gauss3d(True, 3)),
    Op("sk_equalize_adapthist3d", ALL, (2, 6, 24, 48), _adapthist3d, out_dtype=_sk_out, oracle=_o_adapthist3d),
]
OP = {op.name: op for op in OPS}
LAYOUTS = [("D", "D"), ("P", "P"), ("T", "T"), ("U", "U"), ("H", "H"), ("P", "U"), ("U", "P"), ("S", "S")]


def _partner(layout):
    """Layout of the second metric input: always a different one."""
    return {"D": "P", "P": "U", "T": "H", "U": "T", "H": "D", "S": "S"}[layout]


def run(op, dt, src_layout, dst_layout, dev, shape=None, src_canvas=None, kernels=False):
    """Run `op` with its source(s) in src_layout and its image output in dst_layout; every poison / sentinel check
    applies.  Returns (output as a dense numpy array, launched kernel names or None)."""
    from mie_b200 import _ffi

    shape = tuple(shape or op.shape)
    if src_layout == "S":
        shape = (1,) + shape[1:]
    x = rand(dt, shape, 7)
    srcs = []
    if src_canvas is not None:
        srcs.append(src_canvas)
    else:
        c = Canvas(dev, dt, shape, src_layout, "src")
        c.write(x)
        srcs.append(c)
    if op.nsrc == 2:
        c = Canvas(dev, dt, shape, _partner(src_layout), "src")
        c.write(rand(dt, shape, 8))
        srcs.append(c)
    out_dt = op.out_dtype(dt)
    dst = (Dense(dev, out_dt, op.out_shape(shape[0])) if op.out_shape
           else Canvas(dev, out_dt, shape, dst_layout, "dst"))
    op.call.x = x
    what = f"{op.name} {np.dtype(dt).name} src {src_layout} dst {dst_layout} {shape}"
    names = None
    with _ffi.kernel_policy(*op.policy):
        if kernels:
            rc = []
            names = launched_kernels(lambda: rc.append(op.call(dev, srcs, dst, dt, shape)))
            rc = rc[0]
        else:
            rc = op.call(dev, srcs, dst, dt, shape)
        check(rc)
        torch.cuda.synchronize()
    for c in srcs:
        c.check_source_unchanged(what)
    if op.out_shape:
        out = dst.read(what)
    else:
        out = dst.read()
        dst.check_gaps(what)
    return out, names


_REF = {}


def reference(op, dt, n, dev):
    """The same call on a dense copy of the ROI (layout D for every buffer: what the Python functions pass)."""
    key = (op.name, dt, n)
    if key not in _REF:
        shape = (n,) + tuple(op.shape[1:])
        _REF[key] = run(op, dt, "D", "D", dev, shape=shape)[0]
    return _REF[key]


def assert_same(got, ref, what):
    assert got.shape == ref.shape and got.dtype == ref.dtype, what
    same = (got.view(np.uint8) == ref.view(np.uint8)).reshape(got.shape + (-1,)).all(axis=-1) if got.dtype.itemsize > 1 \
        else got == ref
    nbad = int((~same).sum())
    assert nbad == 0, f"{what}: {nbad} of {got.size} values differ from the dense layout, first at " \
                      f"{np.unravel_index(int(np.argmin(same.reshape(-1))), got.shape)}"


CASES = [(name, dt, sl, dl) for name, op in OP.items() for dt in op.dtypes for sl, dl in LAYOUTS
         if not (op.out_shape and sl != dl)]


@pytest.mark.parametrize("name,dt,src_layout,dst_layout", CASES,
                         ids=[f"{n}-{np.dtype(d).name}-{s}{t}" for n, d, s, t in CASES])
def test_layout_matches_dense(dev, name, dt, src_layout, dst_layout):
    op = OP[name]
    got, _ = run(op, dt, src_layout, dst_layout, dev)
    ref = reference(op, dt, got.shape[0], dev)
    assert_same(got, ref, f"{name} {np.dtype(dt).name} {src_layout}->{dst_layout}")


# ------------------------------------------------------------------------------------------------- oracle, directly
ORACLE_CASES = [(name, dt) for name, op in OP.items() if op.oracle for dt in op.dtypes]


@pytest.mark.parametrize("name,dt", ORACLE_CASES, ids=[f"{n}-{np.dtype(d).name}" for n, d in ORACLE_CASES])
def test_padded_layout_matches_oracle(dev, name, dt):
    """Source padded (P), destination misaligned (U) — or dense outputs — against the CPU reference of the dense ROI."""
    op = OP[name]
    got, _ = run(op, dt, "P", "U", dev)
    x = rand(dt, op.shape, 7)
    if op.nsrc == 2:
        ref = op.oracle(x, rand(dt, op.shape, 8), dt)
    else:
        ref = op.oracle(x, dt)
    ref = np.asarray(ref).reshape(got.shape)
    what = f"{name} {np.dtype(dt).name} vs oracle"
    if op.tol == "tolerance":   # MUFU.EX2 colour / patch weights: the bars of the existing tests
        if got.dtype == np.float32 or dt == F32:
            g, r = got.astype(np.float64), ref.astype(np.float64)
            assert float((np.abs(g - r) / np.maximum(np.abs(r), 1e-3)).max()) <= 1e-5, what
        else:
            assert int(np.abs(got.astype(np.int64) - ref.astype(np.int64)).max()) <= 1, what
    elif op.tol is not None:
        assert float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1.0)) <= op.tol, what
    elif op.name == "sqdiff_sums" and dt == F32:
        np.testing.assert_allclose(got, ref, rtol=1e-5, err_msg=what)
    else:
        assert_same(got, ref.astype(got.dtype), what)


def test_dense_layout_equals_the_python_functions(dev):
    """Layout D is what the Python functions pass: their results equal the ABI calls on the D canvases."""
    import mie_b200 as M

    pairs = [("gaussian9", lambda x: M.gaussian_blur2d(x, 9, 1.0)),
             ("unsharp9", lambda x: M.unsharp_mask(x, 9, 1.0)),
             ("equalize", lambda x: M.equalize(x)),
             ("median3", lambda x: M.median_blur(x, 3))]
    for dt in (U16, U8, F32):
        for name, fn in pairs:
            shape = OP[name].shape
            x = rand(dt, shape, 7)
            x = torch.from_numpy(x.view(np.int16)).to(dev).view(torch.uint16) if dt == U16 else torch.from_numpy(x).to(dev)
            api = fn(x)
            api = api.view(torch.int16).cpu().numpy().view(np.uint16) if dt == U16 else api.cpu().numpy()
            assert_same(api.reshape(shape), reference(OP[name], dt, shape[0], dev), f"{name} {np.dtype(dt).name} Python API")
    x = torch.from_numpy(rand(U8, (2, 128, 128), 7)).to(dev)
    assert_same(M.equalize_clahe(x, 2.0, (4, 4)).cpu().numpy(), reference(OP["clahe"], U8, 2, dev), "clahe u8 API")


# ---------------------------------------------------------------------------------------------- which kernel ran
def test_profiler_sees_kernels(dev):
    """The dispatch assertions below are only evidence if kernel names are visible: must fail, never skip."""
    _, names = run(OP["gaussian9"], U16, "D", "D", dev, kernels=True)
    assert names, "torch.profiler reported no CUDA kernel for a dense 9-tap uint16 Gaussian"
    assert ran(names, "gauss_march_kernel"), names


# (op, dtypes, layout, kernels that must run, kernels that must not)
DISPATCH = [
    ("gaussian9", ALL, "P", ["gauss_march_kernel"], []),
    ("gaussian9", ALL, "T", ["gauss_march_kernel"], []),
    ("gaussian9", ALL, "U", ["gauss_tile_kernel"], ["gauss_march_kernel"]),
    ("gaussian5_symmetric", ALL, "U", ["gauss_tile_kernel"], ["gauss_march_kernel"]),
    ("gaussian11x7", ALL, "U", ["gauss_generic_kernel"], ["gauss_march_kernel", "gauss_tile_kernel"]),
    ("chain_march", ALL, "P", ["chain_a_march_kernel"], []),
    ("chain_march", ALL, "T", ["chain_a_march_kernel"], []),
    ("chain_march", ALL, "U", ["chain_a_kernel"], ["chain_a_march_kernel", "chain_a_fast_kernel"]),
    ("clahe", ALL, "P", ["clahe_lut_fast_kernel|clahe_lut_block_kernel", "clahe_apply_fast_kernel"], ["clahe_lut_kernel"]),
    ("clahe", ALL, "U", ["clahe_lut_kernel", "clahe_apply_kernel"], ["clahe_lut_fast_kernel", "clahe_lut_block_kernel",
                                                                     "clahe_apply_fast_kernel"]),
    ("median3", INTS, "P", ["median3x3_packed_kernel"], ["median2d_kernel"]),
    ("median3", (U8,), "H", ["median3x3_packed_kernel"], ["median2d_kernel"]),
    ("median3", (U16, I16), "H", ["median2d_kernel"], ["median3x3_packed_kernel"]),
    ("median3", ALL, "U", ["median2d_kernel"], ["median3x3_packed_kernel", "median3x3_f32_kernel"]),
    ("median3", (F32,), "P", ["median3x3_f32_kernel"], ["median2d_kernel"]),
    ("median3d", (U16, I16), "P", ["median3d_direct_kernel"], []),
    ("median3d", (U16, I16), "H", ["median3d_direct_kernel"], []),
    ("median3d", (U16, I16), "U", ["median3d_packed_kernel"], ["median3d_direct_kernel"]),
    ("median3d_halos", (U16, I16), "P", ["median3d_direct_kernel"], []),
    ("sqdiff_sums", INTS, "D", ["sqdiff_vec_kernel"], ["sqdiff_partial_kernel"]),
    ("sqdiff_sums", INTS, "U", ["sqdiff_partial_kernel"], ["sqdiff_vec_kernel"]),
    ("equalize", INTS, "D", ["equalize_fused_cluster_kernel"], []),
    ("equalize", INTS, "P", ["equalize_fused_cluster_kernel"], []),
    ("equalize", INTS, "T", ["equalize_fused_cluster_kernel"], []),
    ("equalize", ALL, "U", ["equalize_hist_kernel", "equalize_apply_kernel"], ["equalize_fused_cluster_kernel"]),
]
DISPATCH_CASES = [(o, dt, lay, yes, no) for o, dts, lay, yes, no in DISPATCH for dt in dts]


@pytest.mark.parametrize("name,dt,layout,yes,no", DISPATCH_CASES,
                         ids=[f"{o}-{np.dtype(d).name}-{lay}" for o, d, lay, _, _ in DISPATCH_CASES])
def test_layout_dispatch(dev, name, dt, layout, yes, no):
    op = OP[name]
    dst_layout = layout if not op.out_shape else "D"
    got, names = run(op, dt, layout, dst_layout, dev, kernels=True)
    assert names, "no kernel seen"
    for k in yes:
        assert any(ran(names, alt) for alt in k.split("|")), f"{name} {layout}: expected {k}, launched {names}"
    for k in no:
        assert not ran(names, k), f"{name} {layout}: {k} must not run, launched {names}"
    n = op.shape[0]
    assert_same(got, reference(op, dt, n, dev), f"{name} {np.dtype(dt).name} {layout}")


# ------------------------------------------------------------------------------------ plane offsets beyond 32 bits
# (the fused bilateral -> CLAHE needs CLAHE tiles of 32 pixels and more: not on 64 x 64 planes with its 4 x 4 grid)
G_OPS = ["gaussian9", "gaussian11x7", "unsharp_amount", "clahe_hist", "clahe", "clahe_opencv", "clahe16_luts",
         "equalize", "equalize_three_pass", "median3", "median5", "bilateral_exact", "nlm", "chain",
         "sk_equalize_adapthist", "sk_equalize_hist", "sk_denoise_bilateral", "gaussian3d", "sk_equalize_adapthist3d"]


@pytest.mark.parametrize("dt", [U8, U16], ids=["uint8", "uint16"])
def test_plane_offsets_beyond_32_bits(dev, dt):
    """Three planes 2^31 + 48 elements apart (a 4.3 / 8.6 GB canvas, filled once): the third plane starts beyond
    2^32 bytes, so 32-bit plane offsets land on the wrong pixels.  The destination uses the same layout."""
    shape2, shape3 = (3, 64, 64), (3, 4, 32, 32)
    src2 = Canvas(dev, dt, shape2, "G", "src")
    src2.write(rand(dt, shape2, 7))
    failures = []
    for name in G_OPS:
        op = OP[name]
        if dt not in op.dtypes:
            continue
        is3d = len(op.shape) == 4
        shape = shape3 if is3d else shape2
        src = None
        if is3d:
            src = Canvas(dev, dt, shape3, "G", "src")
            src.write(rand(dt, shape3, 7))
        try:
            # destinations wider than the source (float outputs) take P: a G layout of float64 would need 34 GB
            dst_layout = "G" if np.dtype(op.out_dtype(dt)).itemsize <= 2 else "P"
            got, _ = run(op, dt, "G", dst_layout, dev, shape=shape, src_canvas=src if is3d else src2)
            ref, _ = run(op, dt, "D", "D", dev, shape=shape)
            assert_same(got, ref, f"{name} G")
        except AssertionError as e:
            failures.append(str(e).splitlines()[0])
        del src
        torch.cuda.empty_cache()
    assert not failures, failures
