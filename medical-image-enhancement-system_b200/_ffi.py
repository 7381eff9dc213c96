"""ctypes binding of libmie_b200.so (C ABI declared in include/mie.h).

There is deliberately no fallback: if the CUDA library has not been built
(`python __graft_entry__.py` / `_build.build_extension()`), importing any operator
raises.  PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# MIE_B200_LIB: path of an alternative BUILD of the same library (kernel-development A/B runs under benchmarks/dev);
# it selects a file, not a code path — every build exports the same ABI and has no fallback either.
LIB_PATH = os.environ.get("MIE_B200_LIB") or os.path.join(PKG_DIR, "libmie_b200.so")

MIE_U8, MIE_U16, MIE_I16, MIE_F32, MIE_F64 = 0, 1, 2, 3, 4
BORDER = {"constant": 0, "reflect": 1, "replicate": 2, "circular": 3, "symmetric": 4}
# scipy.ndimage / scikit-image mode names -> BORDER names
SCIPY_MODES = {"nearest": "replicate", "reflect": "symmetric", "mirror": "reflect", "constant": "constant",
               "wrap": "circular"}
CLAHE_KORNIA, CLAHE_OPENCV = 0, 1

DTYPE_CODE = {torch.uint8: MIE_U8, torch.uint16: MIE_U16, torch.int16: MIE_I16, torch.float32: MIE_F32}
DTYPE_RANGE = {torch.uint8: (0.0, 255.0), torch.uint16: (0.0, 65535.0), torch.int16: (-32768.0, 32767.0)}

_E_TYPE = {-2}  # -> TypeError
_E_VALUE = {-1, -3, -4, -5, -6, -7, -8, -9, -10, -12}  # -> ValueError

_p, _i, _i64, _f, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t
_planes = [_i64, _i, _i, _i64, _i64, _i64, _i64]  # n, h, w, ssn, ssh, dsn, dsh
_volumes = [_i64, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i64]  # n, d, h, w, ssn, ssd, ssh, dsn, dsd, dsh
_taps = [_p, _i, _p, _i]

SIGNATURES = {
    "mie_abi_version": ([], _i),
    "mie_set_kernel_policy": ([C.c_uint], _i),
    "mie_get_kernel_policy": ([], C.c_uint),
    "mie_error_string": ([_i], C.c_char_p),
    "mie_device_info": ([C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)], _i),
    "mie_gaussian2d": ([_p, _p, _i, _i, *_planes, *_taps, _i, _f, _f, _p], _i),
    "mie_unsharp": ([_p, _p, _i, _i, *_planes, *_taps, _i, _f, _f, _p], _i),
    "mie_unsharp_amount": ([_p, _p, _i, _i, *_planes, *_taps, _i, _f, _i, _f, _f, _p], _i),
    "mie_gaussian3d": ([_p, _p, _i, _i, *_volumes, *_taps, *_taps[:2], _i, _f, _f, _p], _i),
    "mie_unsharp3d": ([_p, _p, _i, _i, *_volumes, *_taps, *_taps[:2], _i, _f, _i, _f, _f, _p], _i),
    "mie_clahe_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_clahe_hist": ([_p, _i, _i64, _i, _i, _i64, _i64, _i, _i, _i, _f, _f, _p, _p], _i),
    "mie_clahe_luts": ([_p, _i, _i64, _i, _i, _i64, _i64, _i, _i, _d, _i, _f, _f, _p, _p], _i),
    "mie_clahe_apply": ([_p, _p, _i, _i, *_planes, _i, _i, _i, _f, _f, _p, _p], _i),
    "mie_clahe": ([_p, _p, _i, _i, *_planes, _i, _i, _d, _i, _f, _f, _p, _sz, _p], _i),
    "mie_clahe16_lut_bytes": ([_i, _i], _sz),
    "mie_clahe16_luts": ([_p, _i64, _i, _i, _i64, _i64, _i, _i, _d, _p, _p], _i),
    "mie_equalize_workspace_bytes": ([_i64], _sz),
    "mie_equalize": ([_p, _p, _i, _i, *_planes, _f, _f, _p, _sz, _p], _i),
    "mie_median2d": ([_p, _p, _i, *_planes, _i, _i, _i, _p], _i),
    "mie_median3d": ([_p, _p, _i, _i, _i, _i, _i64, _i64, _i64, _i64, _p, _p, _i, _p], _i),
    "mie_sk_median": ([_p, _p, _i, *_planes, _p, _i, _i, _i, _d, _p], _i),
    "mie_sk_median3d": ([_p, _p, _i, *_volumes, _p, _i, _i, _i, _i, _d, _p], _i),
    "mie_bilateral": ([_p, _p, _i, _i, *_planes, _p, _i, _i, _f, _i, _f, _f, _p], _i),
    "mie_nlm": ([_p, _p, _i, _i, *_planes, _i, _i, _f, _f, _f, _f, _p], _i),
    "mie_nlm_slow": ([_p, _p, _i, _i, *_planes, _i, _i, _d, _d, _f, _f, _p], _i),
    "mie_metric_workspace_bytes": ([_i64, _i, _i, _i], _sz),
    "mie_sqdiff_sums": ([_p, _p, _i, *_planes, _p, _p, _sz, _p], _i),
    "mie_ssim_sums": ([_p, _p, _i, *_planes, _i, _d, _d, _p, _p, _sz, _p], _i),
    "mie_bilateral_clahe_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_bilateral_clahe_is_fused": ([_i] * 6, _i),
    "mie_bilateral_clahe": ([_p, _p, _i, _i, *_planes, _p, _i, _f, _i, _i, _i, _d, _f, _f, _i, _p, _sz, _p], _i),
    "mie_sk_adapthist_workspace_bytes": ([_i64, _i, _i, _i, _i, _i], _sz),
    "mie_sk_equalize_adapthist": ([_p, _p, _i, _i, *_planes, _i, _i, _d, _i, _p, _sz, _p], _i),
    "mie_sk_adapthist3d_workspace_bytes": ([_i64, _i, _i, _i, _i, _i, _i, _i], _sz),
    "mie_sk_equalize_adapthist3d": ([_p, _p, _i, _i, *_volumes, _i, _i, _i, _d, _i, _p, _sz, _p], _i),
    "mie_sk_equalize_hist_workspace_bytes": ([_i64, _i], _sz),
    "mie_sk_equalize_hist": ([_p, _p, _i, _i, *_planes, _p, _sz, _p], _i),
    "mie_sk_denoise_bilateral": ([_p, _p, _i, _i, *_planes, _i, _i, _i, _d, _p, _p, _p, _p], _i),
    "mie_sk_tv_chambolle_workspace_bytes": ([_i64, _i, _i, _i], _sz),
    "mie_sk_tv_chambolle3d_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_sk_denoise_tv_chambolle": ([_p, _p, _i, _i, *_planes, _d, _d, _i, _p, _p, _sz, _p], _i),
    "mie_sk_denoise_tv_chambolle3d": ([_p, _p, _i, _i, *_volumes, _d, _d, _i, _p, _p, _sz, _p], _i),
    "mie_sk_structural_similarity_workspace_bytes": ([_i64, _i, _i, _i], _sz),
    "mie_sk_structural_similarity3d_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_sk_structural_similarity": (
        [_p, _p, _p, _i, _i, *_planes, _i64, _i64, _i, _p, _i, _d, _d, _d, _p, _p, _sz, _p], _i),
    "mie_sk_structural_similarity3d": (
        [_p, _p, _p, _i, _i, *_volumes, _i64, _i64, _i64, _i, _p, _i, _d, _d, _d, _p, _p, _sz, _p], _i),
    "mie_sk_ridge_filter_workspace_bytes": ([_i64, _i, _i, _i], _sz),
    "mie_sk_ridge_filter3d_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_sk_ridge_filter": (
        [_p, _p, _i, _i, *_planes, _i, _i, _p, _p, _p, _p, _i, _d, _i, _d, _d, _d, _p, _sz, _p], _i),
    "mie_sk_ridge_filter3d": (
        [_p, _p, _i, _i, *_volumes, _i, _i, _p, _p, _p, _p, _i, _d, _i, _d, _d, _d, _p, _sz, _p], _i),
    "mie_sk_hessian_matrix_workspace_bytes": ([_i64, _i, _i, _i], _sz),
    "mie_sk_hessian_matrix3d_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_sk_hessian_matrix": ([_p, _p, _i, _i, *_planes, _i64, _i, _p, _p, _i, _d, _p, _sz, _p], _i),
    "mie_sk_hessian_matrix3d": ([_p, _p, _i, _i, *_volumes, _i64, _i, _p, _p, _i, _d, _p, _sz, _p], _i),
    "mie_sk_hessian_eigvals": ([_p, _p, _i, _i, _i64, _i64, _i64, _p], _i),
    "mie_halo_exchange_available": ([], _i),
    "mie_halo_exchange_z": ([_p, _i, _i, _p, _p, _p, _p, _sz, _p], _i),
    "mie_enable_peer_access": ([_i], _i),
    "mie_ipc_export": ([_p, _p, C.POINTER(_i64)], _i),
    "mie_ipc_open": ([_p, C.POINTER(_p)], _i),
    "mie_ipc_close": ([_p], _i),
    "mie_chain_workspace_bytes": ([_i64, _i, _i, _i, _i], _sz),
    "mie_chain_gauss_clahe_unsharp": (
        [_p, _p, _i, _i, *_planes, *_taps, _i, _i, _d, *_taps, _i, _f, _f, _i, _p, _sz, _p], _i),
    "mie_chain_is_fused": ([_i] * 8, _i),
    "mie_value_range_mode": ([_i, _f, _f], _i),
}

_lib = None


def lib() -> C.CDLL:
    """Load the library (once).  Raises if it has not been built — no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build the sm_100a extension first "
                "(python -c 'import __graft_entry__ as g; g.build()'); there is no CPU or PyTorch fallback")
        handle = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the build is stale
            fn.argtypes, fn.restype = argtypes, restype
        if handle.mie_abi_version() != 1:
            raise RuntimeError("libmie_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = lib().mie_error_string(rc).decode()
    if rc in _E_TYPE:
        raise TypeError(msg)
    if rc in _E_VALUE:
        raise ValueError(msg)
    if rc == -11:
        raise NotImplementedError(msg)
    raise RuntimeError(f"CUDA error {rc}: {msg}")


POLICY = {"generic_gauss": 1, "generic_clahe": 2, "clahe_float_rules": 4, "generic_equalize": 8,
          "equalize_float_rules": 16, "generic_median": 32, "generic_bilateral": 64, "generic_nlm": 128,
          "clahe16_no_cluster": 256, "clahe16_two_sweep": 512, "equalize_three_pass": 1024,
          "bilateral_exact_exp": 2048, "clahe16_full_luts": 4096, "equalize_slab": 8192}


class kernel_policy:
    """Context manager around mie_set_kernel_policy (include/mie.h): force the generic kernel of the named
    operators inside the block — a verification hook for tests, e.g. `with kernel_policy("generic_median"): ...`."""

    def __init__(self, *names: str):
        self.mask = 0
        for n in names:
            self.mask |= POLICY[n]

    def __enter__(self):
        self.prev = lib().mie_get_kernel_policy()
        check(lib().mie_set_kernel_policy(self.prev | self.mask))
        return self

    def __exit__(self, *exc):
        check(lib().mie_set_kernel_policy(self.prev))
        return False


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def call(device: torch.device, name: str, *args) -> None:
    """Enqueue ABI entry point `name` on `device`'s current stream: every entry point that launches work takes its
    stream as the last argument.  A non-zero return code raises (see check)."""
    with torch.cuda.device(device):
        check(getattr(lib(), name)(*args, stream_ptr(device)))


def require_cuda(t: torch.Tensor, name: str = "input") -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: this package has no CPU path")
    if t.dtype not in DTYPE_CODE:
        raise TypeError(f"{name} dtype {t.dtype} not supported (uint8, uint16, int16, float32)")


def value_range_of(t: torch.Tensor, value_range):
    """(lo, hi) used by x01 = (v - lo) / (hi - lo); ignored for float tensors."""
    if t.dtype == torch.float32:
        return 0.0, 1.0
    if value_range is None:
        return DTYPE_RANGE[t.dtype]
    lo, hi = float(value_range[0]), float(value_range[1])
    if not hi > lo:
        raise ValueError("value_range must satisfy hi > lo")
    return lo, hi


def value_range_mode(dtype: torch.dtype, value_range=None) -> str:
    """Which kernels a pixel mapping runs on (host-only query, mie_value_range_mode in include/mie.h):
    'default' — the dtype's own range (or float pixels); 'window' — an integer window the tuned kernels run through
    their divide-free conversion, checked on the host against the IEEE quotient for every code of the dtype;
    'generic' — anything else (the generic kernels compute the mapping with the IEEE division)."""
    if dtype not in DTYPE_CODE:
        raise TypeError(f"dtype {dtype} not supported (uint8, uint16, int16, float32)")
    if dtype == torch.float32 or value_range is None:
        lo, hi = DTYPE_RANGE.get(dtype, (0.0, 1.0))
    else:
        lo, hi = float(value_range[0]), float(value_range[1])
        if not hi > lo:
            raise ValueError("value_range must satisfy hi > lo")
    return {0: "default", 1: "window", -1: "generic"}[lib().mie_value_range_mode(DTYPE_CODE[dtype], lo, hi)]


def as_planes(t: torch.Tensor):
    """(H,W) | (C,H,W) | (B,C,H,W) -> dense tensor + (n, h, w); kornia's
    perform_keep_shape_image contract."""
    if t.dim() < 2 or t.dim() > 4:
        raise ValueError(f"expected (H,W), (C,H,W) or (B,C,H,W); got shape {tuple(t.shape)}")
    t = t.contiguous()
    h, w = t.shape[-2:]
    n = t.numel() // (h * w) if h * w else 0
    return t, n, h, w


def as_volumes(t):
    """(D,H,W) | (B,D,H,W) | (B,C,D,H,W) -> dense tensor + (n, d, h, w): every (D, H, W) volume is one 3-D image, as
    skimage treats a 3-D array.  Checks the argument only: the caller checks the device and dtype (require_cuda)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"input must be a torch.Tensor, got {type(t)}")
    if not 3 <= t.dim() <= 5:
        raise ValueError(f"volumetric=True expects (D,H,W), (B,D,H,W) or (B,C,D,H,W); got shape {tuple(t.shape)}")
    t = t.contiguous()
    d, h, w = (int(s) for s in t.shape[-3:])
    n = t.numel() // (d * h * w) if d * h * w else 0
    return t, n, d, h, w


def plane_layout(n: int, h: int, w: int) -> tuple:
    """The `_planes` arguments of n dense (h, w) planes, the destination in the source's layout.  Entry points that
    read a source only take the first five."""
    return n, h, w, h * w, w, h * w, w


def volume_layout(n: int, d: int, h: int, w: int) -> tuple:
    """The `_volumes` arguments of n dense (d, h, w) volumes, the destination in the source's layout."""
    return n, d, h, w, d * h * w, h * w, w, d * h * w, h * w, w


def _dtype_names(dtypes) -> str:
    return " or ".join(str(dt) for dt in dict.fromkeys(dtypes))


def new_out(x: torch.Tensor, out_dtype, allowed=None, default=None) -> torch.Tensor:
    """Output of `x`'s shape on its device in `out_dtype` (None: `default`, itself defaulting to x's dtype), which
    must be one of `allowed` (default: x's dtype or float32, the rule of the kornia-signature operators)."""
    allowed = (x.dtype, torch.float32) if allowed is None else allowed
    dt = (x.dtype if default is None else default) if out_dtype is None else out_dtype
    if dt not in allowed:
        raise TypeError(f"out_dtype must be {_dtype_names(allowed)}")
    return torch.empty(x.shape, dtype=dt, device=x.device)


def check_out(x: torch.Tensor, out: torch.Tensor, allowed=None) -> torch.Tensor:
    """A caller's output for `x`: contiguous, of x's shape, on x's device, dtype one of `allowed` (as in new_out)."""
    allowed = (x.dtype, torch.float32) if allowed is None else allowed
    if out.shape != x.shape or not out.is_contiguous() or out.device != x.device or out.dtype not in allowed:
        raise ValueError(f"out must be a contiguous tensor of the input's shape on its device, dtype "
                         f"{_dtype_names(allowed)}")
    return out


def use_workspace(device: torch.device, nbytes: int, workspace: torch.Tensor = None) -> torch.Tensor:
    """The uint8 scratch memory of a call that needs `nbytes`: a fresh buffer, or the caller's `workspace` after
    checking it.  The kernels use `nbytes` dense bytes from its first byte, store 32-bit words and load 16-byte
    pieces (MIE_E_ALIGN), so a caller's buffer must be contiguous and 256-byte aligned like a fresh allocation."""
    if workspace is None:
        return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
    if workspace.dtype != torch.uint8 or not workspace.is_contiguous() or workspace.numel() < nbytes or \
            workspace.device != device or workspace.data_ptr() % 256:
        raise ValueError(f"workspace must be a contiguous, 256-byte aligned uint8 tensor of >= {nbytes} bytes on the "
                         "input's device (a fresh torch.empty is; a sliced view such as ws[1:] is not)")
    return workspace
