"""Full-reference quality metrics with sewar's call signatures, computed on the GPU.

`mse`, `rmse`, `psnr`, `ssim` mirror sewar.full_ref (sewar 0.4.6 — reference pyproject.toml:13,
uv.lock:692-700; SURVEY.md §8(f) F4): the evaluation step that follows the enhancement path.  sewar takes
(H, W) or (H, W, C) numpy arrays and averages over channels; here the inputs are CUDA tensors
(H, W) / (C, H, W) / (B, C, H, W) and every leading plane plays the role of a channel.  `per_plane=True`
returns the per-plane values as a float64 CPU tensor instead of their mean (batched evaluation).

The sums run in hand-written sm_100a kernels (csrc/metrics.cu) on the RAW pixel values — exact 64-bit
integer sums for integer tensors — and only the final scalar arithmetic (divide, sqrt, log10) is done
on the host in float64, exactly as numpy would.
"""
from __future__ import annotations

import numpy as np
import torch

from ._ffi import DTYPE_CODE, as_planes, call, lib, plane_layout, require_cuda, use_workspace

__all__ = ["mse", "rmse", "psnr", "ssim", "mae"]

_INT_MAX = {torch.uint8: 255, torch.uint16: 65535, torch.int16: 32767}


def _initial_check(GT: torch.Tensor, P: torch.Tensor):
    # sewar._initial_check: same shape, same dtype
    require_cuda(GT, "GT")
    require_cuda(P, "P")
    if GT.shape != P.shape:
        raise AssertionError(f"Supplied images have different sizes {tuple(GT.shape)} and {tuple(P.shape)}")
    if GT.dtype != P.dtype:
        raise AssertionError(f"Supplied images have different dtypes {GT.dtype} and {P.dtype}")
    if GT.device != P.device:
        raise ValueError("GT and P must live on the same device")
    a, n, h, w = as_planes(GT)
    b, _, _, _ = as_planes(P)
    return a, b, n, h, w


def _max_of(t: torch.Tensor, MAX):
    if MAX is not None:
        return float(MAX)
    if t.dtype not in _INT_MAX:
        raise ValueError("MAX must be given for float tensors (sewar uses np.iinfo(GT.dtype).max)")
    return float(_INT_MAX[t.dtype])


def _sqdiff_sums(GT, P) -> tuple[np.ndarray, int]:
    a, b, n, h, w = _initial_check(GT, P)
    out = torch.empty((max(n, 1), 2), dtype=torch.float64, device=a.device)
    ws = use_workspace(a.device, lib().mie_metric_workspace_bytes(n, h, w, 0))
    call(a.device, "mie_sqdiff_sums", a.data_ptr(), b.data_ptr(), DTYPE_CODE[a.dtype], *plane_layout(n, h, w),
         out.data_ptr(), ws.data_ptr(), ws.numel())
    return out[:n].cpu().numpy(), h * w


def _reduce(values: np.ndarray, per_plane: bool):
    if per_plane:
        return torch.from_numpy(np.ascontiguousarray(values))
    return float(np.mean(values)) if values.size else float("nan")


def mse(GT: torch.Tensor, P: torch.Tensor, *, per_plane: bool = False):
    """sewar.mse: mean squared error."""
    sums, px = _sqdiff_sums(GT, P)
    return _reduce(sums[:, 0] / px, per_plane)


def mae(GT: torch.Tensor, P: torch.Tensor, *, per_plane: bool = False):
    """Mean absolute error (same reduction kernel; not in sewar)."""
    sums, px = _sqdiff_sums(GT, P)
    return _reduce(sums[:, 1] / px, per_plane)


def rmse(GT: torch.Tensor, P: torch.Tensor, *, per_plane: bool = False):
    """sewar.rmse: sqrt(mse) (of the whole image; per plane with per_plane=True)."""
    sums, px = _sqdiff_sums(GT, P)
    if per_plane:
        return torch.from_numpy(np.sqrt(sums[:, 0] / px))
    return float(np.sqrt(np.mean(sums[:, 0] / px)))


def psnr(GT: torch.Tensor, P: torch.Tensor, MAX=None, *, per_plane: bool = False):
    """sewar.psnr: 10 log10(MAX^2 / mse), inf for identical images; MAX defaults to the dtype maximum."""
    mx = _max_of(GT, MAX)
    sums, px = _sqdiff_sums(GT, P)
    m = sums[:, 0] / px
    if not per_plane:
        m = np.array([np.mean(m)])
    with np.errstate(divide="ignore"):
        v = np.where(m == 0.0, np.inf, 10.0 * np.log10(mx ** 2 / np.where(m == 0.0, 1.0, m)))
    return torch.from_numpy(v) if per_plane else float(v[0])


def ssim(GT: torch.Tensor, P: torch.Tensor, ws: int = 11, K1: float = 0.01, K2: float = 0.03, MAX=None,
         fltr_specs=None, mode: str = "valid", *, per_plane: bool = False):
    """sewar.ssim: (ssim, cs) with sewar's default uniform ws x ws window in 'valid' mode.
    Other filters (fltr_specs) and modes are not implemented."""
    if fltr_specs is not None:
        raise NotImplementedError("only sewar's default uniform window (fltr_specs=None) is implemented")
    if mode != "valid":
        raise NotImplementedError("only mode='valid' (sewar's default) is implemented")
    mx = _max_of(GT, MAX)
    a, b, n, h, w = _initial_check(GT, P)
    ws = int(ws)
    if ws < 1 or ws > min(h, w):
        raise ValueError(f"window size {ws} does not fit a {h}x{w} image")
    c1, c2 = (K1 * mx) ** 2, (K2 * mx) ** 2
    out = torch.empty((max(n, 1), 2), dtype=torch.float64, device=a.device)
    wsb = use_workspace(a.device, lib().mie_metric_workspace_bytes(n, h, w, ws))
    call(a.device, "mie_ssim_sums", a.data_ptr(), b.data_ptr(), DTYPE_CODE[a.dtype], *plane_layout(n, h, w), ws,
         float(c1), float(c2), out.data_ptr(), wsb.data_ptr(), wsb.numel())
    vals = out[:n].cpu().numpy() / float((h - ws + 1) * (w - ws + 1))
    if per_plane:
        return torch.from_numpy(np.ascontiguousarray(vals[:, 0])), torch.from_numpy(np.ascontiguousarray(vals[:, 1]))
    return float(np.mean(vals[:, 0])), float(np.mean(vals[:, 1]))
