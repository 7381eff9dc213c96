"""Histogram equalisation operators with kornia's call signatures.

`equalize_clahe` mirrors kornia.enhance.equalize_clahe(input, clip_limit, grid_size,
slow_and_differentiable) and `equalize` mirrors kornia.enhance.equalize(input)
(kornia 0.8.2 — reference pyproject.toml:8, uv.lock:219-230; SURVEY.md §8(a) A1/A2,
§8(b)).  Both run hand-written sm_100a kernels through the C ABI (include/mie.h).

Extension over kornia: uint8 / uint16 / int16 tensors are accepted directly and
returned in the same dtype, using x01 = (v - lo) / (hi - lo) with (lo, hi) =
`value_range` (default: the dtype's full range) and rint(clamp(y,0,1)*(hi-lo))+lo
on the way out.  float32 tensors behave like kornia ([0,1] in, float out).
"""
from __future__ import annotations

import torch

from ._ffi import (CLAHE_KORNIA, CLAHE_OPENCV, DTYPE_CODE, as_planes, call, lib, new_out, plane_layout, require_cuda,
                   use_workspace, value_range_of)

__all__ = ["equalize_clahe", "equalize", "clahe_histograms", "clahe_luts", "clahe_apply", "clahe16_luts"]

# LUT memory the 65 536-bin mode keeps alive at a time (8 MB per 8x8-tile image).  Measured on the config-2 batch:
# 4 / 8 / 16 images per group = 3.22 / 2.70 / 2.54 ms — fewer, fuller launches win even though 128 MB of LUTs
# no longer fit the 126 MB L2 entirely.
CLAHE16_WORKSPACE_BYTES = 512 << 20

_SEMANTICS = {"kornia": CLAHE_KORNIA, "opencv": CLAHE_OPENCV}


def _check_clahe_args(clip_limit, grid_size):
    # same checks, same exception types as kornia.enhance.equalize_clahe
    if not isinstance(clip_limit, float):
        raise TypeError(f"Input clip_limit type is not float. Got {type(clip_limit)}")
    if not isinstance(grid_size, tuple):
        raise TypeError(f"Input grid_size type is not Tuple. Got {type(grid_size)}")
    if len(grid_size) != 2:
        raise TypeError(f"Input grid_size is not a Tuple with 2 elements. Got {len(grid_size)}")
    if isinstance(grid_size[0], float) or isinstance(grid_size[1], float):
        raise TypeError("Input grid_size type is not valid, must be a Tuple[int, int].")
    if grid_size[0] <= 0 or grid_size[1] <= 0:
        raise ValueError(f"Input grid_size elements must be positive. Got {grid_size}")


def equalize_clahe(input: torch.Tensor, clip_limit: float = 40.0, grid_size: tuple = (8, 8),
                   slow_and_differentiable: bool = False, *, value_range=None, semantics: str = "kornia",
                   out_dtype=None) -> torch.Tensor:
    """Contrast-limited adaptive histogram equalisation.

    Shapes (H,W), (C,H,W), (B,C,H,W); the result has the input's shape.
    semantics='kornia': 256 bins on [0,1] data (kornia.enhance.equalize_clahe).
    semantics='opencv': cv2.createCLAHE(clip_limit, (grid_size[1], grid_size[0])).apply, bit for bit —
    256 bins for uint8 tensors, 65 536 bins for uint16 tensors (no quantisation of 12/16-bit data).
    """
    _check_clahe_args(clip_limit, grid_size)
    if slow_and_differentiable:
        raise NotImplementedError("the CUDA kernels are not differentiable (slow_and_differentiable=True)")
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    gh, gw = int(grid_size[0]), int(grid_size[1])
    L = lib()
    if semantics == "opencv" and x.dtype == torch.uint16:
        per_image = L.mie_clahe16_lut_bytes(gh, gw)
        ws_bytes = per_image * max(1, min(n, CLAHE16_WORKSPACE_BYTES // max(per_image, 1))) + 256   # + the value bound
    else:
        ws_bytes = L.mie_clahe_workspace_bytes(n, h, w, gh, gw)
    ws = use_workspace(x.device, ws_bytes)
    call(x.device, "mie_clahe", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), gh, gw, float(clip_limit), _SEMANTICS[semantics], lo, hi, ws.data_ptr(), ws.numel())
    return dst


def clahe_histograms(input: torch.Tensor, grid_size=(8, 8), *, value_range=None, semantics="kornia") -> torch.Tensor:
    """Stage output: raw per-tile histograms, int32 (*, gh, gw, 256)."""
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    gh, gw = int(grid_size[0]), int(grid_size[1])
    hist = torch.empty(x.shape[:-2] + (gh, gw, 256), dtype=torch.int32, device=x.device)
    call(x.device, "mie_clahe_hist", x.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(n, h, w)[:5], gh, gw,
         _SEMANTICS[semantics], lo, hi, hist.data_ptr())
    return hist


def clahe_luts(input: torch.Tensor, clip_limit: float = 40.0, grid_size=(8, 8), *, value_range=None,
               semantics="kornia") -> torch.Tensor:
    """Stage output: clipped / redistributed / cumulated LUTs, uint8 (*, gh, gw, 256)."""
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    gh, gw = int(grid_size[0]), int(grid_size[1])
    luts = torch.empty(x.shape[:-2] + (gh, gw, 256), dtype=torch.uint8, device=x.device)
    call(x.device, "mie_clahe_luts", x.data_ptr(), DTYPE_CODE[x.dtype], *plane_layout(n, h, w)[:5], gh, gw,
         float(clip_limit), _SEMANTICS[semantics], lo, hi, luts.data_ptr())
    return luts


def clahe16_luts(input: torch.Tensor, clip_limit: float = 40.0, grid_size=(8, 8)) -> torch.Tensor:
    """Stage output of the 65 536-bin OpenCV mode: uint16 LUTs (*, gh, gw, 65536) of a uint16 tensor."""
    require_cuda(input)
    x, n, h, w = as_planes(input)
    if x.dtype != torch.uint16:
        raise TypeError("clahe16_luts takes uint16 tensors")
    gh, gw = int(grid_size[0]), int(grid_size[1])
    luts = torch.empty(x.shape[:-2] + (gh, gw, 65536), dtype=torch.uint16, device=x.device)
    call(x.device, "mie_clahe16_luts", x.data_ptr(), *plane_layout(n, h, w)[:5], gh, gw, float(clip_limit),
         luts.data_ptr())
    return luts


def clahe_apply(input: torch.Tensor, luts: torch.Tensor, grid_size=(8, 8), *, value_range=None, semantics="kornia",
                out_dtype=None) -> torch.Tensor:
    """Stage: interpolation pass with caller-supplied LUTs (teacher forcing in the parity tests)."""
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    gh, gw = int(grid_size[0]), int(grid_size[1])
    luts = luts.contiguous()
    if luts.dtype != torch.uint8 or luts.numel() != n * gh * gw * 256 or luts.device != x.device:
        raise ValueError("luts must be a uint8 tensor of n*gh*gw*256 entries on the input's device")
    dst = new_out(x, out_dtype)
    call(x.device, "mie_clahe_apply", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), gh, gw, _SEMANTICS[semantics], lo, hi, luts.data_ptr())
    return dst


def equalize(input: torch.Tensor, *, value_range=None, out_dtype=None) -> torch.Tensor:
    """Global histogram equalisation (kornia.enhance.equalize / torchvision rule), per plane."""
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    dst = new_out(x, out_dtype)
    ws = use_workspace(x.device, lib().mie_equalize_workspace_bytes(n))
    call(x.device, "mie_equalize", x.data_ptr(), dst.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[dst.dtype],
         *plane_layout(n, h, w), lo, hi, ws.data_ptr(), ws.numel())
    return dst
