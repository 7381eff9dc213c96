"""Fused enhancement chain: Gaussian denoise -> CLAHE -> unsharp mask
(BASELINE.json config 2; SURVEY.md §7.3 `chain_gcu`).

Equivalent, bit for bit, to
    unsharp_mask(equalize_clahe(gaussian_blur2d(x01, ...), ...), ...)
evaluated on fp32 [0,1] data and quantised once at the end, but executed in two
kernel launches with one byte per pixel of intermediate traffic.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from ._ffi import (DTYPE_CODE, as_planes, call, check_out, lib, new_out, plane_layout, require_cuda, use_workspace,
                   value_range_of)
from .enhance import _check_clahe_args
from .filters import _border, _check_kernel, _pair_float, _pair_int, get_gaussian_kernel1d

__all__ = ["ChainConfig", "ChainPlan", "ChainRing", "enhance_chain", "chain_workspace_bytes", "bilateral_clahe",
           "BilateralClahePlan", "bilateral_clahe_workspace_bytes"]


@dataclass(frozen=True)
class ChainConfig:
    """Keyword names follow the kornia functions each stage replaces."""
    denoise_kernel_size: object = 9          # gaussian_blur2d(kernel_size=)
    denoise_sigma: object = 1.0              # gaussian_blur2d(sigma=)
    clip_limit: float = 2.0                  # equalize_clahe(clip_limit=)
    grid_size: tuple = (8, 8)                # equalize_clahe(grid_size=)
    sharpen_kernel_size: object = 9          # unsharp_mask(kernel_size=)
    sharpen_sigma: object = 1.0              # unsharp_mask(sigma=)
    border_type: str = "reflect"
    value_range: object = None               # (lo, hi) for integer tensors; None = dtype range


def chain_workspace_bytes(n: int, h: int, w: int, grid_size=(8, 8)) -> int:
    return int(lib().mie_chain_workspace_bytes(n, h, w, int(grid_size[0]), int(grid_size[1])))


def enhance_chain(input: torch.Tensor, config: ChainConfig = ChainConfig(), *, out: torch.Tensor = None,
                  out_dtype=None, workspace: torch.Tensor = None, stages: int = 3) -> torch.Tensor:
    """Run the chain on (H,W) / (C,H,W) / (B,C,H,W) planes resident on the GPU.

    `out` and `workspace` (uint8, >= chain_workspace_bytes) may be supplied so that a
    steady-state loop allocates nothing.  `stages` (1 = first launch, 2 = second launch, 3 = both) exists
    for per-kernel timing in bench.py; leave it at 3.
    """
    cfg = config
    _check_clahe_args(cfg.clip_limit, cfg.grid_size)
    gky, gkx = _pair_int(cfg.denoise_kernel_size, "denoise_kernel_size")
    uky, ukx = _pair_int(cfg.sharpen_kernel_size, "sharpen_kernel_size")
    _check_kernel(gky, gkx)
    _check_kernel(uky, ukx)
    gsy, gsx = _pair_float(cfg.denoise_sigma, "denoise_sigma")
    usy, usx = _pair_float(cfg.sharpen_sigma, "sharpen_sigma")
    _border(cfg.border_type)
    require_cuda(input)
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, cfg.value_range)
    out = new_out(x, out_dtype) if out is None else check_out(x, out)
    gh, gw = int(cfg.grid_size[0]), int(cfg.grid_size[1])
    workspace = use_workspace(x.device, lib().mie_chain_workspace_bytes(n, h, w, gh, gw), workspace)
    wgx, wgy = get_gaussian_kernel1d(gkx, gsx), get_gaussian_kernel1d(gky, gsy)
    wux, wuy = get_gaussian_kernel1d(ukx, usx), get_gaussian_kernel1d(uky, usy)
    call(x.device, "mie_chain_gauss_clahe_unsharp", x.data_ptr(), out.data_ptr(), DTYPE_CODE[x.dtype],
         DTYPE_CODE[out.dtype], *plane_layout(n, h, w), wgx.ctypes.data, gkx, wgy.ctypes.data, gky, gh, gw,
         float(cfg.clip_limit), wux.ctypes.data, ukx, wuy.ctypes.data, uky, _border(cfg.border_type), lo, hi,
         int(stages), workspace.data_ptr(), workspace.numel())
    return out


class ChainPlan:
    """The chain on FIXED device buffers, captured once into a CUDA graph.

    A steady-state loop (same input / output tensors every step, e.g. the slots of the host pipeline's
    ring) then costs one graph launch per step instead of three kernel launches plus the Python argument
    checks, which matters because the whole config-2 step is ~0.2 ms.  `replay()` enqueues the graph on
    the current stream; `input` is read and `out` is written in place each time.
    """

    def __init__(self, input: torch.Tensor, config: ChainConfig = ChainConfig(), *, out: torch.Tensor = None,
                 out_dtype=None, workspace: torch.Tensor = None, stages: int = 3, graph: bool = True):
        require_cuda(input)
        self.input = input
        self.config = config
        self.stages = int(stages)
        x, n, h, w = as_planes(input)
        if out is None:
            dt = x.dtype if out_dtype is None else out_dtype
            out = torch.empty(input.shape, dtype=dt, device=input.device)
        self.out = out
        gh, gw = int(config.grid_size[0]), int(config.grid_size[1])
        # a stage-2-only plan must be given the workspace its stage-1 twin filled
        self.workspace = use_workspace(input.device, chain_workspace_bytes(n, h, w, (gh, gw)), workspace)
        self._graph = None
        self._direct()  # validates the arguments and performs the one-time kernel attribute setup
        if graph and n > 0:
            torch.cuda.synchronize(input.device)
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream(device=input.device)
            with torch.cuda.stream(side):
                with torch.cuda.graph(g, stream=side):
                    self._direct()
            self._graph = g

    def _direct(self):
        enhance_chain(self.input, self.config, out=self.out.view(self.input.shape) if self.out.shape != self.input.shape
                      else self.out, workspace=self.workspace, stages=self.stages)

    def replay(self) -> torch.Tensor:
        if self._graph is not None:
            self._graph.replay()
        else:
            self._direct()
        return self.out


class ChainRing:
    """Steady-state throughput over many independent batches.

    One config-2 step is three launches whose block counts are not multiples of what the GPU holds at once
    (2 048 bands are 2.8 waves of chain_a blocks and 3.5 waves of chain_b blocks), so the last, partial wave of
    each kernel leaves SMs idle: 8 % / 13 % of the kernels' time.  A ring of independent ChainPlans (own input,
    output and workspace — e.g. the slots of a loader's buffer ring) replayed round-robin on their own streams
    lets the next batch's chain_a fill the SMs that the previous batch's chain_b tail no longer uses:
    0.204 -> 0.189 ms per 256-slice batch with two plans (benchmarks/two_stream_probe.py).

        ring = ChainRing([x0, x1])          # two batches in flight
        ring.begin()
        for k in range(steps):
            ring.replay(k)                  # batch k % 2: fill ring.plans[k % 2].input first in a real loop
        ring.join()                         # the caller's stream now waits for everything enqueued
    """

    def __init__(self, inputs, config: ChainConfig = ChainConfig(), *, outs=None, out_dtype=None):
        if len(inputs) < 1:
            raise ValueError("ChainRing needs at least one input batch")
        self.device = inputs[0].device
        outs = outs if outs is not None else [None] * len(inputs)
        self.plans = [ChainPlan(x, config, out=o, out_dtype=out_dtype) for x, o in zip(inputs, outs)]
        with torch.cuda.device(self.device):
            self.streams = [torch.cuda.Stream(device=self.device) for _ in self.plans]

    def begin(self) -> None:
        """Order the ring's streams after everything already enqueued on the caller's current stream."""
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            s.wait_stream(cur)

    def replay(self, k: int) -> torch.Tensor:
        """Enqueue the chain of slot k % len(plans) on that slot's stream; returns its output tensor (valid once
        the slot's stream — or, after join(), the caller's stream — reaches this point)."""
        i = k % len(self.plans)
        with torch.cuda.stream(self.streams[i]):
            return self.plans[i].replay()

    def join(self) -> None:
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            cur.wait_stream(s)


# ---------------------------------------------------------------------------------------------- bilateral -> CLAHE
def bilateral_clahe_workspace_bytes(n: int, h: int, w: int, grid_size=(16, 16)) -> int:
    return int(lib().mie_bilateral_clahe_workspace_bytes(n, h, w, int(grid_size[0]), int(grid_size[1])))


def bilateral_clahe(input: torch.Tensor, kernel_size=9, sigma_color=0.1, sigma_space=(1.5, 1.5), clip_limit: float = 2.0,
                    grid_size: tuple = (16, 16), border_type: str = "reflect", *, value_range=None, out: torch.Tensor = None,
                    out_dtype=None, workspace: torch.Tensor = None, stages: int = 7) -> torch.Tensor:
    """BASELINE.json config 4 as one fused path: equalize_clahe(bilateral_blur(x, kernel_size, sigma_color, sigma_space,
    border_type), clip_limit, grid_size), quantised once at the end to the input's dtype (or float32).

    Bit-identical to `equalize_clahe(bilateral_blur(x, ..., out_dtype=torch.float32), ...)` followed by the integer
    quantisation, but the filtered image never exists: the bilateral kernel emits the CLAHE lookup index of each pixel
    (1 byte) and the tile histograms, and the interpolation pass reads that byte.  Geometry outside the fused kernels'
    reach (see mie_bilateral_clahe in include/mie.h) raises NotImplementedError — call the two operators instead."""
    _check_clahe_args(clip_limit, grid_size)
    require_cuda(input)
    k, kx = _pair_int(kernel_size, "kernel_size")
    if k != kx:
        raise NotImplementedError("the fused path needs a square bilateral window")
    _check_kernel(k, kx)
    sy, sx = _pair_float(sigma_space, "sigma_space")
    x, n, h, w = as_planes(input)
    lo, hi = value_range_of(x, value_range)
    out = new_out(x, out_dtype) if out is None else check_out(x, out)
    gh, gw = int(grid_size[0]), int(grid_size[1])
    workspace = use_workspace(x.device, lib().mie_bilateral_clahe_workspace_bytes(n, h, w, gh, gw), workspace)
    wsp = np.ascontiguousarray(
        (get_gaussian_kernel1d(k, sy)[:, None] * get_gaussian_kernel1d(k, sx)[None, :]).astype(np.float32))
    call(x.device, "mie_bilateral_clahe", x.data_ptr(), out.data_ptr(), DTYPE_CODE[x.dtype], DTYPE_CODE[out.dtype],
         *plane_layout(n, h, w), wsp.ctypes.data, k, float(sigma_color), _border(border_type), gh, gw,
         float(clip_limit), lo, hi, int(stages), workspace.data_ptr(), workspace.numel())
    return out


class BilateralClahePlan:
    """bilateral_clahe on fixed device buffers (input, output, workspace allocated once): `run()` enqueues one pass;
    `stage_ms()` times the three stages separately with CUDA events."""

    def __init__(self, input: torch.Tensor, *, out: torch.Tensor = None, **kwargs):
        require_cuda(input)
        self.input, self.kwargs = input, kwargs
        x, n, h, w = as_planes(input)
        self.out = out if out is not None else torch.empty_like(input)
        grid = kwargs.get("grid_size", (16, 16))
        self.workspace = use_workspace(input.device, bilateral_clahe_workspace_bytes(n, h, w, grid))

    def run(self, stages: int = 7) -> torch.Tensor:
        return bilateral_clahe(self.input, out=self.out, workspace=self.workspace, stages=stages, **self.kwargs)

    def stage_ms(self) -> dict:
        res = {}
        for name, mask in (("bilateral_index_hist", 1), ("hist_to_lut", 2), ("pack_cells+apply_index", 4)):
            self.run(mask)
            torch.cuda.synchronize(self.input.device)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            self.run(mask)
            e1.record()
            torch.cuda.synchronize(self.input.device)
            res[name] = round(e0.elapsed_time(e1), 4)
        return res
