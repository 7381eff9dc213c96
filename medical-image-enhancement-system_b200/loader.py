"""Slice / volume batching loader (SURVEY.md §8(f) F1; named in the north star as a subsystem that
changes): host-resident slice stacks are streamed through the GPU kernels in chunks, with the
host->device copy of chunk k+1, the kernels of chunk k and the device->host copy of chunk k-1
running concurrently on three CUDA streams (PCIe is full duplex, so a step costs about
max(H2D, D2H) instead of their sum plus the kernels).

    pipe = HostSlicePipeline(device, (512, 512), torch.uint16, chunk=32)
    pipe.run(x_host_pinned, y_host_pinned)          # enhance_chain on every slice

Pinned host memory is required for the copies to be asynchronous; `pin()` is a helper.
Integer <-> [0,1] normalisation policy (value_range / HU window) travels in ChainConfig.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch

from ._ffi import use_workspace
from .chain import ChainConfig, chain_workspace_bytes, enhance_chain

__all__ = ["HostSlicePipeline", "HostVolumePipeline", "pin", "enhance_chain_host", "median3d_clahe_host"]


def pin(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_pinned() else t.contiguous().pin_memory()


class HostSlicePipeline:
    """Triple-buffered host -> device -> host pipeline over the leading (slice) dimension.

    `fn(x_dev, out_dev, workspace)` enqueues the device work of one chunk on the current stream;
    the default runs the fused Gaussian -> CLAHE -> unsharp chain.
    """

    def __init__(self, device, slice_shape, dtype, chunk: int = 32, depth: int = 3,
                 config: ChainConfig = ChainConfig(), fn: Optional[Callable] = None, out_dtype=None, taper: bool = True):
        self.device = torch.device(device)
        self.h, self.w = int(slice_shape[-2]), int(slice_shape[-1])
        self.chunk, self.depth, self.config = int(chunk), int(depth), config
        self.taper = bool(taper)
        self.dtype = dtype
        self.out_dtype = dtype if out_dtype is None else out_dtype
        self.fn = fn
        with torch.cuda.device(self.device):
            self.s_in, self.s_comp, self.s_out = (torch.cuda.Stream() for _ in range(3))
            shape = (self.chunk, 1, self.h, self.w)
            self.x = [torch.empty(shape, dtype=dtype, device=self.device) for _ in range(depth)]
            self.y = [torch.empty(shape, dtype=self.out_dtype, device=self.device) for _ in range(depth)]
            ws = chain_workspace_bytes(self.chunk, self.h, self.w, config.grid_size)
            self.ws = [use_workspace(self.device, ws) for _ in range(depth)]
            self.ev_in = [torch.cuda.Event() for _ in range(depth)]
            self.ev_comp = [torch.cuda.Event() for _ in range(depth)]
            self.ev_out = [torch.cuda.Event() for _ in range(depth)]
        self.launches_per_chunk = 3
        # whole-run CUDA graph for repeated calls on the same host buffers (see run())
        self._graph = None
        self._graph_key = None
        self._last_key = None
        self._graph_refs = None

    def _device_work(self, x, y, ws):
        if self.fn is not None:
            self.fn(x, y, ws)
        else:
            enhance_chain(x, self.config, out=y, workspace=ws)

    def run(self, src: torch.Tensor, dst: torch.Tensor, graph: bool = True) -> torch.Tensor:
        """src, dst: host tensors (N, H, W) or (N, 1, H, W), ideally pinned.  Returns dst.  The call
        returns after the last device->host copy has been enqueued AND completed.

        A loop that reuses the same pinned staging buffers (the usual way to feed a GPU) pays the Python
        and launch cost of every chunk — ~0.1 ms each, more than the chunk's kernels — on every call.
        So the second call with the same (src, dst) captures the whole run — every copy, kernel and
        cross-stream dependency of all chunks — into one CUDA graph, and later calls replay it."""
        self._validate(src, dst)
        key = (src.data_ptr(), dst.data_ptr(), tuple(src.shape), src.dtype, dst.dtype)
        if graph and self._graph is not None and self._graph_key == key:
            self._graph.replay()
            torch.cuda.current_stream(self.device).synchronize()
            return dst
        if graph and self._last_key == key and src.is_pinned() and dst.is_pinned() and self.fn is None:
            try:
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream(device=self.device)
                with torch.cuda.stream(side):
                    with torch.cuda.graph(g, stream=side):
                        self._enqueue(src, dst)
                self._graph, self._graph_key, self._graph_refs = g, key, (src, dst)
                return self.run(src, dst, graph=True)
            except RuntimeError:
                # capture refused (e.g. pageable memory): stay eager.  The streams the failed capture forked into are
                # left in an invalidated capture state, so they are replaced along with their events.
                self._graph = None
                torch.cuda.synchronize(self.device)
                with torch.cuda.device(self.device):
                    self.s_in, self.s_comp, self.s_out = (torch.cuda.Stream() for _ in range(3))
                    self.ev_in = [torch.cuda.Event() for _ in range(self.depth)]
                    self.ev_comp = [torch.cuda.Event() for _ in range(self.depth)]
                    self.ev_out = [torch.cuda.Event() for _ in range(self.depth)]
        self._last_key = key
        self._enqueue(src, dst)
        self.s_out.synchronize()
        return dst

    def _validate(self, src: torch.Tensor, dst: torch.Tensor) -> None:
        """A dtype mismatch would be converted silently by copy_ (a blocking CPU cast that defeats the asynchronous
        pipeline, and data then processed with the wrong value range): refuse up front."""
        for name, t in (("src", src), ("dst", dst)):
            if not isinstance(t, torch.Tensor):
                raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
            if t.is_cuda:
                raise ValueError(f"{name} must be a host tensor (use enhance_chain for device tensors)")
            if t.dim() not in (3, 4) or tuple(t.shape[-2:]) != (self.h, self.w) or (t.dim() == 4 and t.shape[1] != 1):
                raise ValueError(f"{name} must be (N, {self.h}, {self.w}) or (N, 1, {self.h}, {self.w}); got {tuple(t.shape)}")
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
        if src.dtype != self.dtype:
            raise TypeError(f"src dtype {src.dtype} does not match the pipeline's dtype {self.dtype}")
        if dst.dtype != self.out_dtype:
            raise TypeError(f"dst dtype {dst.dtype} does not match the pipeline's out_dtype {self.out_dtype}")
        if src.shape[0] != dst.shape[0]:
            raise ValueError("src and dst must hold the same number of slices")

    def schedule(self, n: int):
        """Chunk boundaries [(z0, z1), ...] over n slices.  The copies in the two PCIe directions overlap except while the
        pipeline fills (first upload) and drains (last download), so with `taper` the first and the last chunks are a
        quarter and a half of the regular size: the exposed ends shrink fourfold for a handful of extra launches."""
        c = self.chunk
        head = [c // 4, c // 2] if self.taper and c >= 8 and n >= 3 * c else []
        tail = head[::-1]
        sizes, left = [], n
        for s_ in head:
            sizes.append(s_); left -= s_
        left -= sum(tail)
        while left > 0:
            s_ = min(c, left)
            sizes.append(s_); left -= s_
        sizes += tail
        spans, z = [], 0
        for s_ in sizes:
            spans.append((z, z + s_)); z += s_
        assert z == n
        return spans

    def _enqueue(self, src: torch.Tensor, dst: torch.Tensor) -> None:
        n = src.shape[0]
        s = src.reshape(n, 1, self.h, self.w)
        d = dst.reshape(n, 1, self.h, self.w)
        caller = torch.cuda.current_stream(self.device)
        for st in (self.s_in, self.s_comp, self.s_out):
            st.wait_stream(caller)
        used = [False] * self.depth
        for i, (z0, z1) in enumerate(self.schedule(n)):
            m, k = z1 - z0, i % self.depth
            with torch.cuda.stream(self.s_in):
                if used[k]:
                    self.s_in.wait_event(self.ev_comp[k])    # kernels of the previous user of x[k] are done
                self.x[k][:m].copy_(s[z0:z1], non_blocking=True)
                self.ev_in[k].record(self.s_in)
            with torch.cuda.stream(self.s_comp):
                self.s_comp.wait_event(self.ev_in[k])
                if used[k]:
                    self.s_comp.wait_event(self.ev_out[k])   # previous contents of y[k] have left the device
                self._device_work(self.x[k][:m], self.y[k][:m], self.ws[k])
                self.ev_comp[k].record(self.s_comp)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_comp[k])
                d[z0:z1].copy_(self.y[k][:m], non_blocking=True)
                self.ev_out[k].record(self.s_out)
            used[k] = True
        caller.wait_stream(self.s_in)
        caller.wait_stream(self.s_comp)
        caller.wait_stream(self.s_out)


def enhance_chain_host(src: torch.Tensor, config: ChainConfig = ChainConfig(), *, out: torch.Tensor = None,
                       device="cuda", chunk: int = 32) -> torch.Tensor:
    """One-call convenience: enhance a host-resident slice stack (N, H, W) / (N, 1, H, W) on `device`."""
    if src.is_cuda:
        raise ValueError("enhance_chain_host takes host tensors; use enhance_chain for device tensors")
    src = pin(src)
    if out is None:
        out = torch.empty_like(src).pin_memory()
    pipe = HostSlicePipeline(device, src.shape[-2:], src.dtype, chunk=min(chunk, max(int(src.shape[0]), 1)), config=config)
    return pipe.run(src, out)


class HostVolumePipeline:
    """BASELINE.json config 3 for a HOST-resident volume: (D, H, W) int16 / uint16 / uint8 planes are streamed
    through the GPU in z-chunks — 3x3x3 median (skimage.filters.median semantics) followed by per-slice CLAHE
    — with the upload of chunk k+1, the kernels of chunk k and the download of chunk k-1 overlapping on three
    streams.  A chunk is uploaded together with its two neighbouring planes, which serve as the median's z-halo
    exactly like the planes a neighbouring rank would send (volume.py), so the result is bit-identical to
    processing the whole volume on the device.

        pipe = HostVolumePipeline("cuda:0", (512, 512), torch.int16, chunk=64)
        pipe.run(vol_host_pinned, out_host_pinned)
    """

    def __init__(self, device, plane_shape, dtype, chunk: int = 64, depth: int = 3, clip_limit: float = 2.0,
                 grid_size: tuple = (8, 8), mode: str = "nearest", value_range=None):
        self.device = torch.device(device)
        self.h, self.w = int(plane_shape[-2]), int(plane_shape[-1])
        self.chunk, self.depth = int(chunk), int(depth)
        self.clip_limit, self.grid_size, self.mode, self.value_range = float(clip_limit), tuple(grid_size), mode, value_range
        self.dtype = dtype
        with torch.cuda.device(self.device):
            self.s_in, self.s_comp, self.s_out = (torch.cuda.Stream() for _ in range(3))
            # chunk planes plus one halo plane on either side
            self.x = [torch.empty((self.chunk + 2, self.h, self.w), dtype=dtype, device=self.device) for _ in range(depth)]
            self.y = [None] * depth
            self.ev_in = [torch.cuda.Event() for _ in range(depth)]
            self.ev_comp = [torch.cuda.Event() for _ in range(depth)]
            self.ev_out = [torch.cuda.Event() for _ in range(depth)]

    def run(self, src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
        """src, dst: host tensors (D, H, W), ideally pinned (see pin()).  Returns dst once it is complete."""
        from .enhance import equalize_clahe
        from .filters import median

        if src.is_cuda or dst.is_cuda:
            raise ValueError("HostVolumePipeline takes host tensors")
        if src.dim() != 3 or src.shape != dst.shape or src.shape[1:] != (self.h, self.w):
            raise ValueError("expected (D, H, W) volumes of the pipeline's plane shape")
        if src.dtype != self.dtype or dst.dtype != self.dtype:
            raise TypeError(f"src / dst dtype must be the pipeline's dtype {self.dtype}; got {src.dtype} / {dst.dtype}")
        d = int(src.shape[0])
        caller = torch.cuda.current_stream(self.device)
        for st in (self.s_in, self.s_comp, self.s_out):
            st.wait_stream(caller)
        used = [False] * self.depth
        for i, z0 in enumerate(range(0, d, self.chunk)):
            z1 = min(z0 + self.chunk, d)
            m, k = z1 - z0, i % self.depth
            a, b = max(z0 - 1, 0), min(z1 + 1, d)          # planes uploaded: the chunk and its z-neighbours
            off = z0 - a                                   # 1 when a lower halo plane is present
            with torch.cuda.stream(self.s_in):
                if used[k]:
                    self.s_in.wait_event(self.ev_comp[k])
                self.x[k][:b - a].copy_(src[a:b], non_blocking=True)
                self.ev_in[k].record(self.s_in)
            with torch.cuda.stream(self.s_comp):
                self.s_comp.wait_event(self.ev_in[k])
                if used[k]:
                    self.s_comp.wait_event(self.ev_out[k])
                buf = self.x[k]
                med = median(buf[off:off + m], mode=self.mode, halo_lo=buf[0] if off else None,
                             halo_hi=buf[off + m] if z1 < d else None)
                self.y[k] = equalize_clahe(med.unsqueeze(1), self.clip_limit, self.grid_size,
                                           value_range=self.value_range).squeeze(1)
                self.y[k].record_stream(self.s_out)
                self.ev_comp[k].record(self.s_comp)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(self.ev_comp[k])
                dst[z0:z1].copy_(self.y[k], non_blocking=True)
                self.ev_out[k].record(self.s_out)
            used[k] = True
        self.s_out.synchronize()
        self.s_comp.synchronize()
        return dst


def median3d_clahe_host(vol: torch.Tensor, clip_limit: float = 2.0, grid_size: tuple = (8, 8), *, out: torch.Tensor = None,
                        device="cuda", chunk: int = 64, mode: str = "nearest", value_range=None) -> torch.Tensor:
    """One-call convenience: 3x3x3 median + per-slice CLAHE of a host-resident (D, H, W) volume on `device`."""
    if vol.is_cuda:
        raise ValueError("median3d_clahe_host takes host tensors; use median3d_clahe_slab for device tensors")
    vol = pin(vol)
    if out is None:
        out = torch.empty_like(vol).pin_memory()
    pipe = HostVolumePipeline(device, vol.shape[-2:], vol.dtype, chunk=min(chunk, max(int(vol.shape[0]), 1)),
                              clip_limit=clip_limit, grid_size=grid_size, mode=mode, value_range=value_range)
    return pipe.run(vol, out)
