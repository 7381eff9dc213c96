#!/usr/bin/env python
"""Median with a footprint on the GPU (filters.median / mie_sk_median*): CUDA-event timing of one call after warm-up,
the device time of each kernel from a separate torch.profiler pass, and scipy.ndimage.median_filter (what
skimage.filters.median calls) on the same host.
    python benchmarks/sk_median_quick.py [--out FILE.jsonl]

Inputs are synthetic.phantom_volume (int16 HU; the float32 volume is the same one in float32) and 256 uint16 planes of
synthetic.phantom.  Per case: ms per call; the bytes floor (source read and destination written once) and that floor at
7.7 TB/s (HBM3e data-sheet bandwidth of one B200, not a measured figure); the counted selection work of the radix
kernel (outputs x footprint cells x key bits compares, each one shared-memory load of a key, plus one offset load per 4
outputs); and scipy's time on a 128^3 sub-volume (16 planes for the plane cases), scaled by the voxel ratio and labelled
as scaled.  The 3^3 box on int16 runs both through mie_sk_median3d (the ABI directly: filters.median sends that
footprint to mie_median3d) and through mie_median3d, the comparison that keeps both kernels."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
from scipy import ndimage as ndi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
from mie_b200 import _ffi, filters as F, skimage_compat as S, synthetic  # noqa: E402
from tv_chambolle_quick import card, kernel_times, timed  # noqa: E402

HBM_BYTES_S = 7.7e12
NEAREST = _ffi.BORDER["replicate"]


def sk_median_abi(x, fp, planes):
    """mie_sk_median (n planes of x) or mie_sk_median3d (x one volume) in 'nearest' mode."""
    out = torch.empty_like(x)
    fp8 = np.ascontiguousarray(fp, dtype=np.uint8)
    code = _ffi.DTYPE_CODE[x.dtype]
    if planes:
        n, h, w = x.shape
        _ffi.call(x.device, "mie_sk_median", x.data_ptr(), out.data_ptr(), code, *_ffi.plane_layout(n, h, w),
                  fp8.ctypes.data, *fp8.shape, NEAREST, 0.0)
    else:
        _ffi.call(x.device, "mie_sk_median3d", x.data_ptr(), out.data_ptr(), code, *_ffi.volume_layout(1, *x.shape),
                  fp8.ctypes.data, *fp8.shape, NEAREST, 0.0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    vol = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, seed=0)).to(dev)
    f32 = vol.to(torch.float32).contiguous()
    planes = torch.from_numpy(synthetic.phantom((256, 512, 512), np.uint16, seed=1)).to(dev)
    box3, box5 = np.ones((3, 3, 3), np.uint8), np.ones((5, 5, 5), np.uint8)
    cases = [("512^3 i16 ball(1)", vol, S.ball(1), "sk"), ("512^3 i16 ball(2)", vol, S.ball(2), "sk"),
             ("512^3 i16 ball(3)", vol, S.ball(3), "sk"), ("512^3 i16 box 5^3", vol, box5, "sk"),
             ("512^3 f32 ball(2)", f32, S.ball(2), "sk"),
             ("256 x 512^2 u16 planes disk(3)", planes, S.disk(3), "planes"),
             ("256 x 512^2 u16 planes disk(5)", planes, S.disk(5), "planes"),
             ("512^3 i16 box 3^3 via mie_sk_median3d", vol, box3, "sk"),
             ("512^3 i16 box 3^3 via mie_median3d", vol, box3, "old")]
    records = []
    for name, x, fp, path in cases:
        if path == "old":
            def call(x=x):
                return F.median(x)
        else:
            def call(x=x, fp=fp, path=path):
                return sk_median_abi(x, fp, path == "planes")

        ms = timed(call, 3)
        kt = kernel_times(call, 1)
        cells = int(np.count_nonzero(fp))
        bits = 8 * x.element_size()
        nbytes = 2 * x.numel() * x.element_size()
        floor_ms = nbytes / HBM_BYTES_S * 1e3
        sub = x[:16].cpu().numpy() if path == "planes" else x[:128, :128, :128].cpu().numpy()
        t0 = time.perf_counter()
        if path == "planes":
            for i in range(sub.shape[0]):
                ndi.median_filter(sub[i], footprint=fp.astype(bool), mode="nearest")
        else:
            ndi.median_filter(sub, footprint=fp.astype(bool), mode="nearest")
        scipy_s = time.perf_counter() - t0
        scale = x.numel() / sub.size
        rec = {"case": name, "kernel": "mie_median3d" if path == "old" else "sk_median_kernel", "ms": round(ms, 3),
               "footprint_cells": cells, "key_bits": bits, "bytes_floor": nbytes,
               "bytes_floor_ms": round(floor_ms, 3), "of_bytes_floor": round(floor_ms / ms, 4)}
        if path != "old":
            compares = x.numel() * cells * bits
            rec.update({"selection_compares": compares, "selection_key_loads": compares,
                        "selection_offset_loads": compares // 4,
                        "gcompares_per_s": round(compares / ms / 1e6, 1)})
        rec.update({"scipy_cpu_s_subset": round(scipy_s, 2),
                    "scipy_cpu_subset": "16 planes" if path == "planes" else "128^3",
                    "scipy_cpu_s_scaled_to_full_size": round(scipy_s * scale, 1),
                    "speedup_vs_scipy_scaled": round(scipy_s * scale * 1e3 / ms, 1), "cpu_threads": os.cpu_count(),
                    "kernels_ms": kt})
        rec.update(info)
        print(json.dumps(rec), flush=True)
        records.append(rec)
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for r in records:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
