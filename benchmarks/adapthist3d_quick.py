#!/usr/bin/env python
"""skimage.exposure.equalize_adapthist on whole volumes (skimage_compat.equalize_adapthist(..., volumetric=True)):
CUDA-event timing of one call, and the device time of each kernel from a separate torch.profiler pass.
    python benchmarks/adapthist3d_quick.py

Workloads: a 512^3 int16 CT-like volume with the default 64^3 kernel (float64 and float32 out; 268 MB of input, larger
than the 126 MB L2), a 256^3 uint16 volume with a 32^3 kernel, a batch of 4 x 128^3 (input L2-resident).
bytes floor = the bytes the algorithm must move, from shapes: the input read three times (min / max, region histograms,
blend), the uint16 intermediate written and read once, the output written once; floor_ms = bytes / 7.7 TB/s (HBM3e
data-sheet bandwidth of one B200, not a measured figure)."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mie_b200 import skimage_compat as S, synthetic  # noqa: E402

HBM_BYTES_S = 7.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr.strip()}


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_times(fn, reps=5):
    """Mean device time per call of every kernel the call launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            out[ev.key[:90]] = round(t / reps / 1e3, 4)   # ms per call
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    v512 = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, 0)).to(dev)
    v256 = torch.from_numpy(synthetic.phantom_volume((256, 256, 256), np.uint16, 1)).to(dev)
    b128 = torch.from_numpy(np.stack([synthetic.phantom_volume((128, 128, 128), np.int16, s) for s in range(4)])).to(dev)
    cases = [
        ("512^3 i16 default kernel (64^3) -> float64", lambda: S.equalize_adapthist(v512, volumetric=True), v512, 8),
        ("512^3 i16 default kernel (64^3) -> float32",
         lambda: S.equalize_adapthist(v512, volumetric=True, out_dtype=torch.float32), v512, 4),
        ("256^3 u16 kernel (32, 32, 32) -> float64",
         lambda: S.equalize_adapthist(v256, (32, 32, 32), volumetric=True), v256, 8),
        ("4 x 128^3 i16 default kernel (16^3) -> float64", lambda: S.equalize_adapthist(b128, volumetric=True), b128, 8),
    ]
    for name, fn, x, out_bytes in cases:
        vox = x.numel()
        ms = timed(fn, 10)
        floor_bytes = vox * (3 * x.element_size() + 2 * 2 + out_bytes)
        floor_ms = floor_bytes / HBM_BYTES_S * 1e3
        rec = {"case": name, "ms": round(ms, 4), "gvoxel_s": round(vox / ms / 1e6, 2), "bytes_floor_gb": round(floor_bytes / 1e9, 3),
               "floor_ms": round(floor_ms, 4), "time_over_floor": round(ms / floor_ms, 2), "kernels_ms": kernel_times(fn),
               "device": info["device"], "nvidia_smi": info["nvidia_smi"]}
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
