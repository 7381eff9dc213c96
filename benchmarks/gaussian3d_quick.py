#!/usr/bin/env python
"""skimage.filters.gaussian / unsharp_mask on whole volumes (skimage_compat.gaussian(..., volumetric=True)):
CUDA-event timing of one call, the device time of each kernel from a separate torch.profiler pass, and the obvious
torch alternative — three separable fp32 F.conv3d calls after replicate padding (TF32 off) — on the same volume.
    python benchmarks/gaussian3d_quick.py

Floors, computed from shapes by this script:
  bytes floor = input read once + output written once, at 7.7 TB/s (HBM3e data-sheet bandwidth of one B200, not a
                measured figure);
  FMA floor   = (kx * x-pass rows / h + ky + kz) FMAs per voxel — the x pass also runs on the tile's y-halo rows —
                at 148 SMs x 128 FP32 FMA per clock x clocks.max.sm read from nvidia-smi in the same call (FFMA2 does
                not raise the FMA pipe's rate).  An estimate, not a measurement.
`of_floor` is the larger floor over the measured kernel time."""
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mie_b200 import skimage_compat as S, synthetic  # noqa: E402

HBM_BYTES_S = 7.7e12
SMS, FMA_PER_CLK = 148, 128


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.stdout else q.stderr.strip()
    try:
        mhz = float(line.split(",")[2].split()[0])
    except (IndexError, ValueError):
        mhz = float("nan")
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line, "sm_clock_max_mhz": mhz}


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


def taps(sigma):
    s = float(sigma)
    return 1 if s == 0 else 2 * int(4.0 * s + 0.5) + 1


def fma_per_voxel(h, k):
    """kx * (x-pass rows per column) / h + ky + kz, with the kernel's tile height (gauss3d.cu: 32 rows for radius
    buckets up to 4, 16 above)."""
    kz, ky, kx = k
    r = max(k) // 2
    ty = 32 if r <= 4 else 16
    tiles_y = -(-h // ty)
    return kx * tiles_y * (ty + 2 * (ky // 2)) / h + ky + kz


def conv3d_baseline(x, sig, value_range, amount=None):
    """fp32 torch: map to [0, 1], replicate-pad once, three separable F.conv3d (x, y, z); with `amount`, the unsharp
    mask v + amount * (v - blur) on top (replicate border: compare away from the faces)."""
    lo, hi = value_range
    k = [taps(s) for s in sig]
    ws = [S.get_gaussian_kernel1d(kk, s) if s else np.ones(1, np.float32) for kk, s in zip(k, sig)]
    wz = torch.from_numpy(ws[0]).to(x.device).view(1, 1, -1, 1, 1)
    wy = torch.from_numpy(ws[1]).to(x.device).view(1, 1, 1, -1, 1)
    wx = torch.from_numpy(ws[2]).to(x.device).view(1, 1, 1, 1, -1)
    rz, ry, rx = (kk // 2 for kk in k)

    def run():
        v = x.float() if x.dtype == torch.float32 else (x.float() - lo) / (hi - lo)
        p = F.pad(v.view(1, 1, *x.shape[-3:]), (rx, rx, ry, ry, rz, rz), mode="replicate")
        blur = F.conv3d(F.conv3d(F.conv3d(p, wx), wy), wz)[0, 0]
        return blur if amount is None else v + amount * (v - blur)
    return run


def main():
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    fma_s = SMS * FMA_PER_CLK * info["sm_clock_max_mhz"] * 1e6
    v512 = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, 0)).to(dev)
    f512 = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, 0).astype(np.float32) / 4096.0 + 0.25
                            ).to(dev)
    thick = torch.from_numpy(synthetic.phantom_volume((256, 512, 512), np.int16, 1)).to(dev)
    b128 = torch.from_numpy(np.stack([synthetic.phantom_volume((128, 128, 128), np.uint16, s) for s in range(4)])).to(dev)
    i16 = (-32768.0, 32767.0)
    cases = [
        # name, fn, float32-output fn for the baseline comparison (None: no baseline), input, sigma (z, y, x), value range
        ("512^3 i16 sigma 1 (9 taps per axis), nearest", lambda: S.gaussian(v512, 1.0, volumetric=True),
         lambda: S.gaussian(v512, 1.0, volumetric=True, out_dtype=torch.float32), v512, (1.0, 1.0, 1.0), i16),
        ("512^3 i16 sigma 2 (17 taps per axis), nearest", lambda: S.gaussian(v512, 2.0, volumetric=True),
         lambda: S.gaussian(v512, 2.0, volumetric=True, out_dtype=torch.float32), v512, (2.0, 2.0, 2.0), i16),
        ("512^3 i16 unsharp radius 1 amount 1.5 (reflect)", lambda: S.unsharp_mask(v512, 1.0, 1.5, volumetric=True),
         lambda: S.unsharp_mask(v512, 1.0, 1.5, True, volumetric=True, out_dtype=torch.float32), v512, (1.0, 1.0, 1.0),
         i16),
        ("512^3 f32 sigma 1, nearest", lambda: S.gaussian(f512, 1.0, volumetric=True),
         lambda: S.gaussian(f512, 1.0, volumetric=True), f512, (1.0, 1.0, 1.0), (0.0, 1.0)),
        ("256x512x512 i16 sigma (0.5, 1.5, 1.5) thick slices, nearest",
         lambda: S.gaussian(thick, (0.5, 1.5, 1.5), volumetric=True),
         lambda: S.gaussian(thick, (0.5, 1.5, 1.5), volumetric=True, out_dtype=torch.float32), thick,
         (0.5, 1.5, 1.5), i16),
        ("4 x 128^3 u16 sigma 1, nearest (in + out 33 MB: L2-resident)", lambda: S.gaussian(b128, 1.0, volumetric=True),
         None, b128, (1.0, 1.0, 1.0), (0.0, 65535.0)),
    ]
    for name, fn, fn32, x, sig, vr in cases:
        vox = x.numel()
        d, h, w = x.shape[-3:]
        ms = timed(fn, 20)
        kt = kernel_times(fn)
        kms = sum(t for k, t in kt.items() if "gauss3d" in k)
        k = [taps(s) for s in sig]
        bytes_floor = 2 * vox * x.element_size()
        bytes_ms = bytes_floor / HBM_BYTES_S * 1e3
        fmas = fma_per_voxel(h, k) * vox
        fma_ms = fmas / fma_s * 1e3
        floor_ms = max(bytes_ms, fma_ms)
        rec = {"case": name, "ms": round(ms, 4), "kernel_ms": round(kms, 4), "gvoxel_s": round(vox / ms / 1e6, 2),
               "taps_zyx": k, "bytes_floor_gb": round(bytes_floor / 1e9, 3), "bytes_floor_ms": round(bytes_ms, 4),
               "fma_per_voxel": round(fmas / vox, 2), "fma_floor_ms": round(fma_ms, 4),
               "bound_by": "fma" if fma_ms >= bytes_ms else "bytes", "of_floor": round(floor_ms / kms, 3) if kms else None,
               "kernels_ms": kt}
        if fn32 is not None and x.dim() == 3:
            unsharp = "unsharp" in name
            base = conv3d_baseline(x, sig, vr, 1.5 if unsharp else None)
            rec["conv3d_baseline_ms"] = round(timed(base, 5), 4)
            rec["speedup_vs_conv3d"] = round(rec["conv3d_baseline_ms"] / ms, 2)
            diff = (fn32().float() - base()).abs()
            if unsharp:   # reflect vs replicate border: interior only
                rz, ry, rx = (kk // 2 for kk in k)
                diff = diff[rz:d - rz, ry:h - ry, rx:w - rx]
            rec["max_abs_diff_vs_conv3d" + ("_interior" if unsharp else "")] = float(diff.max())
        rec.update({"device": info["device"], "nvidia_smi": info["nvidia_smi"]})
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
