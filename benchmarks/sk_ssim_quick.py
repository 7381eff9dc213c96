#!/usr/bin/env python
"""skimage.metrics.structural_similarity on the GPU (skimage_compat.structural_similarity): CUDA-event timing of one
call after warm-up, the device time of each kernel from a separate torch.profiler pass, and the numpy twin
(tests/sk_ssim_twin.py, scipy.ndimage) on the same host.
    python benchmarks/sk_ssim_quick.py [--out FILE.jsonl]

Inputs are larger than the 126 MB L2 (two 512^3 int16 volumes are 537 MB), so every call reads them from HBM.  Per case:
ms per call (the call ends in one 8-byte device-to-host copy of mssim); the bytes floor — both inputs read once, plus the
map if written — at 7.7 TB/s (HBM3e data-sheet bandwidth of one B200, not a measured figure); the float64 operations the
line passes and the S formula need, counted from shapes; the workspace bytes; and the twin's time on a 256^3
sub-volume (32 planes for the plane case), scaled by the voxel ratio and labelled as scaled, not run at full size."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
import sk_ssim_twin as T  # noqa: E402
from mie_b200 import _ffi, skimage_compat as S, synthetic  # noqa: E402
from tv_chambolle_quick import card, kernel_times, timed  # noqa: E402

HBM_BYTES_S = 7.7e12


def f64_ops(voxels, ndim, win, gaussian, float64_image):
    """float64 operations per call: every line pass costs 3 per output and quantity (box: add, subtract, divide) or
    1 + 3 r (Gaussian with radius r), over 5 quantities and ndim passes; float64 images add the 3 products and the 23
    operations of the S formula per voxel."""
    per_output = 1 + 3 * (win // 2) if gaussian else 3
    per_voxel = 5 * ndim * per_output + (3 + 23 if float64_image else 0)
    return voxels * per_voxel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    vol = torch.from_numpy(synthetic.phantom_volume((512, 512, 512), np.int16, 0)).to(dev)
    vol_b = S.gaussian(vol, 1.0, volumetric=True)
    f32 = ((vol.to(torch.float64) * 2.0 + 1.0) / 65535.0).to(torch.float32)
    f32_b = ((vol_b.to(torch.float64) * 2.0 + 1.0) / 65535.0).to(torch.float32)
    planes = torch.from_numpy(synthetic.phantom((256, 1, 512, 512), np.uint16, 0)).to(dev)
    planes_b = S.gaussian(planes, 1.0)
    cases = [("512^3 i16 volumetric box7 no map", vol, vol_b, True, dict()),
             ("512^3 i16 volumetric box7 full", vol, vol_b, True, dict(full=True)),
             ("512^3 f32 volumetric box7 no map", f32, f32_b, True, dict(data_range=2.0)),
             ("512^3 i16 volumetric gaussian (11 taps) no map", vol, vol_b, True, dict(gaussian_weights=True)),
             ("256 x 512^2 u16 planes box7 no map", planes, planes_b, False, dict())]
    records = []
    for name, x, y, volumetric, kw in cases:
        ndim = 3 if volumetric else 2
        voxels = x.numel()
        win = 11 if kw.get("gaussian_weights") else 7
        f64_image = x.dtype != torch.float32
        map_bytes = voxels * (8 if f64_image else 4) if kw.get("full") else 0
        floor_ms = (2 * voxels * x.element_size() + map_bytes) / HBM_BYTES_S * 1e3
        code = _ffi.DTYPE_CODE[x.dtype]
        lib = _ffi.lib()
        if volumetric:
            ws = lib.mie_sk_structural_similarity3d_workspace_bytes(1, *x.shape[-3:], code)
        else:
            ws = lib.mie_sk_structural_similarity_workspace_bytes(x.numel() // (512 * 512), 512, 512, code)

        def call(x=x, y=y, kw=kw, volumetric=volumetric):
            return S.structural_similarity(x, y, volumetric=volumetric, **kw)

        ms = timed(call, 5)
        kt = kernel_times(call)
        result = call()
        mssim = result[0] if kw.get("full") else result
        if volumetric:
            sub = (x[:256, :256, :256].cpu().numpy(), y[:256, :256, :256].cpu().numpy())
        else:
            sub = (x[:32, 0].cpu().numpy(), y[:32, 0].cpu().numpy())
        tw_kw = {k: v for k, v in kw.items() if k != "full"}
        t0 = time.perf_counter()
        if volumetric:
            T.structural_similarity(*sub, **tw_kw)
        else:
            for i in range(32):
                T.structural_similarity(sub[0][i], sub[1][i], **tw_kw)
        twin_s = time.perf_counter() - t0
        scale = voxels / sub[0].size
        ops = f64_ops(voxels, ndim, win, kw.get("gaussian_weights", False), f64_image)
        rec = {"case": name, "ms": round(ms, 3), "mssim": float(mssim.mean()) if torch.is_tensor(mssim) else mssim,
               "bytes_floor_ms": round(floor_ms, 4), "of_bytes_floor": round(floor_ms / ms, 3),
               "f64_ops": ops, "f64_gops_per_s": round(ops / ms / 1e6, 1), "workspace_bytes": ws,
               "twin_cpu_s_subset": round(twin_s, 2), "twin_cpu_subset": "256^3" if volumetric else "32 planes",
               "twin_cpu_s_scaled_to_full_size": round(twin_s * scale, 1),
               "speedup_vs_twin_scaled": round(twin_s * scale * 1e3 / ms, 1), "cpu_threads": os.cpu_count(),
               "kernels_ms": kt}
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
