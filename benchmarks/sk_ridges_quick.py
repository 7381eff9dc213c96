#!/usr/bin/env python
"""Hessian ridge filters on the GPU (skimage_compat.frangi / sato): CUDA-event timing of one call after warm-up, the
device time of each kernel from a separate torch.profiler pass, and the numpy twin (tests/sk_ridges_twin.py,
scipy.ndimage + np.linalg.eigvalsh) on the same host.
    python benchmarks/sk_ridges_quick.py [--out FILE.jsonl]

Inputs are synthetic.vessel_volume (bright tubes on soft tissue, so black_ridges=False selects them).  The float32
volume is the int16 one mapped to (HU + 1024) / 4096.  Per case: ms per call; the float64 operations of the line
passes (float64 for every image type, as scipy's lines are), counted exactly from shapes and radii (1 + 3 r per
output: one product for the centre tap, then an add or subtract, a product and an add per pair), and of the epilogue (an estimate: the 2x2 closed form and formula, or four Jacobi sweeps
of three rotations for 3x3); the bytes the passes and epilogues move if every pass read its input and wrote its output
exactly once (the workspace is larger than the 126 MB L2, so this is a floor, not a count of the traffic); that floor
at 7.7 TB/s (HBM3e data-sheet bandwidth of one B200, not a measured figure); the workspace bytes; and the twin's time on
a 128^3 sub-volume (16 planes for the plane case), scaled by the voxel ratio and labelled as scaled."""
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
import sk_ridges_twin as T  # noqa: E402
from mie_b200 import _ffi, skimage_compat as S, synthetic  # noqa: E402
from tv_chambolle_quick import card, kernel_times, timed  # noqa: E402

HBM_BYTES_S = 7.7e12
DEFAULT_SIGMAS = list(range(1, 10, 2))
JACOBI_OPS = 4 * 3 * 30   # four sweeps of three rotations of ~30 float64 operations


def counts(kind, shape_img, n, sigmas, src_bytes, fsz):
    """(pass ops, epilogue ops, bytes) of one call on n images of shape_img."""
    vox = int(np.prod(shape_img)) * n
    ndim = len(shape_img)
    passes = 24 if ndim == 3 else 10
    src_passes = 3 if ndim == 3 else 2      # passes that read the source instead of a float buffer
    nel = 6 if ndim == 3 else 3
    ops = 0
    nbytes = 0
    for s in sigmas:
        r = int(4 * s + 0.5)
        ops += passes * vox * (1 + 3 * r)
        nbytes += src_passes * vox * (src_bytes + fsz) + (passes - src_passes) * vox * 2 * fsz
        nbytes += vox * (nel + 2) * fsz      # epilogue: the elements, the running maximum read and written
    per_voxel = (JACOBI_OPS if ndim == 3 else 8) + 25
    epi = len(sigmas) * vox * per_voxel * (2 if kind == "meijering" else 1)
    return ops, epi, nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    vol_np = synthetic.vessel_volume((512, 512, 512), np.int16, 0)
    vol = torch.from_numpy(vol_np).to(dev)
    f32 = ((vol.to(torch.float32) + 1024.0) / 4096.0).contiguous()
    planes_np = synthetic.vessel_volume((256, 512, 512), np.uint16, 1)
    planes = torch.from_numpy(planes_np).to(dev)
    cases = [("frangi 512^3 i16 volumetric default sigmas black_ridges=False", "frangi", vol, True),
             ("frangi 512^3 f32 volumetric default sigmas black_ridges=False", "frangi", f32, True),
             ("sato 512^3 i16 volumetric default sigmas black_ridges=False", "sato", vol, True),
             ("frangi 256 x 512^2 u16 planes default sigmas black_ridges=False", "frangi", planes, False)]
    records = []
    lib = _ffi.lib()
    for name, kind, x, volumetric in cases:
        code = _ffi.DTYPE_CODE[x.dtype]
        fsz = 4 if x.dtype == torch.float32 else 8
        if volumetric:
            ws = lib.mie_sk_ridge_filter3d_workspace_bytes(1, 512, 512, 512, code)
            shape_img, n = (512, 512, 512), 1
        else:
            ws = lib.mie_sk_ridge_filter_workspace_bytes(x.shape[0], 512, 512, code)
            shape_img, n = (512, 512), x.shape[0]
        fn = getattr(S, kind)

        def call(x=x, fn=fn, volumetric=volumetric):
            return fn(x, black_ridges=False, volumetric=volumetric)

        ms = timed(call, 3)
        kt = kernel_times(call, 1)
        out = call()
        out_max = float(out.max())
        del out
        pass_ops, epi_ops, nbytes = counts(kind, shape_img, n, DEFAULT_SIGMAS, x.element_size(), fsz)
        floor_ms = nbytes / HBM_BYTES_S * 1e3
        sub = x[:128, :128, :128].cpu().numpy() if volumetric else x[:16].cpu().numpy()
        t0 = time.perf_counter()
        if volumetric:
            getattr(T, kind)(sub, black_ridges=False)
        else:
            for i in range(sub.shape[0]):
                getattr(T, kind)(sub[i], black_ridges=False)
        twin_s = time.perf_counter() - t0
        scale = x.numel() / sub.size
        rec = {"case": name, "ms": round(ms, 2), "out_max": out_max,
               "pass_ops": pass_ops, "pass_ops_type": "f64",
               "epilogue_ops_estimate": epi_ops, "epilogue_ops_type": "f32" if fsz == 4 else "f64",
               "pass_gops_per_s": round(pass_ops / ms / 1e6, 1), "bytes_floor": nbytes,
               "bytes_floor_ms": round(floor_ms, 2), "of_bytes_floor": round(floor_ms / ms, 3),
               "workspace_bytes": ws, "twin_cpu_s_subset": round(twin_s, 2),
               "twin_cpu_subset": "128^3" if volumetric else "16 planes",
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
