#!/usr/bin/env python
"""skimage.restoration.denoise_tv_chambolle on the GPU (skimage_compat.denoise_tv_chambolle): CUDA-event timing of
one call, the device time of each kernel from a separate torch.profiler pass, and a torch-eager transcription of the
numpy twin (tests/sk_tv_chambolle_twin.py; one host synchronisation per pass for the stopping test) on the same input.
    python benchmarks/tv_chambolle_quick.py [--out FILE.jsonl]

Per case: passes run; ms per call and per pass; the bytes floor of one pass, computed from shapes as
(2 * ndim * sizeof(float type) + sizeof(src)) bytes per voxel — p read once and written once, the source read once — at
7.7 TB/s (HBM3e data-sheet bandwidth of one B200, not a measured figure), and the fraction of it the pass kernel
reaches; and what the launches after every image has stopped cost: the default max_num_iter=200 call against the
same call with max_num_iter = the passes actually run (same result).  The eps=0, max_num_iter=50 cases run a fixed
number of passes and give the per-pass time directly."""
import argparse
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
    line = q.stdout.strip().splitlines()[0] if q.stdout else q.stderr.strip()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": line}


def timed(fn, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_times(fn, reps=2):
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
            out[ev.key[:60]] = (round(t / reps / 1e3, 4), ev.count // reps)   # (ms per call, launches per call)
    return dict(sorted(out.items(), key=lambda kv: -kv[1][0]))


def eager_tv(image, weight=0.1, eps=2e-4, max_num_iter=200):
    """torch-eager transcription of the twin on one image (float64 / float32 as given)."""
    ndim = image.dim()
    p = torch.zeros((ndim,) + tuple(image.shape), dtype=image.dtype, device=image.device)
    g = torch.zeros_like(p)
    d = torch.zeros_like(image)
    i = 0
    while i < max_num_iter:
        if i > 0:
            d = -p.sum(0)
            for ax in range(ndim):
                d.narrow(ax, 1, image.shape[ax] - 1).add_(p[ax].narrow(ax, 0, image.shape[ax] - 1))
            out = image + d
        else:
            out = image
        E = (d ** 2).sum()
        for ax in range(ndim):
            g[ax].narrow(ax, 0, image.shape[ax] - 1).copy_(torch.diff(out, dim=ax))
        norm = torch.sqrt((g ** 2).sum(0))[None]
        E = E + weight * norm.sum()
        tau = 1.0 / (2.0 * ndim)
        norm *= tau / weight
        norm += 1.0
        p -= tau * g
        p /= norm
        E = float(E) / image.numel()
        if i == 0:
            e_init = e_prev = E
        elif abs(e_prev - E) < eps * e_init:
            break
        else:
            e_prev = E
        i += 1
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = card()
    print(json.dumps(info), flush=True)
    v = synthetic.phantom_volume((512, 512, 512), np.int16, 0)
    vol_i16 = torch.from_numpy(v).to(dev)
    vol_f32 = ((vol_i16.to(torch.float64) * 2.0 + 1.0) / 65535.0).to(torch.float32)   # img_as_float scale
    del v
    planes = torch.from_numpy(synthetic.phantom((256, 1, 512, 512), np.uint16, 0)).to(dev)
    cases = [("512^3 i16 volumetric", vol_i16, True), ("512^3 f32 volumetric", vol_f32, True),
             ("256 x 512^2 u16 planes", planes, False)]
    records = []
    for name, x, volumetric in cases:
        ndim = 3 if volumetric else 2
        n = x.numel() // (x.shape[-1] * x.shape[-2] * (x.shape[-3] if volumetric else 1))
        fsz = 4 if x.dtype == torch.float32 else 8
        floor_ms = x.numel() * (2 * ndim * fsz + x.element_size()) / HBM_BYTES_S * 1e3
        for kw in (dict(), dict(eps=0.0, max_num_iter=50)):
            iters = torch.zeros(n, dtype=torch.int32, device=dev)

            def call(kw=kw, iters=iters):
                return S._denoise_tv_chambolle(x, kw.get("weight", 0.1), kw.get("eps", 2e-4), kw.get("max_num_iter", 200),
                                               None, None, volumetric, iters)

            ms = timed(call, 3)
            its = iters.cpu().numpy()
            passes = int(its.max())
            kt = kernel_times(call)
            pass_ms = sum(t for k, (t, _) in kt.items() if "sk_tv_pass" in k)
            pass_launches = sum(c for k, (_, c) in kt.items() if "sk_tv_pass" in k)
            rec = {"case": name + (" eps=0 max_num_iter=50" if kw else " default"), "passes_run": passes,
                   "passes_run_min": int(its.min()), "ms": round(ms, 3), "ms_per_pass": round(ms / passes, 4),
                   "pass_kernel_ms_total": round(pass_ms, 3), "pass_launches": pass_launches,
                   "bytes_floor_ms_per_pass": round(floor_ms, 4), "kernels_ms": kt}
            if kw:   # every launch does full work: kernel time per pass against the floor
                rec["pass_kernel_ms_per_pass"] = round(pass_ms / pass_launches, 4)
                rec["of_bytes_floor"] = round(floor_ms / (pass_ms / pass_launches), 3)
            else:    # the launches after the last image stopped
                ms_exact = timed(lambda: S._denoise_tv_chambolle(x, 0.1, 2e-4, passes, None, None, volumetric, None), 3)
                rec["ms_with_max_num_iter_eq_passes"] = round(ms_exact, 3)
                rec["post_convergence_launches_ms"] = round(ms - ms_exact, 3)
                if n == 1:
                    img = x.to(torch.float64) * 2.0 + 1.0 if x.dtype == torch.int16 else x
                    img = img / 65535.0 if x.dtype == torch.int16 else img
                    rec["eager_torch_ms"] = round(timed(lambda: eager_tv(img), 1), 2)
                    rec["speedup_vs_eager"] = round(rec["eager_torch_ms"] / ms, 2)
                    ref = eager_tv(img)
                    rec["max_abs_diff_vs_eager"] = float((call().to(torch.float64) - ref.to(torch.float64)).abs().max())
                    del ref
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
