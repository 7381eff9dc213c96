import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import mie_b200
from mie_b200 import synthetic
from mie_b200.loader import HostSlicePipeline
dev = torch.device("cuda:0")
x_host = torch.from_numpy(synthetic.phantom((256, 1, 512, 512), np.uint16, seed=0)).pin_memory()
y_host = torch.empty_like(x_host).pin_memory()
# raw PCIe numbers
xd = torch.empty_like(x_host, device=dev)
for name, fn in (("h2d", lambda: xd.copy_(x_host, non_blocking=True)), ("d2h", lambda: y_host.copy_(xd, non_blocking=True))):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): fn()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print(name, round(ms, 3), "ms", round(134.2 / ms, 1), "GB/s")
for chunk in (64, 32, 16):
    for depth, taper in ((3, False), (3, True), (4, True)):
        pipe = HostSlicePipeline(dev, (512, 512), torch.uint16, chunk=chunk, depth=depth, taper=taper)
        for _ in range(2): pipe.run(x_host, y_host)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(5): pipe.run(x_host, y_host)
        e1.record(); torch.cuda.synchronize()
        ok = bool((y_host == ref).all()) if "ref" in globals() else None
        if "ref" not in globals(): ref = y_host.clone()
        print("chunk", chunk, "depth", depth, "taper", taper, "same-as-first", ok, round(e0.elapsed_time(e1) / 5, 3), "ms; wall", round((time.perf_counter() - t0) / 5 * 1e3, 3))
