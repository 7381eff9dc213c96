import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, mie_b200 as M
from mie_b200 import synthetic
x=torch.from_numpy(synthetic.phantom_volume((1,512,512),np.int16,0)).cuda().unsqueeze(1)
for vr in (None,(-1024.0,3071.0),(-1000.5,3000.0)):
    p=M.ChainPlan(x, M.ChainConfig(value_range=vr))
    for _ in range(5): p.replay()
    torch.cuda.synchronize(); e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200): p.replay()
    e1.record(); torch.cuda.synchronize(); print("single slice chain i16 value_range",vr, round(e0.elapsed_time(e1)/200*1e3,1),"us")
