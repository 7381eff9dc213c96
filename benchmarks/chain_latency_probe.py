import os, sys; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, mie_b200 as M
from mie_b200 import synthetic
for nb in (1,2,4,8,16,32):
    x=torch.from_numpy(synthetic.phantom((nb,1,512,512),np.uint16,0)).cuda()
    p=M.ChainPlan(x)
    for _ in range(5): p.replay()
    torch.cuda.synchronize(); e0=torch.cuda.Event(enable_timing=True); e1=torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200): p.replay()
    e1.record(); torch.cuda.synchronize(); print("batch",nb, round(e0.elapsed_time(e1)/200*1e3,1),"us")
