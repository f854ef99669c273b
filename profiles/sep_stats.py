import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gym-soccer-2d-env_b200")); sys.path.insert(0, ROOT)
import torch, bench
from soccer2d_b200 import Soccer2DVecEnv
n=1<<16; dev=torch.device("cuda:0")
gen=torch.Generator(device=dev).manual_seed(99)
env=Soccer2DVecEnv(n, scenario="fullgame", device=dev, seed=0, substeps=1)
env.reset_torch()
prev=None
for c in range(1,61):
    a=bench.commands(torch, gen, dev, (n,1,22))
    env.step_torch(a)
    if c in (5,10,15,20,30,40,50,60):
        pl=env.fullgame_planes(); sep=pl["ef"][:n,1].clone()
        # a scan happened this cycle if sep was re-measured: can't see directly; report distribution
        q=torch.quantile(sep, torch.tensor([0.1,0.25,0.5,0.75,0.9],device=dev))
        print(c, "sep quantiles", [round(float(x),2) for x in q], "frac sep<0.6+1.0:", float((sep<1.6).float().mean()), "frac<0.6:", float((sep<0.6).float().mean()), "frac sep<2.6", float((sep<2.6).float().mean()))
