"""ncu driver for the kernels outside prof_driver.py: the opt-in banded pipeline and the interp1 shared-memory path."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import armadillocudalinearinterpolation_b200 as B
import bench
plan = B.Interp2Plan(*bench.make_grid(), flags=B.Interp2Plan.FORCE_BANDS)
g = torch.Generator(device="cuda").manual_seed(2235)
xq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
yq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
zq = torch.empty_like(xq)
for _ in range(2): plan.scattered(xq, yq, out=zq)
torch.cuda.synchronize()
plan.close()
xg = np.linspace(-3.0, 3.0, 1000)
p1 = B.Interp1Plan(xg, np.sin(xg))
q = xq * 6.0 - 3.0
for _ in range(2): p1(q, out=zq)
torch.cuda.synchronize()
