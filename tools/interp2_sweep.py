import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import armadillocudalinearinterpolation_b200 as B
NQ = 50_000_000
g = torch.Generator(device="cuda").manual_seed(1)
xq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
yq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
zq = torch.empty_like(xq)
prop = torch.cuda.get_device_properties(0)
print("L2", prop.L2_cache_size / 2**20, "MiB")
for dt in (np.float64, np.float32):
  xq_, yq_, zq_ = (xq, yq, zq) if dt == np.float64 else (xq.float(), yq.float(), zq.float())
  for n in (1024, 2048, 2560, 2896, 3200, 3584, 4096, 5792):
    x = np.linspace(0, 1, n).astype(dt); z = np.random.default_rng(0).standard_normal((n, n)).astype(dt)
    for zpol in ("1", "0"):
        os.environ.update({"B200_INTERP2_SMEM": "0", "B200_INTERP2_CELLS": "0", "B200_INTERP2_ZPOL": zpol})
        plan = B.Interp2Plan(x, x, z)
        for _ in range(3): plan.scattered(xq_, yq_, out=zq_)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5): plan.scattered(xq_, yq_, out=zq_)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        print(f"{dt.__name__} n={n:5d} Z={n*n*np.dtype(dt).itemsize/2**20:7.1f} MiB zpol={zpol}  {ms:7.3f} ms  {NQ/ms/1e6:7.2f} Gpts/s", flush=True)
        plan.close()
