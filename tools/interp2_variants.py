import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import armadillocudalinearinterpolation_b200 as B
import bench
grid = bench.make_grid()
g = torch.Generator(device="cuda").manual_seed(2235)
NQ = bench.NQ
xq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
yq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
ref = None
def run(tag, env):
    global ref
    for k in ("B200_INTERP2_SMEM", "B200_INTERP2_CELLS", "B200_L2_FETCH"):
        os.environ.pop(k, None)
    os.environ.update(env)
    plan = B.Interp2Plan(*grid)
    zq = torch.empty_like(xq)
    for _ in range(3): plan.scattered(xq, yq, out=zq)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): plan.scattered(xq, yq, out=zq)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    if ref is None: ref = zq.clone()
    same = torch.equal(zq, ref)
    print(f"{tag:40s} {ms:8.3f} ms  {NQ/ms/1e6:8.2f} Gpts/s  alg {2.534e9/ms/1e6:7.1f} GB/s  bit-identical {same}", flush=True)
    plan.close()
run("V0 global tables, col-major Z", {"B200_INTERP2_SMEM": "0", "B200_INTERP2_CELLS": "0"})
run("V1 smem axes, col-major Z", {"B200_INTERP2_SMEM": "1", "B200_INTERP2_CELLS": "0"})
run("V2 smem axes, cells", {"B200_INTERP2_SMEM": "1", "B200_INTERP2_CELLS": "1"})
run("V3 smem axes, cells, L2 fetch 32", {"B200_INTERP2_SMEM": "1", "B200_INTERP2_CELLS": "1", "B200_L2_FETCH": "32"})
run("V1 + L2 fetch 32", {"B200_INTERP2_SMEM": "1", "B200_INTERP2_CELLS": "0", "B200_L2_FETCH": "32"})
run("V0 + L2 fetch 32", {"B200_INTERP2_SMEM": "0", "B200_INTERP2_CELLS": "0", "B200_L2_FETCH": "32"})
run("V2 again, L2 fetch 64", {"B200_INTERP2_SMEM": "1", "B200_INTERP2_CELLS": "1", "B200_L2_FETCH": "64"})
# oracle check on a slice
from oracle import oracle_py as O
zo = O.interp2_scattered(*grid, xq[:200000].cpu().numpy(), yq[:200000].cpu().numpy(), nthreads=8)
print("oracle bit-exact:", np.array_equal(ref[:200000].cpu().numpy(), zo))
