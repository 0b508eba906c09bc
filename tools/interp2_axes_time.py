"""Headline kernel with linspace (affine), B200_INTERP_AFFINE=0 (shared-memory tables) and non-uniform axes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import armadillocudalinearinterpolation_b200 as B
n = 4096
z = np.asfortranarray(np.random.default_rng(2234).standard_normal((n, n)))
nq = 100_000_000
g = torch.Generator(device="cuda").manual_seed(2235)
xq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
yq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
zq = torch.empty_like(xq)
r = np.random.default_rng(9)
def cums():
    a = np.cumsum(0.5 + r.random(n)); return (a - a[0]) / (a[-1] - a[0])
for name, x, y, aff in (("linspace, affine", np.linspace(0, 1, n), np.linspace(0, 1, n), "1"),
                        ("linspace, tables in shared memory", np.linspace(0, 1, n), np.linspace(0, 1, n), "0"),
                        ("non-uniform axes (bucket tables in shared memory)", cums(), cums(), "1")):
    os.environ["B200_INTERP_AFFINE"] = aff
    plan = B.Interp2Plan(x, y, z)
    for _ in range(3): plan.scattered(xq, yq, out=zq)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): plan.scattered(xq, yq, out=zq)
    e1.record(); torch.cuda.synchronize()
    print(f"{name}: {e0.elapsed_time(e1) / 10:.3f} ms per 1e8 queries")
    plan.close()
