"""Scattered interp2, 1e8 queries: column-major Z vs 2x2 corner records vs overlapping 4x4 tiles, by grid size."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import armadillocudalinearinterpolation_b200 as B
P = B.Interp2Plan
nq = 100_000_000
g = torch.Generator(device="cuda").manual_seed(2235)
xq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
yq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
zq = torch.empty_like(xq)
dts = [np.float32] if (len(sys.argv) > 1 and sys.argv[1] == "f32") else [np.float64]
for dt in dts:
    tq = torch.float64 if dt == np.float64 else torch.float32
    xqq, yqq, zqq = xq.to(tq), yq.to(tq), zq.to(tq)
    for n in ((724, 1024, 1448, 2048, 2896, 3584, 4096, 5793, 8192) if len(sys.argv) < 3 else (4096, 4608, 5120, 5793, 6500)):
        x = np.linspace(0, 1, n).astype(dt); y = np.linspace(0, 1, n).astype(dt)
        z = np.asfortranarray(np.random.default_rng(1).standard_normal((n, n)).astype(dt))
        row = f"{dt.__name__} n={n:5d} |Z|={n * n * z.itemsize / 2**20:7.1f} MiB:"
        ref = None
        for name, flags in (("raw", P.NO_CELLS | P.NO_TILES), ("records", P.FORCE_CELLS), ("tiles", P.FORCE_TILES), ("default", 0)):
            if name == "records" and n > 6000: row += "  records    -  "; continue
            plan = P(x, y, z, flags=flags)
            for _ in range(2): plan.scattered(xqq, yqq, out=zqq)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5): plan.scattered(xqq, yqq, out=zqq)
            e1.record(); torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 5
            if ref is None: ref = zqq.clone()
            ok = torch.equal(ref.view(torch.int64 if dt == np.float64 else torch.int32), zqq.view(torch.int64 if dt == np.float64 else torch.int32))
            row += f"  {name} {ms:6.3f}{'' if ok else ' MISMATCH'}"
            plan.close()
        print(row, flush=True)
