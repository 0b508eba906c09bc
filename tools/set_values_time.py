"""Time of replacing a plan's values in place on the device (b200_interp2_plan_set_values_dev /
b200_interp1_plan_set_values_dev), against what a caller pays without it: destroying the plan and creating a new one
from the same grid.

Each case is timed with CUDA events over --calls calls (default 200) that alternate between two source buffers:
  eager  the C-ABI called from a tight ctypes loop on one stream (what a Python caller gets);
  graph  the same calls captured once into a CUDA graph and replayed (launch overhead removed).
The 4096^2 sources are 128 MiB (f64) / 64 MiB (f32) each, so two of them and the plan's tables do not fit the 126 MB
L2; the interp1 case (8 MB sources) is launch-sized and runs from L2.  The floor of a case is its bytes (read + write,
every byte once; halo re-reads are expected to hit L2) over the measured HBM copy peak (MEASURED_PEAKS.json when
present, else 6537 GB/s, the figure measured on B200 that DESIGN.md quotes).  Destroy + create is timed with the host
clock from a pageable column-major numpy Z, median of --reps.

    python tools/set_values_time.py --out profiles/set_values_b200.md
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def copy_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json"
    return 6537.0, "6537 GB/s (measured HBM copy peak quoted in DESIGN.md)"


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return out[0].strip()


def per_call_us(torch, calls, enqueue):
    """enqueue(i) queues call i on the current stream; returns (eager us/call, graph us/call)."""
    for i in range(4):
        enqueue(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(calls):
        enqueue(i)
    b.record()
    b.synchronize()
    eager = a.elapsed_time(b) * 1e3 / calls
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(calls):
            enqueue(i)
    g.replay()
    torch.cuda.synchronize()
    a.record()
    g.replay()
    b.record()
    b.synchronize()
    return eager, a.elapsed_time(b) * 1e3 / calls


def create_destroy_ms(make, reps):
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        p = make()
        p.close()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096, help="interp2 grid: n x n")
    ap.add_argument("--ng", type=int, default=1_000_000, help="interp1 knots")
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="markdown report (a .json with the same stem is written beside it)")
    args = ap.parse_args()

    import torch
    import armadillocudalinearinterpolation_b200 as B
    from armadillocudalinearinterpolation_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs a B200")
    lib = _lib.lib()
    gpu = card()
    peak, peak_src = copy_peak()
    n, calls = args.n, args.calls
    rows = []

    P = B.Interp2Plan
    x = np.linspace(0.0, 1.0, n); y = np.linspace(0.0, 1.0, n)
    ntile = ((n - 1) // 3 + 1) ** 2
    for label, dt, flags, table_bytes in (
            ("interp2 f64, default plan (tiles)", np.float64, 0, ntile * 16 * 8),
            ("interp2 f64, FORCE_CELLS (records)", np.float64, P.FORCE_CELLS, n * n * 4 * 8),
            ("interp2 f32, default plan (column-major only)", np.float32, 0, 0)):
        esz = np.dtype(dt).itemsize
        tdt = torch.float64 if dt == np.float64 else torch.float32
        z = np.asfortranarray(np.random.default_rng(1).standard_normal((n, n)).astype(dt))
        plan = P(x.astype(dt), y.astype(dt), z, flags=flags)
        nbytes = 2 * n * n * esz + table_bytes
        g = torch.Generator(device="cuda").manual_seed(2)
        for order in ("column-major", "row-major"):
            if order == "column-major":
                src = [torch.randn((n, n), generator=g, device="cuda", dtype=tdt).t() for _ in range(2)]
                ld, rm = n, 0
            else:
                src = [torch.randn((n, n), generator=g, device="cuda", dtype=tdt) for _ in range(2)]
                ld, rm = n, 1
            ptr = [C.c_void_p(s.data_ptr()) for s in src]

            def enqueue(i):
                st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                _lib.check(lib.b200_interp2_plan_set_values_dev(plan._h, ptr[i & 1], C.c_size_t(ld), C.c_int(rm), st))
            eager, graph = per_call_us(torch, calls, enqueue)
            rows.append(dict(case=label, source=order, bytes=nbytes, eager_us=eager, graph_us=graph))
            del src
        plan.close()
        zx, zy = x.astype(dt), y.astype(dt)
        rows.append(dict(case=label, source="destroy + create (host Z)", bytes=None,
                         create_ms=create_destroy_ms(lambda: P(zx, zy, z, flags=flags), args.reps)))
        del z
        torch.cuda.empty_cache()

    ng = args.ng
    xg = np.linspace(0.0, 1.0, ng)
    yg = np.sin(2 * np.pi * xg)
    p1 = B.Interp1Plan(xg, yg)
    src = [torch.randn(ng, device="cuda", dtype=torch.float64) for _ in range(2)]
    ptr = [C.c_void_p(s.data_ptr()) for s in src]

    def enqueue1(i):
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(lib.b200_interp1_plan_set_values_dev(p1._h, ptr[i & 1], st))
    eager, graph = per_call_us(torch, calls, enqueue1)
    label = f"interp1 f64, {ng} knots (lookup mode {p1.lookup_mode})"
    rows.append(dict(case=label, source="device vector", bytes=ng * (8 + 8 + 32), eager_us=eager, graph_us=graph))
    p1.close()
    rows.append(dict(case=label, source="destroy + create (host Y)", bytes=None,
                     create_ms=create_destroy_ms(lambda: B.Interp1Plan(xg, yg), args.reps)))

    lines = [f"# set_values_dev: plan values replaced in place ({n}^2 interp2, {ng}-knot interp1)", "",
             f"Card: {gpu} (name, power limit; read by nvidia-smi in the same run).  Copy peak: {peak:.0f} GB/s "
             f"({peak_src}).  {calls} calls per case alternating two sources; CUDA events.", "",
             "| case | source | bytes (MB) | floor (us) | eager (us/call) | graph (us/call) | floor / graph | destroy + create (ms) |",
             "|---|---|---|---|---|---|---|---|"]
    for r in rows:
        if r.get("bytes"):
            floor = r["bytes"] / (peak * 1e9) * 1e6
            r["floor_us"] = floor
            r["frac_of_floor"] = floor / r["graph_us"]
            lines.append(f"| {r['case']} | {r['source']} | {r['bytes'] / 1e6:.0f} | {floor:.1f} | {r['eager_us']:.1f} | "
                         f"{r['graph_us']:.1f} | {r['frac_of_floor']:.2f} | |")
        else:
            lines.append(f"| {r['case']} | {r['source']} | | | | | | {r['create_ms']:.1f} |")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
        with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
            json.dump(dict(card=gpu, copy_peak_gbs=peak, copy_peak_source=peak_src, calls=calls, rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
