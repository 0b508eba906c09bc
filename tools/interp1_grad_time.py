"""Time of the derivative calls of interp1 on device buffers: b200_interp1_exec_dev (value), b200_interp1_grad_dev (value
+ slope) and b200_interp1_adjoint_dev (G = W^T g), for the lookup modes of BASELINE config 1 and the shared-memory path.

Cases: 1e6 f64 knots, linspace (mode 0) and ragged (mode 1), x 1e7 and 1e8 queries, sorted and unsorted; 1e3 linspace
knots x 1e8 unsorted queries (mode 2); 1e6 f32 linspace knots x 1e8 unsorted queries.  Call times are CUDA events over
--calls back-to-back calls on one stream.  At 1e7 queries every call takes the next of 8 rotating buffer sets (as
bench.py does), so the streams are never L2-resident; 1e8-query streams are far larger than L2.  The adjoint's stages
(keys, CUB radix sort, segment offsets, terms, levels of the blocked sum) are kernel durations from torch.profiler over
one call; the sort's kernels are cub::DeviceRadixSort::SortPairs itself on the pipeline's keys.  Gradient - value is set
against the 8 extra bytes per f64 query (4 per f32 query) at the HBM copy peak (MEASURED_PEAKS.json when present, else
6537 GB/s).  Also the adjoint of 1e8 queries that all fall in one segment, on the 1e3-knot plan, beside the uniformly
spread 1e8 adjoint on that plan.

    python tools/interp1_grad_time.py --out profiles/interp1_grad_b200.md
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def copy_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"])
    return 6537.0


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return out[0].strip()


def ms_per_call(torch, calls, enqueue):
    for r in range(2):
        enqueue(r)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for r in range(calls):
        enqueue(r)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls


STAGES = (("keys", "interp1_adjoint_keys_kernel"), ("sort", "cub"), ("offsets", "adjoint_offsets_kernel"),
          ("terms", "interp1_adjoint_terms_kernel"), ("sum", "interp1_adjoint_level_kernel"))


def stage_ms(torch, enqueue):
    """Kernel time per adjoint stage (ms) from one profiled call."""
    from torch.profiler import ProfilerActivity, profile
    enqueue(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        enqueue(0)
        torch.cuda.synchronize()
    out = {k: 0.0 for k, _ in STAGES}
    for e in prof.key_averages():
        us = getattr(e, "self_device_time_total", None)
        if us is None:
            us = getattr(e, "self_cuda_time_total", 0.0)
        for k, pat in STAGES:
            if pat in e.key and "cudaLaunch" not in e.key:
                out[k] += us / 1e3
                break
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import armadillocudalinearinterpolation_b200 as B
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    peak = copy_peak()
    P = lambda t: C.c_void_p(t.data_ptr())

    def stream():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    rng = np.random.default_rng(0)
    grids = {
        "1e6 linspace f64": np.linspace(0.0, 1.0, 1_000_000),
        "1e6 ragged f64": None,
        "1e3 linspace f64": np.linspace(0.0, 1.0, 1000),
        "1e6 linspace f32": np.linspace(0.0, 1.0, 1_000_000).astype(np.float32),
    }
    xr = np.cumsum(0.3 + rng.random(1_000_000))
    grids["1e6 ragged f64"] = (xr - xr[0]) / (xr[-1] - xr[0])
    cases = [("1e6 linspace f64", nq, order) for nq in (10_000_000, 100_000_000) for order in ("sorted", "unsorted")]
    cases += [("1e6 ragged f64", nq, order) for nq in (10_000_000, 100_000_000) for order in ("sorted", "unsorted")]
    cases += [("1e3 linspace f64", 100_000_000, "unsorted"), ("1e6 linspace f32", 100_000_000, "unsorted")]

    raw = {"card": card(), "calls": args.calls, "peak_gbs": peak, "cases": [], "one_segment": {}}
    gen = torch.Generator(device="cuda").manual_seed(1)
    for gname, nq, order in cases:
        x = grids[gname]
        tdt = torch.float64 if x.dtype == np.float64 else torch.float32
        plan = B.Interp1Plan(x, np.sin(7 * x.astype(np.float64)).astype(x.dtype))
        nrot = 8 if nq <= 10_000_000 else 1
        sets = []
        for _ in range(nrot):
            xi = torch.rand(nq, generator=gen, device="cuda", dtype=torch.float64).to(tdt)
            if order == "sorted":
                xi = torch.sort(xi).values
            sets.append((xi, torch.randn(nq, generator=gen, device="cuda", dtype=tdt), torch.empty_like(xi),
                         torch.empty_like(xi)))
        need = C.c_size_t()
        _lib.check(lib.b200_interp1_adjoint_workspace(plan._h, C.c_size_t(nq), C.byref(need)))
        ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
        G = torch.empty(x.size, dtype=tdt, device="cuda")

        def value(r):
            xi, _, yi, _ = sets[r % nrot]
            _lib.check(lib.b200_interp1_exec_dev(plan._h, P(xi), C.c_size_t(nq), P(yi), None, C.c_double(np.nan),
                                                 stream()))

        def grad(r):
            xi, _, yi, dy = sets[r % nrot]
            _lib.check(lib.b200_interp1_grad_dev(plan._h, P(xi), C.c_size_t(nq), P(yi), P(dy), C.c_double(np.nan),
                                                 stream()))

        def adjoint(r, xs=None):
            xi, g, _, _ = sets[r % nrot]
            _lib.check(lib.b200_interp1_adjoint_dev(plan._h, P(xi if xs is None else xs), P(g), C.c_size_t(nq), P(G),
                                                    P(ws), C.c_size_t(need.value), stream()))

        rec = dict(grid=gname, nq=nq, order=order, mode=plan.lookup_mode,
                   value_ms=ms_per_call(torch, args.calls, value), grad_ms=ms_per_call(torch, args.calls, grad),
                   adjoint_ms=ms_per_call(torch, args.calls, adjoint), stages_ms=stage_ms(torch, adjoint),
                   extra_floor_ms=(8.0 if tdt == torch.float64 else 4.0) * nq / (peak * 1e9) * 1e3)
        raw["cases"].append(rec)
        print(json.dumps(rec), flush=True)
        if gname == "1e3 linspace f64":
            xs = torch.full((nq,), float(x[400] + 0.37 * (x[401] - x[400])), dtype=tdt, device="cuda")
            xs += torch.rand(nq, generator=gen, device="cuda", dtype=tdt) * float(0.5 * (x[401] - x[400]))
            t1 = ms_per_call(torch, args.calls, lambda r: adjoint(r, xs))
            raw["one_segment"] = dict(nq=nq, adjoint_ms=t1, spread_adjoint_ms=rec["adjoint_ms"],
                                      stages_ms=stage_ms(torch, lambda r: adjoint(r, xs)))
            print(json.dumps(raw["one_segment"]), flush=True)
            del xs
        del sets, ws, G
        plan.close()
        torch.cuda.empty_cache()

    lines = [f"# interp1 derivatives ({raw['card']})", "",
             f"Device buffers; CUDA events over {args.calls} calls; 1e7-query cases rotate 8 buffer sets; copy peak "
             f"{peak:.0f} GB/s.  `python tools/interp1_grad_time.py` (raw: interp1_grad_b200.json).", "",
             "| grid | queries | order | mode | value call | gradient call | gradient - value | extra bytes at copy peak "
             "| adjoint |", "|---|---|---|---|---|---|---|---|---|"]
    for c in raw["cases"]:
        lines.append(f"| {c['grid']} | {c['nq']:.0e} | {c['order']} | {c['mode']} | {c['value_ms']:.3f} ms | "
                     f"{c['grad_ms']:.3f} ms | {c['grad_ms'] - c['value_ms']:+.3f} ms | {c['extra_floor_ms']:.3f} ms | "
                     f"{c['adjoint_ms']:.3f} ms |")
    lines += ["", "Adjoint stages (one profiled call; sort = CUB `SortPairs` itself, the floor of this algorithm):", "",
              "| grid | queries | order | keys | sort | offsets | terms | blocked sum |", "|---|---|---|---|---|---|---|---|"]
    for c in raw["cases"]:
        st = c["stages_ms"]
        lines.append(f"| {c['grid']} | {c['nq']:.0e} | {c['order']} | " +
                     " | ".join(f"{st[k]:.3f} ms" for k, _ in STAGES) + " |")
    o = raw["one_segment"]
    if o:
        st = o["stages_ms"]
        lines += ["", f"One segment: {o['nq']:.0e} queries all in one segment of the 1e3-knot plan, adjoint "
                  f"{o['adjoint_ms']:.3f} ms against {o['spread_adjoint_ms']:.3f} ms for uniformly spread queries "
                  f"({o['adjoint_ms'] / o['spread_adjoint_ms']:.2f}x); stages " +
                  ", ".join(f"{k} {st[k]:.3f} ms" for k, _ in STAGES) + "."]
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
        with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
            json.dump(raw, f, indent=1, default=str)


if __name__ == "__main__":
    main()
