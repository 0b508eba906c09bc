"""Time of the derivative calls of scattered interp2 on the headline plan (4096^2 f64, linspace axes, 4x4 tiles):
b200_interp2_scattered_dev (value), b200_interp2_scattered_grad_dev (value + gradient) and
b200_interp2_scattered_adjoint_dev (G = W^T g), on device buffers, for uniformly random and cell-sorted queries.

Call times are CUDA events over --calls back-to-back calls on one stream.  The adjoint's stages (keys, CUB radix sort,
segment offsets, terms, nodes) are kernel durations from torch.profiler over one call; the sort's kernels are
cub::DeviceRadixSort::SortPairs itself on the pipeline's keys, the floor of this algorithm.  Achieved bandwidth of the
other stages is their algorithmic bytes (every byte once, gathers counted at their useful size) over their time,
against the HBM copy peak (MEASURED_PEAKS.json when present, else 6537 GB/s).  Also the degenerate adjoint: every
query in one cell (the four nodes add their terms serially).

    python tools/interp2_grad_time.py --out profiles/interp2_grad_b200.md
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
    for _ in range(2):
        enqueue()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        enqueue()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / calls


STAGES = (("keys", "adjoint_keys_kernel"), ("sort", "cub"), ("offsets", "adjoint_offsets_kernel"),
          ("terms", "adjoint_terms_kernel"), ("nodes", "adjoint_nodes_kernel"))


def stage_ms(torch, enqueue):
    """Kernel time per adjoint stage (ms) from one profiled call."""
    from torch.profiler import ProfilerActivity, profile
    enqueue()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        enqueue()
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
    ap.add_argument("--nq", type=int, default=100_000_000)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    import armadillocudalinearinterpolation_b200 as B
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    peak = copy_peak()
    x, y, z = bench.make_grid()
    nx, ny = x.size, y.size
    plan = B.Interp2Plan(x, y, z)
    nq = args.nq
    gen = torch.Generator(device="cuda").manual_seed(1)
    xq = torch.rand(nq, generator=gen, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0]
    yq = torch.rand(nq, generator=gen, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0]
    g = torch.randn(nq, generator=gen, device="cuda", dtype=torch.float64)
    cell = ((xq - x[0]) / (x[-1] - x[0]) * (nx - 1)).floor() * ny + ((yq - y[0]) / (y[-1] - y[0]) * (ny - 1)).floor()
    o = cell.argsort()
    sets = {"random": (xq, yq), "cell-sorted": (xq[o].contiguous(), yq[o].contiguous())}
    del cell, o
    zq, dx, dy = (torch.empty_like(xq) for _ in range(3))
    G = torch.empty((ny, nx), dtype=torch.float64, device="cuda")
    need = C.c_size_t()
    _lib.check(lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(nq), C.byref(need)))
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr())

    def stream():
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def adjoint(qx, qy, gg, n):
        _lib.check(lib.b200_interp2_scattered_adjoint_dev(plan._h, P(qx), P(qy), P(gg), C.c_size_t(n), P(G), C.c_size_t(nx), 1,
                                                       P(ws), C.c_size_t(need.value), stream()))

    rows, raw = [], {"card": card(), "nq": nq, "calls": args.calls, "peak_gbs": peak, "cases": {}}
    for name, (qx, qy) in sets.items():
        t_val = ms_per_call(torch, args.calls, lambda: _lib.check(lib.b200_interp2_scattered_dev(
            plan._h, P(qx), P(qy), C.c_size_t(nq), P(zq), C.c_double(np.nan), stream())))
        t_grad = ms_per_call(torch, args.calls, lambda: _lib.check(lib.b200_interp2_scattered_grad_dev(
            plan._h, P(qx), P(qy), C.c_size_t(nq), P(zq), P(dx), P(dy), C.c_double(np.nan), stream())))
        t_adj = ms_per_call(torch, args.calls, lambda: adjoint(qx, qy, g, nq))
        st = stage_ms(torch, lambda: adjoint(qx, qy, g, nq))
        raw["cases"][name] = dict(value_ms=t_val, grad_ms=t_grad, adjoint_ms=t_adj, stages_ms=st)
        rows.append((name, t_val, t_grad, t_adj, st))
    # the degenerate adjoint: every query in one cell
    degen = {}
    for n1 in (1_000_000, 10_000_000):
        xs = torch.full((n1,), float(x[100] + 0.3 * (x[101] - x[100])), dtype=torch.float64, device="cuda")
        ys = torch.full((n1,), float(y[7] + 0.6 * (y[8] - y[7])), dtype=torch.float64, device="cuda")
        degen[n1] = ms_per_call(torch, 3, lambda: adjoint(xs, ys, g, n1))
    raw["one_cell_ms"] = degen

    ncells = nx * ny
    stage_bytes = {"keys": 24.0 * nq, "offsets": 4.0 * (ncells + 1), "terms": 64.0 * nq, "nodes": 32.0 * nq + 12.0 * ncells}
    extra_floor_ms = 16.0 * nq / (peak * 1e9) * 1e3
    lines = [f"# interp2 derivatives on the headline plan ({raw['card']})", "",
             f"4096^2 f64, linspace axes, 4x4 tiles; {nq:.0e} device queries; CUDA events over {args.calls} calls; "
             f"copy peak {peak:.0f} GB/s.  `python tools/interp2_grad_time.py` (raw: interp2_grad_b200.json).", "",
             "| queries | value call | gradient call | gradient - value | 16 B/query at copy peak | adjoint |",
             "|---|---|---|---|---|---|"]
    for name, tv, tg, ta, _ in rows:
        lines.append(f"| {name} | {tv:.3f} ms | {tg:.3f} ms | {tg - tv:+.3f} ms | {extra_floor_ms:.3f} ms | {ta:.3f} ms |")
    lines += ["", "Adjoint stages (one profiled call; achieved = algorithmic bytes / time):", "",
              "| queries | stage | time | bytes | achieved | of copy peak |", "|---|---|---|---|---|---|"]
    for name, _, _, _, st in rows:
        for k, _ in STAGES:
            if k == "sort":
                lines.append(f"| {name} | sort (CUB SortPairs, the floor) | {st[k]:.3f} ms | | | |")
            else:
                gbs = stage_bytes[k] / (st[k] * 1e-3) / 1e9 if st[k] > 0 else float("nan")
                lines.append(f"| {name} | {k} | {st[k]:.3f} ms | {stage_bytes[k] / 1e9:.2f} GB | {gbs:.0f} GB/s | "
                             f"{gbs / peak:.2f} |")
    lines += ["", "Degenerate adjoint, every query in one cell: " +
              ", ".join(f"{n:.0e} queries {t:.1f} ms" for n, t in degen.items()), ""]
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text)
        with open(os.path.splitext(args.out)[0] + ".json", "w") as f:
            json.dump(raw, f, indent=1, default=str)


if __name__ == "__main__":
    main()
