"""Time of the derivative calls of tensor-grid interp2 on the headline plan (4096^2 f64 and f32, linspace axes) at
1e4 x 1e4 sorted outputs, on device buffers:

  * gradient: b200_interp2_grid_dev (value) against b200_interp2_grid_grad_dev (value + both slopes), both pass orders;
  * adjoint: b200_interp2_grid_adjoint_dev against b200_interp2_scattered_adjoint_dev on the 1e8-query mesh (the route a
    user had before), time and workspace bytes, with g column- and row-major;
  * a heavily loaded adjoint: a 16 x 16 Z under 4096 x 4096 outputs (~2.6e5 terms per node, added serially);
  * grid_torch forward + backward (gradients to XI, YI and Z).

Call times are CUDA events over --calls back-to-back calls on one stream after two warm-up calls.  The floors are
bytes only, at the HBM copy peak (MEASURED_PEAKS.json when present, else 6537 GB/s): gradient 3 outputs x 8 B + Z once,
adjoint g once + G once.  The card's name and power limit are read in the same run.

    python tools/interp2_grid_grad_time.py --out profiles/interp2_grid_grad_b200.md
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "interp2_grid_grad_b200.md"))
    args = ap.parse_args()
    import torch
    import bench
    import armadillocudalinearinterpolation_b200 as B
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    peak = copy_peak()
    name = card()
    P = lambda t: C.c_void_p(t.data_ptr())
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rows, res = [], {"card": name, "copy_peak_gbs": peak}
    x, y, z = bench.make_grid()
    n = 10_000
    gen = torch.Generator(device="cuda").manual_seed(1)

    # ---- gradient ----
    for dt, tdt in ((np.float64, torch.float64), (np.float32, torch.float32)):
        esz = np.dtype(dt).itemsize
        tx = torch.sort(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0])[0].to(tdt)
        ty = torch.sort(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0])[0].to(tdt)
        out = [torch.empty(n * n, dtype=tdt, device="cuda") for _ in range(3)]
        for order in (0, B.Interp2Plan.ORDER_YX):
            plan = B.Interp2Plan(x.astype(dt), y.astype(dt), z.astype(dt), flags=order)
            v = ms_per_call(torch, args.calls, lambda: lib.b200_interp2_grid_dev(
                plan._h, P(tx), C.c_size_t(n), P(ty), C.c_size_t(n), P(out[0]), C.c_double(0.0), st()))
            g = ms_per_call(torch, args.calls, lambda: lib.b200_interp2_grid_grad_dev(
                plan._h, P(tx), C.c_size_t(n), P(ty), C.c_size_t(n), *(P(o) for o in out), C.c_double(0.0), st()))
            floor = (3 * n * n * esz + z.size * esz) / (peak * 1e6)
            key = f"grad_{np.dtype(dt).name}_{'yx' if order else 'xy'}"
            res[key] = {"value_ms": v, "grad_ms": g, "floor_ms": floor}
            rows.append(f"| gradient {np.dtype(dt).name}, {'Y first' if order else 'X first'} | value {v:.3f} ms | "
                        f"value + gradient {g:.3f} ms | floor {floor:.3f} ms ({floor / g:.0%}) |")
            plan.close()
        del out

    # ---- adjoint at the benchmark shape, against the scattered adjoint on the mesh ----
    plan = B.Interp2Plan(x, y, z)
    tx = torch.sort(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0])[0]
    ty = torch.sort(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0])[0]
    g = torch.randn(n, n, generator=gen, device="cuda", dtype=torch.float64)   # row-major (nyi, nxi)
    G = torch.empty((y.size, x.size), dtype=torch.float64, device="cuda")
    need = C.c_size_t()
    assert lib.b200_interp2_grid_adjoint_workspace(plan._h, C.c_size_t(n), C.c_size_t(n), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    floor = (g.numel() * 8 + G.numel() * 8) / (peak * 1e6)
    res["adjoint_grid_workspace_bytes"] = need.value
    gc = g.t().contiguous()   # the same g column-major: storage (nxi, nyi)
    for label, gs, ldg, rm in (("g column-major", gc, n, 0), ("g row-major", g, n, 1)):
        t = ms_per_call(torch, args.calls, lambda: lib.b200_interp2_grid_adjoint_dev(
            plan._h, P(tx), C.c_size_t(n), P(ty), C.c_size_t(n), P(gs), C.c_size_t(ldg), rm, P(G),
            C.c_size_t(x.size), 1, P(ws), C.c_size_t(need.value), st()))
        res[f"adjoint_grid_{'row' if rm else 'col'}_ms"] = t
        rows.append(f"| grid adjoint, 1e4 x 1e4, {label} | {t:.3f} ms | workspace {need.value / 1e6:.2f} MB | "
                    f"floor {floor:.3f} ms ({floor / t:.0%}) |")
    xq = tx.repeat_interleave(n); yq = ty.repeat(n); gflat = gc.view(-1)
    assert lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(n * n), C.byref(need)) == 0
    res["adjoint_mesh_workspace_bytes"] = need.value
    ws2 = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    t = ms_per_call(torch, max(3, args.calls // 4), lambda: lib.b200_interp2_scattered_adjoint_dev(
        plan._h, P(xq), P(yq), P(gflat), C.c_size_t(n * n), P(G), C.c_size_t(x.size), 1, P(ws2), C.c_size_t(need.value),
        st()))
    res["adjoint_mesh_ms"] = t
    rows.append(f"| scattered adjoint on the 1e8-query mesh | {t:.3f} ms | workspace {need.value / 1e9:.2f} GB "
                f"(+ {2 * xq.numel() * 8 / 1e9:.1f} GB of mesh coordinates) | |")
    del xq, yq, ws2

    # ---- autograd ----
    XI = tx.clone().requires_grad_(); YI = ty.clone().requires_grad_()
    Zt = torch.from_numpy(np.ascontiguousarray(z)).cuda().requires_grad_()

    def fb():
        out = plan.grid_torch(XI, YI, Zt)
        out.backward(g)
    t = ms_per_call(torch, max(3, args.calls // 4), fb)
    res["grid_torch_fwd_bwd_ms"] = t
    rows.append(f"| grid_torch forward + backward (XI, YI, Z), 1e4 x 1e4 | {t:.3f} ms | | |")
    plan.close()
    del g, gc, G, ws

    # ---- heavily loaded nodes ----
    xs = np.linspace(0.0, 1.0, 16); ys = np.linspace(0.0, 1.0, 16)
    small = B.Interp2Plan(xs, ys, np.random.default_rng(0).standard_normal((16, 16)))
    m = 4096
    tx = torch.linspace(0.0, 1.0, m, dtype=torch.float64, device="cuda"); ty = tx.clone()
    g = torch.randn(m, m, generator=gen, device="cuda", dtype=torch.float64)
    G = torch.empty((16, 16), dtype=torch.float64, device="cuda")
    assert lib.b200_interp2_grid_adjoint_workspace(small._h, C.c_size_t(m), C.c_size_t(m), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    t = ms_per_call(torch, max(3, args.calls // 4), lambda: lib.b200_interp2_grid_adjoint_dev(
        small._h, P(tx), C.c_size_t(m), P(ty), C.c_size_t(m), P(g), C.c_size_t(m), 1, P(G), C.c_size_t(16), 1, P(ws),
        C.c_size_t(need.value), st()))
    res["adjoint_loaded_16x16_ms"] = t
    rows.append(f"| grid adjoint, 16 x 16 Z under 4096 x 4096 (~{4 * (m / 15) ** 2:.1e} terms per interior node) | "
                f"{t:.3f} ms | | |")
    small.close()

    md = [f"# Tensor-grid interp2 derivatives on {name} (name, power limit)", "",
          "Written by `tools/interp2_grid_grad_time.py`; CUDA events over back-to-back calls after warm-up. Headline plan "
          "4096^2 linspace axes; 1e4 x 1e4 sorted outputs. Floors are bytes only at the copy peak "
          f"{peak:.0f} GB/s.", "", "| call | time | | floor |", "|---|---|---|---|"] + rows
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    open(args.out, "w").write("\n".join(md) + "\n")
    json.dump(res, open(os.path.splitext(args.out)[0] + ".json", "w"), indent=1)
    print("\n".join(md))


if __name__ == "__main__":
    main()
