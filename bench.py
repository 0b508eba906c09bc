#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json metric:
"interp points/s & map evals/s at 1/2/4/8 B200; achieved HBM GB/s vs peak").

    python bench.py --gpus N --steps K --warmup W            # this implementation
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # + a seeded sample of the last timed step's outputs

Workload of the headline line (BASELINE.json configs[1]): 2-D bilinear interpolation of a
4096x4096 float64 column-major grid at 1e8 scattered queries per GPU ("step" = one pass over
the 1e8 queries).  `value` is device-resident throughput (CUDA events on the launching stream);
`e2e` is the same pass through the host-buffer C-ABI call b200_interp2_scattered with pinned
host buffers, H2D/D2H inside the timed region.  `extra` carries the other BASELINE configs
(1-D interp at 1e6 knots / 1e7 queries, one map evaluation of the parameters.hpp default
ensemble, the finite-difference Jacobian) measured the same way, shorter.

N > 1: launched by torchrun, one rank per GPU.  The interpolation shards by queries with no
collective (weak scaling: 1e8 queries per rank).  The Jacobian in `extra` shards its
(column, realisation) work items over the ranks and gathers positions with one NCCL all-gather.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NX = NY = 4096
METRIC = "interp points/s (2-D bilinear, 4096x4096 f64 grid, 1e8 scattered queries)"   # both arms
WORKLOAD = "interp2_scattered_f64_4096x4096_1e8_queries_per_gpu"
GRID_DESC = "4096x4096 float64 column-major (128 MiB), seed 2234"
NQ = 100_000_000
ALG_BYTES_PER_QUERY = 24            # xq, yq in + zq out, float64 (SURVEY.md §8d)
ALG_BYTES_GRID = 8 * NX * NY        # the grid is read once
Z_DRIVER = np.array([np.float32(0.3310), np.float32(0.6914), np.float32(1.3557)], dtype=np.float64)
BETA = float(np.float32(13.0589))


def headline_config(n_gpus):
    """`config` of the JSON line — identical for this implementation and for --impl reference
    (the driver compares the two arms' configs)."""
    return {"workload": WORKLOAD,
            "grid": GRID_DESC,
            "queries": "1e8 (x,y) ~ U[0,1]^2 per GPU, unsorted, seed 2235+rank",
            "l2": "inputs larger than L2 (1.6 GB of queries + 0.8 GB of outputs per step)",
            "parallelism": f"query shards x{n_gpus}, no collective"}


def source_stamp(files):
    """sha1 over the kernel sources a static ncu figure was captured for (staleness check)."""
    import hashlib
    h = hashlib.sha1()
    for f in files:
        with open(os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


INTERP2_SOURCES = ("interp2.cu", "interp_common.cuh", "common.cuh")
EDM_SOURCES = ("edm.cu", "common.cuh")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_SAMPLE = 1 << 22               # float64 outputs kept by --dump-outputs: 32 MiB of the 800 MB a step writes
DUMP_SEED = 2238


def dump_outputs(out_dir, torch, zq):
    """Write a fixed, seeded sample of the headline step's outputs to out_dir/interp2_scattered_zq.npy (float64),
    so that two builds run with the same arguments can be compared output for output.  The sample is the
    outputs at the sorted unique indices of DUMP_SAMPLE draws from default_rng(DUMP_SEED).integers(0, NQ)."""
    idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, zq.numel(), DUMP_SAMPLE))
    sample = zq[torch.from_numpy(idx).to(zq.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "interp2_scattered_zq.npy"), sample)


def make_grid():
    rng = np.random.default_rng(2234)
    x = np.linspace(0.0, 1.0, NX)
    y = np.linspace(0.0, 1.0, NY)
    z = np.sin(2 * np.pi * x)[None, :] * np.cos(2 * np.pi * y)[:, None] + 0.1 * rng.standard_normal((NY, NX))
    return x, y, np.asfortranarray(z)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md), through
    NVML (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints):
    the timed region lasts tens of milliseconds, too short for an `nvidia-smi -lms` process."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t = index, [], False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # CUDA_VISIBLE_DEVICES remaps indices; resolve through the PCI bus id of the torch device
            import torch
            bus = torch.cuda.get_device_properties(index).pci_bus_id if hasattr(torch.cuda.get_device_properties(index), "pci_bus_id") else None
            self.h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    h = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(h).bus == bus:
                        self.h = h
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.rows.append((sm, mx, rs, pw))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.t.join(timeout=1)
        sm = [r[0] for r in self.rows]
        reasons = set()
        for r in self.rows:
            for bit, name in self.REASONS.items():
                if r[2] & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(r[1] for r in self.rows)) if sm else None,
                "power_w_max": max((r[3] for r in self.rows), default=None), "samples": len(sm), "reasons": sorted(reasons)}


def cpu_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_interp2(sample, threads, grid=None):
    """The reference-side CPU path for configs[1]: the oracle's restatement of arma::interp2
    applied per scattered point, OpenMP over queries.  Returns points/s."""
    from oracle import oracle_py as O
    x, y, z = grid or make_grid()
    rng = np.random.default_rng(2235)
    xq = rng.random(sample); yq = rng.random(sample)
    O.interp2_scattered(x, y, z, xq[:100000], yq[:100000], nthreads=threads)  # touch + warm
    t = time.perf_counter()
    O.interp2_scattered(x, y, z, xq, yq, nthreads=threads)
    return sample / (time.perf_counter() - t)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  Armadillo is absent
    from the image and the reference has no interp2 call site (SURVEY.md §0), so this is the
    oracle port of arma::interp2's algorithm on all host threads.  One step = a bounded sample
    (2e7 of the 1e8 queries); --warmup W untimed and exactly --steps K timed steps, like the other arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    grid = make_grid()
    sample = 20_000_000
    from oracle import oracle_py as O
    x, y, z = grid
    rng = np.random.default_rng(2235)
    xq = rng.random(sample); yq = rng.random(sample)
    for _ in range(max(args.warmup, 0)):
        O.interp2_scattered(x, y, z, xq, yq, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        O.interp2_scattered(x, y, z, xq, yq, nthreads=threads)
    sec = (time.perf_counter() - t0) / args.steps
    v = sample / sec
    line = {"impl": "reference", "metric": METRIC,
            "value": v, "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": headline_config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "points/s", "cores": threads, "kind": "port",
                             "sample": f"{sample} of the 1e8 scattered queries per step, oracle restatement of arma::interp2, OpenMP over queries"},
            "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def time_steps(torch, fn, steps, warmup, dist=None):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, CUDA events on
    the current stream; returns total ms (max over ranks)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        dist.barrier()
    return ms


def wall_steps(torch, fn, steps, warmup, dist=None):
    """Host-visible timing for calls that synchronise internally (host-buffer C-ABI entry points)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0)
    if dist:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        dist.barrier()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--config5-full", action="store_true", help="(default now) profile-map stability at R = 1000 (1e6 neurons per column)")
    ap.add_argument("--no-config5-full", action="store_true", help="skip the R = 1000 profile-map stability")
    ap.add_argument("--only-config5", action="store_true", help="of the secondary workloads run only the profile-map stability")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write a seeded sample of the last step's outputs (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)      # both arms: at least 3 warm-up steps
    if args.impl == "reference":
        return run_reference(args)

    # stdout carries exactly ONE line, the JSON; whatever libraries print there on the way (NCCL's version banner
    # of the in-process communicators, for one) goes to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import armadillocudalinearinterpolation_b200 as B
    from armadillocudalinearinterpolation_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    B.set_device(local)
    dist = None
    cpu_group = None
    if world > 1:
        # keep stdout to the one JSON line (NCCL prints its version banner there otherwise)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        import torch.distributed as dist_
        dist_.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_
        cpu_group = dist.new_group(backend="gloo")     # host-side waits (no GPU kernel spinning on an idle rank's device)
    n_gpus = world

    # ---------------- headline: interp2 scattered, 1e8 queries / GPU ----------------
    grid = make_grid()
    plan = B.Interp2Plan(*grid)
    g = torch.Generator(device="cuda").manual_seed(2235 + rank)
    xq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
    yq = torch.rand(NQ, generator=g, device="cuda", dtype=torch.float64)
    zq = torch.empty_like(xq)
    step = lambda: plan.scattered(xq, yq, out=zq)
    sampler = ClockSampler(local)
    from armadillocudalinearinterpolation_b200 import _lib as L_
    L_.lib().b200_launch_count.restype = C.c_ulonglong
    time_steps(torch, step, 1, args.warmup, dist)       # warm-up outside the sampled window
    sampler.start()
    launches0 = L_.lib().b200_launch_count()
    ms = time_steps(torch, step, args.steps, 0, dist)
    gpu_launches = int(L_.lib().b200_launch_count() - launches0)   # counted by the library at every launch site
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, zq)      # now: the secondary workloads below reuse zq
    ms_per_step = ms / args.steps
    value = n_gpus * NQ / (ms_per_step * 1e-3)
    peak, peak_src = measured_peak()
    alg_bytes = ALG_BYTES_PER_QUERY * NQ + ALG_BYTES_GRID
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
    # dram__bytes of the same kernel from the committed ncu capture (tools/make_profiles.py); the capture
    # carries a hash of the kernel sources it was taken for, so a stale figure is flagged, not silently reused
    traffic, traffic_note = None, "no ncu capture committed"
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            rec = json.load(open(tpath)).get("interp2_scattered_f64", {})
            traffic = rec.get("dram_bytes_per_launch")
            stamp = rec.get("source_sha1")
            now = source_stamp(INTERP2_SOURCES)
            traffic_note = (f"ncu --set full capture {rec.get('capture', '?')}, kernel sources unchanged since (sha1 {now})"
                            if stamp == now else
                            f"STALE: captured for kernel sources {stamp}, this build is {now}")
        except Exception:
            traffic = None

    # ---------------- e2e: host buffers through the C-ABI ----------------
    hx = torch.empty(NQ, dtype=torch.float64).pin_memory()
    hy = torch.empty(NQ, dtype=torch.float64).pin_memory()
    hz = torch.empty(NQ, dtype=torch.float64).pin_memory()
    hx.copy_(xq); hy.copy_(yq)
    torch.cuda.synchronize()
    hxn, hyn, hzn = hx.numpy(), hy.numpy(), hz.numpy()
    e2e_steps = max(3, min(args.steps, 10))
    e2e_ms = wall_steps(torch, lambda: plan.scattered(hxn, hyn, out=hzn), e2e_steps, 1, dist) / e2e_steps
    e2e_val = n_gpus * NQ / (e2e_ms * 1e-3)
    zq_host = zq.cpu().numpy()
    check_all_bits = bool(np.array_equal(hzn.view(np.int64), zq_host.view(np.int64)))   # all 1e8 outputs, bit for bit
    check = float(np.nanmax(np.abs(hzn - zq_host)))
    # the same call with PAGEABLE buffers (what a plain arma::vec is): staged through the library's pinned ring
    pxn, pyn, pzn = np.array(hxn), np.array(hyn), np.empty_like(hzn)
    pg_steps = 3
    pg_ms = wall_steps(torch, lambda: plan.scattered(pxn, pyn, out=pzn), pg_steps, 1, dist) / pg_steps
    pageable_bits = bool(np.array_equal(pzn.view(np.int64), zq_host.view(np.int64)))
    del hx, hy, hz, pxn, pyn, pzn, zq_host

    # machine ceiling for this access pattern, measured live: independent 32-byte gathers from a
    # 512 MiB table (every L2 miss fills a 128-byte line on B200, so uniformly random queries are
    # bounded by this, not by the streaming copy rate)
    g_ms, g_rate = L_.bench_random_gather(512 << 20, NQ)
    tile_bytes = (((NX - 1) // 3 + 1) * ((NY - 1) // 3 + 1)) * 128      # the table the kernel actually gathers from
    g2_ms, g2_rate = L_.bench_random_gather(tile_bytes, NQ)
    fp64_peak = L_.bench_fp64_fma()

    line = {"metric": METRIC,
            "value": value, "unit": "points/s", "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": headline_config(n_gpus),
            "layout": "linspace axes recognised as affine at plan time (knots recomputed in registers; other axes are staged in shared memory by TMA bulk copy); Z as overlapping 4x4 tiles, one 128-byte line per cell (228 MiB)",
            "gpu_launches": gpu_launches,
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "points/s", "h2d_bytes_per_step": 16 * NQ, "d2h_bytes_per_step": 8 * NQ,
                    "ms_per_step": e2e_ms, "api": "b200_interp2_scattered (pinned host buffers, 2-slot chunked pipeline)",
                    "all_1e8_outputs_bitwise_equal_to_device_path": check_all_bits,
                    "max_abs_diff_vs_device_path": check,
                    "pageable_host_buffers": {"value": n_gpus * NQ / (pg_ms * 1e-3), "ms_per_step": pg_ms,
                                              "bitwise_equal": pageable_bits,
                                              "note": "same call with ordinary (pageable) numpy / arma::vec buffers"}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_note,
                         # what the DRAM interface actually moved: every L2 miss of a random query fills a whole
                         # 128-byte line although 32 bytes of it are used, so the kernel saturates HBM in real bytes
                         # (this line) while its algorithmic bytes are a quarter of that (`frac`)
                         "dram_GBps_actual": (traffic / (ms_per_step * 1e6)) if traffic else None,
                         "dram_frac_of_peak_actual": (traffic / (ms_per_step * 1e6) / peak) if traffic else None,
                         "peak_source": peak_src, "kernel": "interp2_scattered_smem_kernel<double, tiles>",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         # what bounds uniformly random queries on a 128 MiB grid, as numbers: one table line per
                         # query is the minimum (four corners in one 128-byte line), and this GPU delivers random
                         # lines from a table of this size at the rate measured live below — the floor is the
                         # slower of that and the HBM streaming time of the algorithmic bytes
                         "floor": {"ms": max(1e3 * alg_bytes / (peak * 1e9), g2_ms),
                                   "hbm_stream_ms": 1e3 * alg_bytes / (peak * 1e9),
                                   "random_line_gather_ms": g2_ms,
                                   "derivation": "max(algorithmic bytes / measured HBM copy peak, 1e8 / measured random 32-byte gather rate from a table of the tile table's size [b200_bench_random_gather, same run])"},
                         "frac_of_floor": max(1e3 * alg_bytes / (peak * 1e9), g2_ms) / ms_per_step,
                         "random_gather_ceiling": {"gathers_per_s": g_rate, "ms_for_1e8": g_ms,
                                                   "frac_of_ceiling": (NQ / (ms_per_step * 1e-3)) / g_rate,
                                                   "note": "1e8 independent 32-byte gathers from a 512 MiB table (the size of the 2x2 corner records), same GPU, same run"},
                         "random_gather_ceiling_tile_table": {"gathers_per_s": g2_rate, "ms_for_1e8": g2_ms, "table_bytes": tile_bytes,
                                                              "frac_of_ceiling": (NQ / (ms_per_step * 1e-3)) / g2_rate,
                                                              "note": "same micro-benchmark on a table of the size of the 4x4 tiles: one 32-byte gather and nothing else per query"}}}

    # ---------------- secondary workloads ----------------
    if not args.no_extra:
        extra = {}
        try:
            if not args.only_config5:
                # configs[0]: 1-D, 1e6 knots, 1e7 queries; 8 rotating query/output buffer pairs (1.28 GB)
                # so that consecutive launches never find their streams in L2
                rng = np.random.default_rng(1234)
                ng, ni, nbuf = 1_000_000, 10_000_000, 8
                for kind in ("uniform", "nonuniform"):
                    xg = np.linspace(0.0, 1.0, ng) if kind == "uniform" else np.cumsum(0.5 + rng.random(ng))
                    xg = (xg - xg[0]) / (xg[-1] - xg[0])
                    yg = np.sin(2 * np.pi * xg) + 0.1 * np.random.default_rng(1235).standard_normal(ng)
                    p1 = B.Interp1Plan(xg, yg)
                    for order in ("unsorted", "sorted"):
                        g1 = torch.Generator(device="cuda").manual_seed(1236)
                        qs = [torch.rand(ni, generator=g1, device="cuda", dtype=torch.float64) for _ in range(nbuf)]
                        if order == "sorted":
                            qs = [q.sort().values for q in qs]
                        outs = [torch.empty_like(q) for q in qs]
                        state = {"i": 0}

                        def step1():
                            i = state["i"] % nbuf
                            state["i"] += 1
                            p1(qs[i], out=outs[i])
                        k1 = max(args.steps, 200)      # >= 100 back-to-back launches: one launch is launch-overhead-sized (SURVEY 8d)
                        ms1 = time_steps(torch, step1, k1, 3, dist) / k1
                        gbs = (16 * ni + 16 * ng) / (ms1 * 1e-3) / 1e9
                        extra[f"interp1_f64_1e6knots_1e7queries_{kind}_{order}"] = {
                            "points_per_s": n_gpus * ni / (ms1 * 1e-3), "ms_per_launch": ms1, "lookup_mode": p1.lookup_mode,
                            "algorithmic_GBps": gbs, "roofline_frac": gbs / peak}
                        del qs, outs
                    p1.close()
                # what bounds UNSORTED queries on a 1e6-knot grid: one L2 gather per query (the 32 MB of segment records are
                # L2-resident); the machine's rate for that, measured live: independent 32-byte gathers from a 32 MiB table
                g1_ms, g1_rate = L_.bench_random_gather(32 << 20, 10_000_000)
                for kind in ("uniform", "nonuniform"):
                    rec = extra[f"interp1_f64_1e6knots_1e7queries_{kind}_unsorted"]
                    rec["l2_gather_floor"] = {"gathers_per_s": g1_rate, "us_for_1e7": g1_ms * 1e3,
                                              "frac_of_floor": g1_ms / rec["ms_per_launch"],
                                              "note": "1e7 independent 32-byte gathers from a 32 MiB (L2-resident) table, nothing else in the kernel"}
                # FP32 variants of configs[0] (SURVEY 8d: 88 MB of algorithmic bytes)
                xg32 = np.linspace(0.0, 1.0, ng).astype(np.float32); yg32 = np.sin(2 * np.pi * xg32).astype(np.float32)
                xg32 = np.unique(xg32)
                p32 = B.Interp1Plan(xg32, yg32[:xg32.size])
                for order in ("unsorted", "sorted"):
                    g1 = torch.Generator(device="cuda").manual_seed(1236)
                    qs = [torch.rand(ni, generator=g1, device="cuda", dtype=torch.float32) for _ in range(nbuf)]
                    if order == "sorted":
                        qs = [q.sort().values for q in qs]
                    outs = [torch.empty_like(q) for q in qs]
                    state = {"i": 0}

                    def step32():
                        i = state["i"] % nbuf
                        state["i"] += 1
                        p32(qs[i], out=outs[i])
                    k1 = max(args.steps, 200)      # >= 100 back-to-back launches: one launch is launch-overhead-sized (SURVEY 8d)
                    ms1 = time_steps(torch, step32, k1, 3, dist) / k1
                    gbs = (8 * ni + 8 * xg32.size) / (ms1 * 1e-3) / 1e9
                    extra[f"interp1_f32_1e6knots_1e7queries_uniform_{order}"] = {
                        "points_per_s": n_gpus * ni / (ms1 * 1e-3), "ms_per_launch": ms1, "lookup_mode": p32.lookup_mode,
                        "algorithmic_GBps": gbs, "roofline_frac": gbs / peak}
                    del qs, outs
                p32.close()
                # steady state of the large-grid path: same 1e6 uniform knots, 1e8 sorted / unsorted queries in one launch
                xg = np.linspace(0.0, 1.0, ng); yg = np.sin(2 * np.pi * xg)
                p1 = B.Interp1Plan(xg, yg)
                gl = torch.Generator(device="cuda").manual_seed(1237)
                ql = torch.rand(NQ, generator=gl, device="cuda", dtype=torch.float64)
                ol = torch.empty_like(ql)
                for order in ("unsorted", "sorted"):
                    if order == "sorted":
                        ql = ql.sort().values
                    nl = max(5, args.steps // 2)
                    msl = time_steps(torch, lambda: p1(ql, out=ol), nl, 3, dist) / nl
                    gbs = (16 * NQ + 16 * ng) / (msl * 1e-3) / 1e9
                    extra[f"interp1_f64_1e6knots_1e8queries_uniform_{order}"] = {
                        "points_per_s": n_gpus * NQ / (msl * 1e-3), "ms_per_launch": msl, "lookup_mode": p1.lookup_mode,
                        "algorithmic_GBps": gbs, "roofline_frac": gbs / peak}
                p1.close(); del ql, ol
                # coarse profile -> fine ensemble: 1e3 knots staged in shared memory, 1e8 queries (1.6 GB of streams)
                xg = np.linspace(-3.0, 3.0, 1000); yg = np.sin(xg)
                p1 = B.Interp1Plan(xg, yg)
                gs = torch.Generator(device="cuda").manual_seed(77)
                qsm = torch.rand(NQ, generator=gs, device="cuda", dtype=torch.float64) * 6.0 - 3.0
                osm = torch.empty_like(qsm)
                nsm = max(5, args.steps // 2)
                mssm = time_steps(torch, lambda: p1(qsm, out=osm), nsm, 3, dist) / nsm
                gbs = (16 * NQ + 16 * 1000) / (mssm * 1e-3) / 1e9
                extra["interp1_f64_1e3knots_1e8queries_smem"] = {"points_per_s": n_gpus * NQ / (mssm * 1e-3), "ms_per_launch": mssm,
                                                                 "lookup_mode": p1.lookup_mode, "algorithmic_GBps": gbs, "roofline_frac": gbs / peak}
                p1.close(); del qsm, osm
                # configs[1] grid shape (Armadillo's own interp2 API): 1e4 x 1e4 sorted points
                g2 = torch.Generator(device="cuda").manual_seed(2236)
                xi = torch.rand(10_000, generator=g2, device="cuda", dtype=torch.float64).sort().values
                yi = torch.rand(10_000, generator=g2, device="cuda", dtype=torch.float64).sort().values
                msg = time_steps(torch, lambda: plan.grid(xi, yi), max(5, args.steps // 2), 3, dist) / max(5, args.steps // 2)
                gb = (8 * 1e8 + ALG_BYTES_GRID + 16 * 1e4) / (msg * 1e-3) / 1e9
                extra["interp2_grid_f64_1e4x1e4"] = {"points_per_s": n_gpus * 1e8 / (msg * 1e-3), "ms_per_launch": msg,
                                                     "algorithmic_GBps": gb, "roofline_frac": gb / peak}
                # configs[1] through the opt-in L2-banded pipeline (partition by record band -> band-major
                # interpolation -> un-permute; profiles/interp2_banded_r1.md): same queries, same bits
                pb = B.Interp2Plan(*grid, flags=B.Interp2Plan.FORCE_BANDS)
                zb = torch.empty_like(zq)
                nbd = max(5, args.steps // 2)
                msb = time_steps(torch, lambda: pb.scattered(xq, yq, out=zb), nbd, 3, dist) / nbd
                plan.scattered(xq, yq, out=zq)
                same = bool(torch.equal(zb.view(torch.int64), zq.view(torch.int64)))
                extra["interp2_scattered_f64_banded_pipeline_opt_in"] = {
                    "points_per_s": n_gpus * NQ / (msb * 1e-3), "ms_per_call": msb, "kernels_per_call": 3,
                    "algorithmic_GBps": alg_bytes / (msb * 1e-3) / 1e9, "roofline_frac": alg_bytes / (msb * 1e-3) / 1e9 / peak,
                    "bitwise_equal_to_direct_kernel": same}
                pb.close(); del zb
                # FP32 variants of configs[1] (64 MiB grid: column-major Z is the layout the plan picks)
                x32, y32, z32 = grid[0].astype(np.float32), grid[1].astype(np.float32), grid[2].astype(np.float32)
                pf = B.Interp2Plan(x32, y32, z32)
                xq32, yq32 = xq.to(torch.float32), yq.to(torch.float32)
                zq32 = torch.empty_like(xq32)
                nf = max(5, args.steps // 2)
                msf = time_steps(torch, lambda: pf.scattered(xq32, yq32, out=zq32), nf, 3, dist) / nf
                gbf = (12 * NQ + 4 * NX * NY) / (msf * 1e-3) / 1e9
                extra["interp2_scattered_f32_4096x4096_1e8"] = {"points_per_s": n_gpus * NQ / (msf * 1e-3), "ms_per_launch": msf,
                                                                "algorithmic_GBps": gbf, "roofline_frac": gbf / peak}
                xi32, yi32 = xi.to(torch.float32), yi.to(torch.float32)
                msgf = time_steps(torch, lambda: pf.grid(xi32, yi32), nf, 3, dist) / nf
                gbgf = (4 * 1e8 + 4 * NX * NY + 8 * 1e4) / (msgf * 1e-3) / 1e9
                extra["interp2_grid_f32_1e4x1e4"] = {"points_per_s": n_gpus * 1e8 / (msgf * 1e-3), "ms_per_launch": msgf,
                                                     "algorithmic_GBps": gbgf, "roofline_frac": gbgf / peak}
                pf.close(); del xq32, yq32, zq32
                # write-only ceiling of this GPU (a kernel that only stores): what the grid kernel is up against
                wbuf = torch.empty(NQ, dtype=torch.float64, device="cuda")
                msw = time_steps(torch, lambda: wbuf.fill_(1.5), 10, 3, dist) / 10
                extra["write_only_ceiling_GBps"] = 8 * NQ / (msw * 1e-3) / 1e9
                del wbuf
                # configs[1] with tile-sorted queries (SURVEY 8d variant iii): same points, ordered by grid cell
                cell = (xq * (NX - 1)).floor().to(torch.int64) * NY + (yq * (NY - 1)).floor().to(torch.int64)
                order = cell.argsort()
                del cell
                xs, ys = xq[order], yq[order]
                del order
                nst = max(5, args.steps // 2)
                mss = time_steps(torch, lambda: plan.scattered(xs, ys, out=zq), nst, 3, dist) / nst
                gbs = alg_bytes / (mss * 1e-3) / 1e9
                extra["interp2_scattered_f64_cell_sorted_queries"] = {"points_per_s": n_gpus * NQ / (mss * 1e-3), "ms_per_launch": mss,
                                                                      "algorithmic_GBps": gbs, "roofline_frac": gbs / peak}
                del xs, ys
                # configs[2]: one map evaluation, parameters.hpp default ensemble (R=1000, N=1024, M=3, T=5).
                # Roofline convention frozen in BASELINE.md §3: unit of work = neuron-event update, F_alg = 10 FP64
                # flops per update (calibrated once against ncu SASS op counts: (2 dfma + dadd + dmul) / updates = 9.8),
                # peak = the FP64 FMA issue ceiling measured live by b200_bench_fp64_fma.  The event loop is a serial
                # dependency chain, so the fraction is low by construction; chain_cycles_per_event says how long one
                # event of one ring takes end to end.
                F_ALG = 10.0
                for sigma in (0.0, 0.5):
                    m = B.EventDrivenMap([BETA], 1000, noNeurons=1024)
                    m.SetParameterStdDev(sigma); m.SetSeed(42); m.EnableTiming(True)
                    for _ in range(3):
                        m.ComputeF(Z_DRIVER)
                    reps = 10
                    t0 = time.perf_counter()
                    evolve_ms = []
                    for _ in range(reps):
                        m.ComputeF(Z_DRIVER)
                        evolve_ms.append(m.LastEvolveMs())
                    call_ms = 1e3 * (time.perf_counter() - t0) / reps
                    cnt = m.LastCounters()
                    ev_ms = float(np.mean(evolve_ms))
                    updates = cnt["events"] * 1024
                    tflops = updates * F_ALG / (ev_ms * 1e-3) / 1e12
                    rec = {
                        "evals_per_s_per_gpu": 1e3 / call_ms, "ms_per_compute_f": call_ms, "evolve_kernel_ms": ev_ms,
                        "events": cnt["events"], "neuron_event_updates_per_s": updates / (ev_ms * 1e-3),
                        "candidates": cnt["candidates"], "newton_its": cnt["newton_its"],
                        "roofline": {"bound": "fp64 pipe (latency-bound in practice)", "achieved": tflops, "peak": fp64_peak,
                                     "unit": "TFLOP/s", "frac": tflops / fp64_peak,
                                     "convention": "10 FP64 flops per neuron-event update (BASELINE.md §3), peak = live DFMA issue ceiling",
                                     "chain_cycles_per_event": ev_ms * 1e-3 * (clocks.get("sm_mhz") or 1965.0) * 1e6 / (cnt["events"] / 1000.0)}}
                    m.close()
                    if rank == 0 and n_gpus == 1 and not args.no_cpu:
                        # CPU baseline of the same evaluation: the oracle's restatement of lift -> evolve -> restrict,
                        # OpenMP over realisations, on a bounded sample of the 1000 realisations
                        from oracle import oracle_py as O
                        th = cpu_threads()
                        rs = 2 * th
                        cfg = O.edm_cfg(R=1000, N=1024, sigma=sigma, seed=42)
                        O.edm_compute_f(cfg, Z_DRIVER, r_begin=0, r_end=th, nthreads=th, aux=False)
                        tc = time.perf_counter()
                        O.edm_compute_f(cfg, Z_DRIVER, r_begin=0, r_end=rs, nthreads=th, aux=False)
                        sec = (time.perf_counter() - tc) * 1000.0 / rs          # seconds per full 1000-realisation evaluation
                        rec["cpu_baseline"] = {"value": 1.0 / sec, "unit": "map evals/s", "cores": th, "kind": "port",
                                               "sample": f"{rs} of the 1000 realisations, scaled; oracle restatement of EventDrivenMap::ComputeF"}
                    extra[f"map_eval_R1000_N1024_sigma{sigma}"] = rec
                # the state the reference driver ends in (Driver.cu:68-71: N = 512) and the reference's own device
                # arithmetic (FP32): its unmodified kernels take 14.0 ms (N = 1024) / 3.2 ms (N = 512) per ComputeF on
                # the same GPU (BASELINE.md 5b, tools/ref_time.py, profiles/r2_reference_time.txt)
                for prec, nn in (("f64", 512), ("f32", 512), ("f32", 1024)):
                    m = B.EventDrivenMap([BETA], 1000, noNeurons=nn, precision=prec)
                    m.EnableTiming(True)
                    for _ in range(3):
                        m.ComputeF(Z_DRIVER)
                    evs = []
                    for _ in range(5):
                        m.ComputeF(Z_DRIVER); evs.append(m.LastEvolveMs())
                    extra[f"map_eval_R1000_N{nn}_{prec}"] = {"evolve_kernel_ms": float(np.mean(evs)), "events": m.LastCounters()["events"],
                                                            "arithmetic": "FP32 (the reference's device precision)" if prec == "f32" else "FP64"}
                    m.close()
                if rank == 0 and n_gpus == 1 and not args.no_cpu:
                    # the baseline beside it: the UNMODIFIED reference (oracle/_ref: its own FP32 kernels, compiled for
                    # sm_100a where B200_REFERENCE_DIR names it at build time) timed on this GPU — a baseline leg, never the thing shipped
                    # (in a child process: the reference's error convention is exit(-1), EventDrivenMap.cu:18-54)
                    try:
                        import re, subprocess
                        if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libedm_ref.so")):
                            out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_time.py")], capture_output=True,
                                                 text=True, timeout=120)
                            got = {f"R1000_N{m_.group(1)}": float(m_.group(2))
                                   for m_ in re.finditer(r"R=1000 N=(\d+): ([0-9.]+) ms per ComputeF", out.stdout)}
                            extra["reference_own_kernels_on_this_gpu"] = (
                                {"ms_per_compute_f": got,
                                 "what": "EventDrivenMap::ComputeF of the unmodified reference (EventDrivenMap.cu, FP32 device arithmetic), host clock around its blocking calls"}
                                if got else {"unavailable": (out.stderr or out.stdout)[-200:]})
                    except Exception as e:
                        extra["reference_own_kernels_on_this_gpu"] = {"unavailable": repr(e)[:200]}
                # configs[3]: finite-difference Jacobian (n+1 = 4 evaluations x 1000 realisations), work
                # items sharded over the ranks, positions gathered with one NCCL all-gather
                jm = parallel.ShardedJacobian([BETA], 1000, noNeurons=1024, group=dist)
                for _ in range(3):
                    jm.ComputeDFDU(Z_DRIVER, 1e-2)
                reps = 10
                msj = wall_steps(torch, lambda: jm.ComputeDFDU(Z_DRIVER, 1e-2), reps, 0, dist) / reps
                extra["fd_jacobian_n3_R1000_N1024"] = {"jacobians_per_s": 1e3 / msj, "map_evals_per_s": 4e3 / msj,
                                                       "ms_per_jacobian": msj, "ranks": n_gpus, "scaling": "strong",
                                                       "collective": "all_gather of (items x 3) positions" if world > 1 else "none"}
            # configs[4]: stability analysis on a 1e3-dim coarse PROFILE (profile map: n = 2 x 500 knots),
            # 1001 evaluations per Jacobian; columns sharded over the ranks, residual columns all-gathered.
            # R = 64 realisations per column by default (--config5-full: R = 1000, i.e. 1e6 neurons per column)
            fm = B.EventDrivenMap([BETA], 1, noNeurons=1024)
            fm.SetDebugFlag(True); fm.ComputeF(Z_DRIVER)
            lv, ls = fm.DebugFetch("lift_v")[0], fm.DebugFetch("lift_s")[0]
            fm.close()
            nc = 500
            xf = -3.0 + 6.0 / 1024 * np.arange(1024); xc = -3.0 + 6.0 / nc * np.arange(nc)
            u0 = np.concatenate([np.interp(xc, xf, lv), np.interp(xc, xf, ls)])
            for R5 in ([64] if args.no_config5_full else [64, 1000]):   # R = 1000: 1e6 neurons per column (BASELINE config 5)
                pj = parallel.ShardedJacobian([BETA], R5, noNeurons=1024, group=dist, shard="columns")
                pj.engine.map.SetTimeHorizon(1.0)
                pj.SetProfileMode(nc)
                J5 = pj.ComputeDFDU(u0, 1e-3)
                reps5 = 1 if R5 >= 1000 else 3
                ms5 = wall_steps(torch, lambda: pj.ComputeDFDU(u0, 1e-3), reps5, 0, dist) / reps5
                t0 = time.perf_counter()
                lam = np.linalg.eigvals(J5 + np.eye(2 * nc)) if rank == 0 else None
                eig_ms = 1e3 * (time.perf_counter() - t0)
                extra[f"profile_stability_n1000_N1024_R{R5}"] = {
                    "ms_per_jacobian": ms5, "map_evals_per_s": 1001e3 / ms5, "columns": 1001, "rings": 1001 * R5,
                    "neurons_per_column": 1024 * R5, "time_horizon": 1.0, "ranks": n_gpus, "scaling": "strong",
                    "unstable_eigenvalues": int(np.sum(np.abs(lam) > 1.0)) if rank == 0 else None,
                    "host_eig_ms_numpy": eig_ms, "collective": "all_gather of 1001 residual columns (8 MB)" if world > 1 else "none",
                    "launcher": "one process per GPU (torchrun), torch.distributed NCCL all_gather_into_tensor"}
                pj.engine.map.close()
                del pj
            # ---- configs[3] and [4] through the product's own C++ classes (host layer over the C-ABI) ----
            # Rank 0 drives 1 and then all n_gpus devices IN ONE PROCESS (EventDrivenMapB200::SetDevices: column / item
            # shards, one ncclAllGather inside libb200edm.so); the other ranks wait on the host (gloo), their GPUs idle.
            cpp = {}
            try:
              if rank == 0:
                host = C.CDLL(os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "lib", "libb200host.so"))
                host.b200_host_last_error.restype = C.c_char_p
                dp = lambda a: a.ctypes.data_as(C.c_void_p)
                dev_sets = [1] + ([n_gpus] if n_gpus > 1 else [])

                def newton(ndev, mode=1):
                    sol = np.zeros(3); hist = np.full(11, np.nan); nh = C.c_int(); J = np.zeros((3, 3), order="F"); msv = np.zeros(2)
                    devs = (C.c_int * ndev)(*range(ndev))
                    rc = host.b200_host_edm_newton_multi(C.c_double(BETA), 1000, 1024, dp(Z_DRIVER), 3, C.c_double(1e-4), 10,
                                                         C.c_double(1e-2), mode, C.c_double(0.0), ndev, devs, dp(sol), dp(hist),
                                                         C.byref(nh), dp(J), dp(msv))
                    if rc < 0:
                        raise RuntimeError(host.b200_host_last_error().decode())
                    return rc, sol, hist[:nh.value], J, msv

                res = {nd: newton(nd) for nd in dev_sets}
                # mode 3: the reference's call sequence (ComputeF after the update, ComputeDFDU — which repeats F — on the
                # next turn) instead of one batched F + dF/dU per iterate; same iterates
                res_seq = {nd: newton(nd, 3) for nd in dev_sets}
                r1 = res[1]
                cpp["newton_config4_R1000_N1024"] = {
                    "driver_settings": "Driver.cu:28-37 (tol 1e-4, <= 10 iterations, FD eps 1e-2), Jacobian through ComputeDFDU",
                    "converged": bool(r1[0] == 1), "iterations": int(len(r1[2]) - 1), "solution": r1[1].tolist(),
                    "final_residual": float(r1[2][-1]),
                    "solve_ms": {str(nd): float(res[nd][4][0]) for nd in dev_sets},
                    "solve_ms_reference_call_sequence": {str(nd): float(res_seq[nd][4][0]) for nd in dev_sets},
                    "evaluation": "F(u) never evaluated twice per iteration (AbstractNonlinearProblemFused): one GPU — Jacobian from the residual in hand (n evaluations); several GPUs — F and dF/dU of every iterate in one batch",
                    "jacobian_ms": {str(nd): float(res[nd][4][1]) for nd in dev_sets},
                    "bitwise_equal_across_device_counts": all(
                        np.array_equal(res[nd][1], r1[1]) and np.array_equal(res[nd][2], r1[2]) and np.array_equal(res[nd][3], r1[3])
                        for nd in dev_sets),
                    "bitwise_equal_to_reference_call_sequence": all(
                        np.array_equal(res_seq[nd][1], r1[1]) and np.array_equal(res_seq[nd][2], r1[2]) and np.array_equal(res_seq[nd][3], r1[3])
                        for nd in dev_sets)}

                def stability(R, ndev):
                    n = 2 * nc
                    msv = np.zeros(3); J = np.zeros((n, n), order="F"); re = np.zeros(n); im = np.zeros(n)
                    devs = (C.c_int * ndev)(*range(ndev))
                    cnt = host.b200_host_profile_stability(C.c_double(BETA), R, 1024, nc, C.c_double(1.0), dp(u0), C.c_double(1e-3),
                                                           ndev, devs, dp(msv), dp(J), dp(re), dp(im))
                    if cnt <= -1000:
                        raise RuntimeError(host.b200_host_last_error().decode())
                    return cnt, J, msv

                for R in ([64] if args.no_config5_full else [64, 1000]):
                    sres = {nd: stability(R, nd) for nd in dev_sets}
                    s1 = sres[1]
                    lam_np = np.linalg.eigvals(s1[1] + np.eye(2 * nc))
                    cpp[f"stability_config5_n1000_N1024_R{R}"] = {
                        "call": "Stability::ComputeNumUnstableEigenvalues(u) = FD Jacobian (1001 evaluations) + arma::eig_gen (cuSOLVER GEEV behind the shim)",
                        "neurons_per_column": 1024 * R, "unstable_eigenvalues": int(s1[0]),
                        "numpy_count_on_same_jacobian": int(np.sum(np.abs(lam_np) > 1.0)),
                        "whole_call_ms": {str(nd): float(sres[nd][2][0]) for nd in dev_sets},
                        "jacobian_ms": {str(nd): float(sres[nd][2][1]) for nd in dev_sets},
                        "eig_gen_ms": {str(nd): float(sres[nd][2][2]) for nd in dev_sets},
                        "bitwise_equal_across_device_counts": all(np.array_equal(sres[nd][1], s1[1]) and sres[nd][0] == s1[0] for nd in dev_sets)}
            except Exception as e:      # the headline line must still be printed
                cpp["error"] = f"{type(e).__name__}: {e}"
            if cpu_group is not None:
                dist.barrier(group=cpu_group)
            extra["cpp_host_layer"] = cpp
        except Exception as e:
            if world > 1:       # several ranks: a one-sided failure would leave the others in a collective
                raise
            import traceback
            extra["error"] = f"{type(e).__name__}: {e}"
            print(traceback.format_exc(), file=sys.stderr)
        line["extra"] = extra

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    if rank == 0 and n_gpus == 1 and not args.no_cpu:
        th = cpu_threads()
        sample = 20_000_000
        v = cpu_interp2(sample, th, grid)
        line["cpu_baseline"] = {"value": v, "unit": "points/s", "cores": th, "kind": "port",
                                "sample": f"{sample} of 1e8 scattered queries, oracle restatement of arma::interp2, OpenMP over queries"}
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist:
        os.dup2(2, 1)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
