"""Tensor-grid interp2 (b200_interp2_grid, b200_interp2_grid_dev, b200_interp2_f64 / _f32, Interp2Plan.grid) against
the CPU oracle: every output of the benchmark's 1e4 x 1e4 grid, every build of the grid kernel (element type x rows
per thread x pass order) at every output alignment, the device call's launch boundary, the host call's column
blocks, query orders that walk the kernel's column cache through each of its cases, and special values.  Also the
operand checks of the Python value calls on CUDA tensors.

Bits are compared on integer views, so -0.0 counts; NaN is compared by position only (payloads may differ between the
host and the device).  Device outputs are written into a buffer filled with a sentinel, which must survive outside
the nxi * nyi outputs."""
import ctypes as C
import os

import numpy as np
import pytest

from armadillocudalinearinterpolation_b200 import _lib

pytestmark = pytest.mark.gpu

# plan2_grid_main / plan2_grid_host (interp2.cu)
GRID_COLS = 32                          # kGridCols: output columns per block
COLS_PER_LAUNCH = 65535 * GRID_COLS     # gridDim.y limit: past this many columns the device call launches again
HOST_BLOCK_BYTES = 32 << 20             # the host call produces ZI in column blocks of at most this size
SENTINEL = -1234.5678
NT = os.cpu_count() or 8


def ints(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def same_ints(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(ints(np.ravel(a, "F")), ints(np.ravel(b, "F")))


def same_as_oracle(a, ref, chunk=1 << 24):
    """Equal bits wherever the oracle is not NaN, NaN at the same places.  Column-major ZI is compared in memory order
    and in chunks, without a copy of a 1e8-output grid."""
    a, ref = np.asarray(a), np.asarray(ref)
    if a.shape != ref.shape or a.dtype != ref.dtype:
        return False
    fa, fr = np.ravel(a, "F"), np.ravel(ref, "F")
    for s in range(0, fa.size, chunk):
        x, r = fa[s:s + chunk], fr[s:s + chunk]
        nx, nr = np.isnan(x), np.isnan(r)
        if not (np.array_equal(nx, nr) and np.array_equal(ints(x)[~nx], ints(r)[~nr])):
            return False
    return True


def kernel_rows(nyi, addr, esz):
    """Output rows per thread (V) that plan2_grid_main picks: 4 or 2 when nyi is a multiple of it and every column
    of ZI starts aligned to V elements, else 1."""
    if nyi % 4 == 0 and addr % (4 * esz) == 0:
        return 4
    if nyi % 2 == 0 and addr % (2 * esz) == 0:
        return 2
    return 1


def grid_dev(plan, xi, yi, extrap, offset=0, tail=67):
    """b200_interp2_grid_dev with ZI at `offset` elements into a buffer filled with SENTINEL.  Asserts that every
    element outside ZI still holds it.  Returns (status, ZI as an (nyi, nxi) array, ZI's device address)."""
    import torch
    nxi, nyi = xi.numel(), yi.numel()
    n = nxi * nyi
    buf = torch.full((offset + n + tail,), SENTINEL, dtype=xi.dtype, device=xi.device)
    zi = buf[offset:offset + n]
    rc = _lib.lib().b200_interp2_grid_dev(plan._h, C.c_void_p(xi.data_ptr()), C.c_size_t(nxi),
                                          C.c_void_p(yi.data_ptr()), C.c_size_t(nyi), C.c_void_p(zi.data_ptr()),
                                          C.c_double(extrap), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    s = ints(np.array([SENTINEL], h.dtype))[0]
    assert np.all(ints(h[:offset]) == s) and np.all(ints(h[offset + n:]) == s), "grid_dev wrote outside ZI"
    return rc, h[offset:offset + n].reshape(nxi, nyi).T, zi.data_ptr()


def grid_host(plan, xi, yi, extrap, tail=67):
    """b200_interp2_grid into a host buffer filled with SENTINEL; the same check and returns as grid_dev."""
    nxi, nyi = xi.size, yi.size
    n = nxi * nyi
    buf = np.full(n + tail, SENTINEL, plan.dtype)
    rc = _lib.lib().b200_interp2_grid(plan._h, C.c_void_p(xi.ctypes.data), C.c_size_t(nxi), C.c_void_p(yi.ctypes.data),
                                      C.c_size_t(nyi), C.c_void_p(buf.ctypes.data), C.c_double(extrap))
    assert np.all(ints(buf[n:]) == ints(np.array([SENTINEL], plan.dtype))[0]), "grid wrote outside ZI"
    return rc, buf[:n].reshape(nxi, nyi).T


def ragged(rng, n, dt):
    """strictly ascending, unevenly spaced knots (no affine axis)"""
    x = np.unique(np.cumsum(0.25 + rng.random(n)).astype(dt))
    assert x.size == n
    return x


def special_z(rng, ny, nx, dt):
    """Z with NaN, +-inf, -0.0 and subnormals, some of them on the last row and the last column"""
    z = rng.standard_normal((ny, nx)).astype(dt)
    tiny = np.finfo(dt).smallest_subnormal
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, tiny, -3 * tiny, 7 * tiny], dt)
    k = min(z.size - 4, 3 * specials.size)
    if k > 0:
        z.reshape(-1)[rng.choice(z.size, k, replace=False)] = np.resize(specials, k)
    z[-1, -1] = -0.0
    z[-1, 0] = tiny
    z[0, -1] = -5 * tiny
    if nx > 2:
        z[-1, nx // 2] = np.inf
    if ny > 2:
        z[ny // 2, -1] = np.nan
    return z


def walk(k, dt):
    """Queries along one axis (knots k) that take the grid kernel's column cache through each of its cases:
    every knot in order (the new bracket starts where the old one ended), the last knot alternating with the other
    knots (a bracket with bx == ax next to ordinary ones), long runs of one value, a descending run, out-of-range and
    NaN queries between two queries on one bracket, +-inf, and the neighbours of both ends."""
    k = np.asarray(k, dt)
    lo, hi = k[0], k[-1]
    inner = k[:-1][np.unique(np.linspace(0, k.size - 2, min(k.size - 1, 24)).astype(int))]
    inner = np.concatenate([inner, k[-2:-1]])             # ... including the last-but-one knot (ax == previous bx)
    j = k.size // 2 if k.size > 2 else 0
    a, b = k[j] + (k[j + 1] - k[j]) / dt(4), k[j] + (k[j + 1] - k[j]) * dt(0.75)    # two queries in one bracket
    far = (hi - lo) / dt(8)
    s = max(1, k.size // 30)
    parts = [
        k,
        np.stack([np.full(inner.size, hi), inner], 1).ravel(),
        np.full(40, k[j]), np.full(40, a),
        np.sort(np.concatenate([k[::s], (k[:-1:s] + k[1::s]) / dt(2)]))[::-1],
        [a, lo - far, b, a, np.nan, b, b, hi + far, a, hi, np.nan, hi, hi, lo - far, hi],
        [np.inf, a, -np.inf, b],
        [np.nextafter(lo, dt(-np.inf)), lo, np.nextafter(lo, dt(np.inf)),
         np.nextafter(hi, dt(-np.inf)), hi, np.nextafter(hi, dt(np.inf))],
    ]
    return np.concatenate([np.asarray(p, dt) for p in parts])


def queries(rng, k, n, dt):
    """walk(k) followed by uniform queries over the axis and 5 % beyond it, n in all"""
    w = walk(k, dt)
    assert n >= w.size
    span = float(k[-1] - k[0])
    return np.concatenate([w, rng.uniform(k[0] - 0.05 * span, k[-1] + 0.05 * span, n - w.size).astype(dt)])


# ---- the benchmark's grid at full size ----

def bench_queries(torch):
    """XI and YI as bench.py draws them: 1e4 sorted uniform values each from one seeded CUDA generator, XI first"""
    g = torch.Generator(device="cuda").manual_seed(2236)
    xi = torch.rand(10_000, generator=g, device="cuda", dtype=torch.float64).sort().values
    yi = torch.rand(10_000, generator=g, device="cuda", dtype=torch.float64).sort().values
    return xi, yi


def test_benchmark_grid_every_output(b200, oracle):
    """The 1e4 x 1e4 grid bench.py times, on the benchmark's plans (4096^2 linspace axes; f64 with tiles, f32 on
    column-major Z): all 1e8 outputs in both pass orders and both types, and the host call (24 column blocks in two
    alternating slots, the last one ragged) with the device call's bits."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    P = b200.Interp2Plan
    xi, yi = bench_queries(torch)
    hxi, hyi = xi.cpu().numpy(), yi.cpu().numpy()

    plan = P(x, y, z)
    dev = plan.grid(xi, yi).cpu().numpy()
    assert same_as_oracle(dev, oracle.interp2_grid(x, y, z, hxi, hyi, nthreads=NT))
    cols = HOST_BLOCK_BYTES // (hyi.size * 8)
    assert (cols, -(-hxi.size // cols), hxi.size % cols) == (419, 24, 363)
    assert same_ints(plan.grid(hxi, hyi), dev)
    plan.close()
    del dev

    plan = P(x, y, z, flags=P.ORDER_YX)
    dev = plan.grid(xi, yi).cpu().numpy()
    assert same_as_oracle(dev, oracle.interp2_grid(x, y, z, hxi, hyi, nthreads=NT, y_first=True))
    plan.close()
    del dev

    x32, y32, z32 = x.astype(np.float32), y.astype(np.float32), z.astype(np.float32)
    xi32, yi32 = xi.to(torch.float32), yi.to(torch.float32)
    plan = P(x32, y32, z32)
    dev = plan.grid(xi32, yi32).cpu().numpy()
    assert same_as_oracle(dev, oracle.interp2_grid(x32, y32, z32, xi32.cpu().numpy(), yi32.cpu().numpy(), nthreads=NT))
    plan.close()


# ---- every kernel build, every output alignment ----

def test_every_grid_kernel_build_at_every_output_alignment(b200, oracle):
    """f64 / f32 x both pass orders x nyi in {4k, 4k+2, 4k+1} x ZI at 0, 1 or 2 elements past an aligned address:
    the outputs equal the oracle's and nothing outside ZI is written.  The cases must reach all twelve builds
    interp2_grid_kernel<T, V, YFIRST> under plan2_grid_main's rule for V."""
    import torch
    P = b200.Interp2Plan
    builds = set()
    for dt in (np.float64, np.float32):
        rng = np.random.default_rng(51)
        x, y = ragged(rng, 70, dt), ragged(rng, 50, dt)
        z = special_z(rng, y.size, x.size, dt)
        xi = queries(rng, x, 10 * GRID_COLS + 5, dt)          # ten full column tiles and a ragged one
        esz = np.dtype(dt).itemsize
        for y_first in (False, True):
            plan = P(x, y, z, flags=P.ORDER_YX if y_first else 0)
            for nyi in (1200, 1202, 1201):                   # over several 128-thread blocks of rows at any V
                yi = queries(rng, y, nyi, dt)
                ref = oracle.interp2_grid(x, y, z, xi, yi, extrap=0.75, nthreads=NT, y_first=y_first)
                txi, tyi = torch.from_numpy(xi).cuda(), torch.from_numpy(yi).cuda()
                for offset in (0, 1, 2):
                    rc, got, addr = grid_dev(plan, txi, tyi, 0.75, offset)
                    v = kernel_rows(nyi, addr, esz)
                    case = (np.dtype(dt).name, y_first, nyi, offset, v)
                    assert rc == 0, case
                    assert same_as_oracle(got, ref), case
                    builds.add((np.dtype(dt).name, v, y_first))
            plan.close()
    assert builds == {(t, v, f) for t in ("float64", "float32") for v in (1, 2, 4) for f in (False, True)}


# ---- launch and column-block boundaries ----

def check_empty_calls(plan, dt):
    """nxi = 0 or nyi = 0: status 0 and nothing written, on the device and the host call"""
    import torch
    q = np.linspace(0.0, 1.0, 5).astype(dt)
    tq = torch.from_numpy(q).cuda()
    empty, tempty = q[:0], tq[:0]
    for a, b in ((empty, q), (q, empty)):
        assert grid_host(plan, a, b, 0.5)[0] == 0
    for a, b in ((tempty, tq), (tq, tempty)):
        assert grid_dev(plan, a, b, 0.5)[0] == 0


@pytest.mark.parametrize("dt,nyi,y_first", [(np.float64, 4, False), (np.float32, 3, True)])
def test_device_call_over_two_launches(b200, oracle, dt, nyi, y_first):
    """nxi = 65535 * 32 + 77 columns: the device call launches twice, the second time from column k_begin > 0."""
    import torch
    rng = np.random.default_rng(52)
    x, y = ragged(rng, 300, dt), ragged(rng, 200, dt)
    z = special_z(rng, y.size, x.size, dt)
    nxi = COLS_PER_LAUNCH + 77
    # unsorted, so that no column tile of the second launch repeats the first launch's
    xi = rng.uniform(x[0] - 1, x[-1] + 1, nxi).astype(dt)
    w = walk(x, dt)
    xi[-w.size:] = w
    xi[:w.size] = w[::-1]
    yi = np.array([y[0], y[-1], y[7] + (y[8] - y[7]) / dt(3), np.nan], dt)[:nyi]
    P = b200.Interp2Plan
    plan = P(x, y, z, flags=P.ORDER_YX if y_first else 0)
    rc, got, _ = grid_dev(plan, torch.from_numpy(xi).cuda(), torch.from_numpy(yi).cuda(), 1.5)
    assert rc == 0
    assert same_as_oracle(got, oracle.interp2_grid(x, y, z, xi, yi, extrap=1.5, nthreads=NT, y_first=y_first))
    check_empty_calls(plan, dt)
    plan.close()


def test_host_call_one_column_per_block(b200, oracle):
    """nyi = 2^22 + 3 f64 rows: one column of ZI is over the host call's 32 MiB block, so each block is one column,
    alternating between the two slots; the device call gives the same bits."""
    import torch
    rng = np.random.default_rng(53)
    x, y = ragged(rng, 300, np.float64), ragged(rng, 200, np.float64)
    z = special_z(rng, y.size, x.size, np.float64)
    nyi = (1 << 22) + 3
    assert HOST_BLOCK_BYTES // (nyi * 8) == 0
    xi = np.array([x[0], x[150] + 0.3, np.nan, x[-1], x[-1] + 2.0])
    yi = queries(rng, y, nyi, np.float64)
    plan = b200.Interp2Plan(x, y, z)
    rc, host = grid_host(plan, xi, yi, -2.0)
    assert rc == 0
    assert same_as_oracle(host, oracle.interp2_grid(x, y, z, xi, yi, extrap=-2.0, nthreads=NT))
    rc, dev, _ = grid_dev(plan, torch.from_numpy(xi).cuda(), torch.from_numpy(yi).cuda(), -2.0)
    assert rc == 0 and same_ints(dev, host)
    check_empty_calls(plan, np.float64)
    plan.close()


# ---- query orders and special values ----

def plan_axes(kind, dt):
    rng = np.random.default_rng(54)
    if kind == "2x2":
        return np.array([-1.5, 2.0], dt), np.array([0.25, 3.0], dt)
    if kind == "ragged":
        return ragged(rng, 300, dt), ragged(rng, 200, dt)
    if kind == "affine":
        return np.linspace(-1.0, 2.0, 257).astype(dt), np.linspace(0.0, 1.0, 129).astype(dt)
    return ragged(rng, 20_000, dt), ragged(rng, 16, dt)      # "long_x": the X axis is 20 000 knots long


@pytest.mark.parametrize("kind", ["2x2", "ragged", "affine", "long_x"])
@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_query_orders_and_special_values(b200, oracle, dt, y_first, kind):
    """walk() on both axes, Z with special values, extrap NaN, finite and +inf (where (1-0)*inf + 0*inf is NaN), on
    the host and the device call.  The grid reads only column-major Z, so every plan layout gives the same bits."""
    import torch
    P = b200.Interp2Plan
    x, y = plan_axes(kind, dt)
    rng = np.random.default_rng(55)
    z = special_z(rng, y.size, x.size, dt)
    xi, yi = queries(rng, x, walk(x, dt).size + 37, dt), queries(rng, y, walk(y, dt).size + 29, dt)
    txi, tyi = torch.from_numpy(xi).cuda(), torch.from_numpy(yi).cuda()
    layouts = [0, P.FORCE_CELLS, P.FORCE_TILES, P.NO_CELLS | P.NO_TILES, P.FORCE_CELLS | P.FORCE_BANDS] \
        if kind == "ragged" else [0]
    refs = {e: oracle.interp2_grid(x, y, z, xi, yi, extrap=e, nthreads=NT, y_first=y_first)
            for e in (np.nan, 1.75, np.inf)}
    for layout in layouts:
        plan = P(x, y, z, flags=layout | (P.ORDER_YX if y_first else 0))
        for e, ref in refs.items():
            assert same_as_oracle(plan.grid(xi, yi, extrap=e), ref), (layout, e)
            dev = plan.grid(txi, tyi, extrap=e)
            torch.cuda.synchronize()
            assert same_as_oracle(dev.cpu().numpy(), ref), (layout, e)
        plan.close()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_one_shot_interp2_over_several_host_blocks(b200, oracle, dt):
    """b200.interp2 (b200_interp2_f64 / _f32: plan, host grid call, destroy) on a ragged 3000 x 3000 grid with a ZI
    of several 32 MiB column blocks."""
    rng = np.random.default_rng(56)
    x, y = ragged(rng, 3000, dt), ragged(rng, 3000, dt)
    z = special_z(rng, y.size, x.size, dt)
    xi, yi = np.sort(queries(rng, x, 4000, dt)), queries(rng, y, 5000, dt)
    assert xi.size * yi.size * np.dtype(dt).itemsize > 2 * HOST_BLOCK_BYTES
    assert same_as_oracle(b200.interp2(x, y, z, xi, yi, extrap=-0.5),
                          oracle.interp2_grid(x, y, z, xi, yi, extrap=-0.5, nthreads=NT))


# ---- operand checks of the value calls on CUDA tensors ----

def test_device_value_calls_reject_bad_operands(b200):
    """A tensor of the other dtype, a strided view, a YQ longer than XQ and a wrong `out` raise TypeError or
    ValueError, and the plans give the same bits afterwards.  Every misuse stays inside its allocation (larger
    tensors, views of longer storage), so even a wrapper without the checks would touch no foreign memory."""
    import torch
    rng = np.random.default_rng(57)
    x = np.linspace(0.0, 1.0, 40); y = np.linspace(0.0, 1.0, 30); z = rng.standard_normal((30, 40))
    n = 1000
    big = torch.rand(2 * n + 1, device="cuda", dtype=torch.float64)
    xq, yq = big[:n], big[n:2 * n]
    p2 = {np.float64: b200.Interp2Plan(x, y, z), np.float32: b200.Interp2Plan(x.astype(np.float32),
                                                                             y.astype(np.float32), z.astype(np.float32))}
    p1 = {np.float64: b200.Interp1Plan(x, z[0]), np.float32: b200.Interp1Plan(x.astype(np.float32),
                                                                             z[0].astype(np.float32))}
    ops = {np.float64: (xq, yq), np.float32: (xq.float(), yq.float())}

    def results():
        out = []
        for dt, (a, b) in ops.items():
            out += [p2[dt].grid(a, b[:50]), p2[dt].scattered(a, b), p1[dt](a)]
        torch.cuda.synchronize()
        return [t.cpu().numpy() for t in out]

    before = results()
    x32, y32 = ops[np.float32]
    wide32 = torch.empty(2 * n, device="cuda", dtype=torch.float32)        # n f32 views of 8n bytes
    bad = [
        (TypeError, lambda: p2[np.float32].grid(xq, y32)),                  # float64 tensor on an f32 plan
        (TypeError, lambda: p2[np.float32].grid(x32, yq)),
        (TypeError, lambda: p2[np.float32].scattered(xq, y32)),
        (TypeError, lambda: p2[np.float32].scattered(x32, yq)),
        (TypeError, lambda: p1[np.float32](xq)),
        (TypeError, lambda: p2[np.float64].grid(big[::2], yq)),             # strided views
        (TypeError, lambda: p2[np.float64].grid(xq, big[::2])),
        (TypeError, lambda: p2[np.float64].scattered(big[::2][:n], yq)),
        (TypeError, lambda: p2[np.float64].scattered(xq, big[1::2])),
        (TypeError, lambda: p1[np.float64](big[::2])),
        (ValueError, lambda: p2[np.float64].scattered(xq, big[n:])),       # YQ longer than XQ
        (ValueError, lambda: p2[np.float64].scattered(xq, yq, out=torch.empty(n + 1, device="cuda", dtype=torch.float64))),
        (TypeError, lambda: p2[np.float64].scattered(xq, yq, out=wide32[:n])),
        (TypeError, lambda: p2[np.float64].scattered(xq, yq, out=torch.empty(2 * n, device="cuda", dtype=torch.float64)[::2])),
        (ValueError, lambda: p1[np.float64](xq, out=torch.empty(n + 1, device="cuda", dtype=torch.float64))),
        (TypeError, lambda: p1[np.float64](xq, out=wide32[:n])),
        (TypeError, lambda: p1[np.float64](xq, out=torch.empty(2 * n, device="cuda", dtype=torch.float64)[::2])),
    ]
    for i, (err, call) in enumerate(bad):
        with pytest.raises(err):
            call()
        torch.cuda.synchronize()
        assert all(same_ints(a, b) for a, b in zip(results(), before)), i
