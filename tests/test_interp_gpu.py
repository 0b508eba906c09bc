"""GPU parity tests of interp1 / interp2 through the C-ABI: bit-exact values and bracket
indices against the CPU oracle and the committed golden fixtures; size-independent properties
at BASELINE.json's full sizes."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "interp_golden.npz"))


def same_bits(a, b):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("kind", ["uniform", "general", "two"])
def test_interp1_golden(b200, tag, kind):
    g = lambda k: GOLD[f"i1_{tag}_{kind}_{k}"]
    yi, idx = b200.interp1(g("xg"), g("yg"), g("xi"), extrap=-7.0, return_index=True)
    assert same_bits(yi, g("yi"))           # bit-exact blend
    assert np.array_equal(idx, g("idx"))    # bit-exact bracket


@pytest.mark.parametrize("tag", ["f64", "f32"])
@pytest.mark.parametrize("y_first", [False, True])
def test_interp2_golden(b200, tag, y_first):
    """Both orders of Armadillo's two separable passes (default: along X, then Y; B200_INTERP2_ORDER_YX: the
    mirrored order), every layout of the scattered path and the tensor-grid kernel, including the corner cases
    that tell the orders apart: NaN in one coordinate with the other out of range (the LAST pass decides) and a
    finite extrap value blended with itself by the second pass."""
    g = lambda k: GOLD[f"i2_{tag}_{k}"]
    sfx = "_yx" if y_first else ""
    P = b200.Interp2Plan
    order = P.ORDER_YX if y_first else 0
    for layout in (0, P.FORCE_CELLS, P.FORCE_TILES, P.NO_CELLS | P.NO_TILES, P.FORCE_CELLS | P.FORCE_BANDS):
        plan = P(g("x"), g("y"), g("z"), flags=order | layout)
        assert same_bits(plan.scattered(g("xq"), g("yq"), extrap=3.5), g("zq" + sfx)), layout
        if layout & P.FORCE_BANDS:     # the banded pipeline serves device buffers
            import torch
            zq = plan.scattered(torch.from_numpy(g("xq")).cuda(), torch.from_numpy(g("yq")).cuda(), extrap=3.5)
            torch.cuda.synchronize()
            assert same_bits(zq.cpu().numpy(), g("zq" + sfx))
        assert same_bits(plan.grid(g("xi"), g("yi")), g("zi" + sfx))
        assert same_bits(plan.grid(g("xi"), g("yi"), extrap=3.5), g("zi_e" + sfx))
    if not y_first:
        assert same_bits(b200.interp2(g("x"), g("y"), g("z"), g("xi"), g("yi")), g("zi"))
    # the two orders agree to rounding wherever both are finite
    a, b = g("zq"), g("zq_yx")
    ok = ~np.isnan(a) & ~np.isnan(b)
    assert np.max(np.abs(a[ok] - b[ok])) <= 4 * np.finfo(a.dtype).eps * max(1.0, np.max(np.abs(a[ok])))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("kind,expect_mode", [("linspace", None), ("cumsum", 1), ("clustered", 1), ("pow2", 0)])
def test_interp1_vs_oracle(b200, oracle, dt, kind, expect_mode):
    rng = np.random.default_rng(11)
    ng = 200001
    if kind == "linspace":
        xg = np.linspace(0.0, 1.0, ng)
    elif kind == "pow2":
        xg = np.arange(ng, dtype=np.float64) / 262144.0           # exactly uniform in binary
    elif kind == "cumsum":
        xg = np.cumsum(0.5 + rng.random(ng)); xg = (xg - xg[0]) / (xg[-1] - xg[0])
    else:  # pathological: most knots packed into a sliver (exercises the bounded binary search)
        xg = np.concatenate([np.linspace(0, 1e-3, ng - 100), np.linspace(0.1, 1.0, 100)])
    xg = np.unique(xg.astype(dt))
    yg = (np.sin(2 * np.pi * xg) + 0.1 * rng.standard_normal(xg.size)).astype(dt)
    xi = rng.uniform(-0.01, 1.01, 1_000_003).astype(dt)                   # odd length: scalar tail
    xi[:6] = [xg[0], xg[-1], np.nan, xg[7], xg[-2], np.nextafter(xg[-1], dt(2))]
    xi[1000:1100] = xg[500:600]                                           # exact knot hits
    plan = b200.Interp1Plan(xg, yg)
    if expect_mode is not None:
        assert plan.lookup_mode == expect_mode
    yi, idx = plan(xi, extrap=-3.0, return_index=True)
    yo, io = oracle.interp1(xg, yg, xi, extrap=-3.0, nthreads=8)
    assert same_bits(yi, yo)
    assert np.array_equal(idx, io)
    # sorted queries (Armadillo's internal order) against Armadillo's literal scan
    xs = np.sort(xi[~np.isnan(xi)])
    ys, ids = plan(xs, extrap=-3.0, return_index=True)
    yo, io = oracle.interp1(xg, yg, xs, extrap=-3.0, scan=True)
    assert same_bits(ys, yo) and np.array_equal(ids, io)


def test_interp1_device_buffers_unaligned_and_values_update(b200, oracle):
    import torch
    rng = np.random.default_rng(12)
    xg = np.cumsum(0.5 + rng.random(5000)); yg = rng.standard_normal(5000)
    plan = b200.Interp1Plan(xg, yg)
    xi = rng.uniform(xg[0], xg[-1], 100001)
    t = torch.from_numpy(xi).cuda()
    y = plan(t)                                   # aligned device buffers: vector kernel
    torch.cuda.synchronize()
    assert same_bits(y.cpu().numpy(), oracle.interp1(xg, yg, xi, want_idx=False))
    y = plan(t[1:].contiguous()[1:])              # fresh aligned copy
    t2 = t[1:]                                    # 8-byte offset view: unaligned -> scalar kernel
    out = torch.empty(t2.numel() + 1, dtype=torch.float64, device="cuda")[1:]
    plan(t2, out=out)
    torch.cuda.synchronize()
    assert same_bits(out.cpu().numpy(), oracle.interp1(xg, yg, xi[1:], want_idx=False))
    yg2 = rng.standard_normal(5000)               # new coarse profile on the same knots
    plan.set_values(yg2)
    assert same_bits(plan(xi), oracle.interp1(xg, yg2, xi, want_idx=False))
    assert plan(np.array([])).size == 0           # empty batch


def test_interp1_errors(b200):
    with pytest.raises(b200.B200Error) as e:
        b200.interp1(np.array([0.0, 0.0, 1.0]), np.zeros(3), np.array([0.5]))
    assert e.value.status == -3
    with pytest.raises(b200.B200Error) as e:
        b200.interp1(np.array([0.0]), np.zeros(1), np.array([0.5]))
    assert e.value.status == -4
    with pytest.raises(b200.B200Error) as e:
        b200.interp1(np.array([0.0, np.nan, 1.0]), np.zeros(3), np.array([0.5]))
    assert e.value.status == -7


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_interp2_vs_oracle(b200, oracle, dt):
    rng = np.random.default_rng(13)
    nx, ny = 513, 384
    x = np.unique(np.cumsum(0.5 + rng.random(nx)).astype(dt)); y = np.linspace(-2, 3, ny).astype(dt)
    z = rng.standard_normal((y.size, x.size)).astype(dt)
    plan = b200.Interp2Plan(x, y, z)
    nq = 300_001
    xq = rng.uniform(x[0] - 1, x[-1] + 1, nq).astype(dt); yq = rng.uniform(-2.1, 3.1, nq).astype(dt)
    xq[:5] = [x[0], x[-1], np.nan, x[3], x[-1]]; yq[:5] = [y[0], y[-1], 0.0, np.nan, y[0]]
    for extrap in (np.nan, 2.25):
        assert same_bits(plan.scattered(xq, yq, extrap=extrap), oracle.interp2_scattered(x, y, z, xq, yq, extrap=extrap, nthreads=8))
    xi = rng.uniform(x[0] - 1, x[-1] + 1, 333).astype(dt)
    for nyi in (1000, 1002, 777):                # multiple of 4: 32-byte stores, even: 16-byte, odd: scalar
        yi = rng.uniform(-2.1, 3.1, nyi).astype(dt)
        assert same_bits(plan.grid(xi, yi, extrap=0.5), oracle.interp2_grid(x, y, z, xi, yi, extrap=0.5, nthreads=8))


def test_interp2_device_buffers(b200, oracle):
    import torch
    rng = np.random.default_rng(14)
    x = np.linspace(0, 1, 256); y = np.linspace(0, 1, 128); z = rng.standard_normal((128, 256))
    plan = b200.Interp2Plan(x, y, z)
    xq = rng.random(50000); yq = rng.random(50000)
    zq = plan.scattered(torch.from_numpy(xq).cuda(), torch.from_numpy(yq).cuda())
    torch.cuda.synchronize()
    assert same_bits(zq.cpu().numpy(), oracle.interp2_scattered(x, y, z, xq, yq))
    zi = plan.grid(torch.from_numpy(xq[:100]).cuda(), torch.from_numpy(yq[:64]).cuda())
    torch.cuda.synchronize()
    assert same_bits(zi.cpu().numpy(), oracle.interp2_grid(x, y, z, xq[:100], yq[:64]))


def _config1_inputs(kind):
    """BASELINE config 1 exactly as bench.py builds it (1e6 knots; SURVEY 8d seeds)."""
    ng = 1_000_000
    rng = np.random.default_rng(1234)
    xg = np.linspace(0.0, 1.0, ng) if kind == "uniform" else np.cumsum(0.5 + rng.random(ng))
    xg = (xg - xg[0]) / (xg[-1] - xg[0])
    yg = np.sin(2 * np.pi * xg) + 0.1 * np.random.default_rng(1235).standard_normal(ng)
    return xg, yg


@pytest.mark.parametrize("kind", ["uniform", "nonuniform"])
@pytest.mark.parametrize("order", ["unsorted", "sorted"])
def test_full_size_config1_bit_exact(b200, oracle, kind, order):
    """BASELINE config 1 at its stated size — 1e6 knots x 1e7 queries, the bench's knots, values and
    seeds — compared with the oracle on EVERY query: values bit for bit, bracket indices equal
    (oracle = restatement of arma::interp1's interp1_helper_linear; parity with a real Armadillo
    build is unpinned, Armadillo being absent from the image)."""
    xg, yg = _config1_inputs(kind)
    ni = 10_000_000
    xi = np.random.default_rng(1236).uniform(xg[0], xg[-1], ni)
    if order == "sorted":
        xi.sort()
    xi[:3] = [xg[0], xg[-1], xg[ni % xg.size]]
    plan = b200.Interp1Plan(xg, yg)
    yi, idx = plan(xi, return_index=True)
    yo, io = oracle.interp1(xg, yg, xi, nthreads=os.cpu_count() or 8)
    assert same_bits(yi, yo)
    assert np.array_equal(idx, io)
    # size-independent properties on top: brackets bracket, knot hits return the knot value
    ng = xg.size
    assert idx.min() >= 0 and idx.max() <= ng - 1
    assert np.all(xg[idx] <= xi) and np.all(xi[idx < ng - 1] < xg[np.minimum(idx + 1, ng - 1)][idx < ng - 1])
    hits = plan(xg[::997], return_index=True)
    assert np.array_equal(hits[0], yg[::997]) and np.array_equal(hits[1], np.arange(ng)[::997])


def test_full_size_config2_headline_plan_bit_exact(b200, oracle):
    """BASELINE config 2 at its stated size through the HEADLINE plan of bench.py: the 4096^2 f64 grid of
    seed 2234 with the default layout (overlapping 4x4 tiles, linspace axes recognised as affine) and all
    1e8 queries of seed 2235 (torch's CUDA generator, as in the bench), every output compared bit for bit
    with the oracle (restatement of arma::interp2 per point; Armadillo itself is absent, parity unpinned).
    Also the host-buffer (e2e) path and a linear-reproduction property."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    plan = b200.Interp2Plan(x, y, z)
    g = torch.Generator(device="cuda").manual_seed(2235)
    nq = bench.NQ
    xq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
    yq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64)
    zq = plan.scattered(xq, yq)
    torch.cuda.synchronize()
    hx, hy, hz = xq.cpu().numpy(), yq.cpu().numpy(), zq.cpu().numpy()
    ref = oracle.interp2_scattered(x, y, z, hx, hy, nthreads=os.cpu_count() or 8)
    assert same_bits(hz, ref)
    # host-buffer C-ABI path (pageable numpy buffers): same bits on all 1e8 outputs
    assert same_bits(plan.scattered(hx, hy), ref)
    del ref, hz
    # property at full size: a bilinear function is reproduced to rounding
    zb = (2.0 * x[None, :] - 0.5) * (0.25 * y[:, None] + 1.0)
    pb = b200.Interp2Plan(x, y, zb)
    err = (pb.scattered(xq, yq) - (2.0 * xq - 0.5) * (0.25 * yq + 1.0)).abs().max().item()
    assert err < 5e-15


def test_interp2_banded_then_grid_then_banded_one_plan(b200, oracle):
    """Regression (round-1 advisor finding): the grid prologue used to free the banded pipeline's scratch
    without resetting its capacity, so banded -> grid -> banded on ONE plan ran on freed memory."""
    import torch
    rng = np.random.default_rng(23)
    x = np.unique(np.cumsum(0.5 + rng.random(513))); y = np.linspace(-2, 3, 384)
    z = rng.standard_normal((y.size, x.size))
    plan = b200.Interp2Plan(x, y, z, flags=b200.Interp2Plan.FORCE_CELLS | b200.Interp2Plan.FORCE_BANDS)
    nq = 300_001
    xq = rng.uniform(x[0], x[-1], nq); yq = rng.uniform(-2, 3, nq)
    tx, ty = torch.from_numpy(xq).cuda(), torch.from_numpy(yq).cuda()
    ref = oracle.interp2_scattered(x, y, z, xq, yq, nthreads=8)
    z1 = plan.scattered(tx, ty); torch.cuda.synchronize()
    assert same_bits(z1.cpu().numpy(), ref)
    xi = np.sort(rng.uniform(x[0], x[-1], 700)); yi = np.sort(rng.uniform(-2, 3, 300))
    assert same_bits(plan.grid(xi, yi), oracle.interp2_grid(x, y, z, xi, yi))       # first grid call: allocates
    z2 = plan.scattered(tx, ty); torch.cuda.synchronize()
    assert same_bits(z2.cpu().numpy(), ref)
    xi2 = np.sort(rng.uniform(x[0], x[-1], 1500))
    assert same_bits(plan.grid(xi2, yi), oracle.interp2_grid(x, y, z, xi2, yi))     # larger: re-allocates
    z3 = plan.scattered(tx, ty); torch.cuda.synchronize()
    assert same_bits(z3.cpu().numpy(), ref)
    plan.close()


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_interp2_axes_too_large_for_shared_memory(b200, oracle, dt):
    """Knot vectors beyond the shared-memory budget fall back to the global-table kernel: same bits."""
    rng = np.random.default_rng(15)
    nx, ny = (14500, 16) if dt == np.float64 else (29000, 16)
    x = np.unique(np.cumsum(0.5 + rng.random(nx)).astype(dt)); y = np.linspace(0, 1, ny).astype(dt)
    z = rng.standard_normal((y.size, x.size)).astype(dt)
    plan = b200.Interp2Plan(x, y, z)
    xq = rng.uniform(x[0], x[-1], 200_000).astype(dt); yq = rng.random(200_000).astype(dt)
    assert same_bits(plan.scattered(xq, yq), oracle.interp2_scattered(x, y, z, xq, yq, nthreads=8))


def test_interp2_layout_flags_give_identical_bits(b200, oracle):
    """Column-major gathers and 2x2 corner records are two layouts of the same arithmetic."""
    import ctypes as C
    from armadillocudalinearinterpolation_b200 import _lib
    rng = np.random.default_rng(16)
    x = np.linspace(0, 1, 300); y = np.linspace(0, 1, 200); z = np.asfortranarray(rng.standard_normal((200, 300)))
    xq = rng.uniform(-0.1, 1.1, 100_000); yq = rng.uniform(-0.1, 1.1, 100_000)
    ref = oracle.interp2_scattered(x, y, z, xq, yq, extrap=1.5)
    L = _lib.lib()
    for flags in (1, 2, 32):   # B200_INTERP2_NO_CELLS, B200_INTERP2_FORCE_CELLS, B200_INTERP2_FORCE_TILES
        h = C.c_void_p()
        _lib.check(L.b200_interp2_plan_create_ex(0, x.ctypes.data_as(C.c_void_p), C.c_size_t(x.size), y.ctypes.data_as(C.c_void_p),
                                                 C.c_size_t(y.size), z.ctypes.data_as(C.c_void_p), C.c_uint(flags), C.byref(h)))
        out = np.empty_like(xq)
        _lib.check(L.b200_interp2_scattered(h, xq.ctypes.data_as(C.c_void_p), yq.ctypes.data_as(C.c_void_p), C.c_size_t(xq.size),
                                            out.ctypes.data_as(C.c_void_p), C.c_double(1.5)))
        L.b200_interp2_plan_destroy(h)
        assert same_bits(out, ref)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("kind", ["linspace", "cumsum", "clustered"])
def test_interp1_small_grid_shared_memory_path(b200, oracle, dt, kind):
    """Coarse profile -> fine ensemble: grids of a few thousand knots are staged in shared memory
    (lookup mode 2); same bits and brackets as the oracle."""
    rng = np.random.default_rng(17)
    ng = 4001
    if kind == "linspace":
        xg = np.linspace(-3.0, 3.0, ng)
    elif kind == "cumsum":
        xg = np.cumsum(0.5 + rng.random(ng))
    else:
        xg = np.concatenate([np.linspace(0, 1e-3, ng - 50), np.linspace(0.1, 1.0, 50)])
    xg = np.unique(xg.astype(dt))
    yg = rng.standard_normal(xg.size).astype(dt)
    xi = rng.uniform(xg[0] - 0.1, xg[-1] + 0.1, 1_000_001).astype(dt)
    xi[:4] = [xg[0], xg[-1], np.nan, xg[17]]
    plan = b200.Interp1Plan(xg, yg)
    assert plan.lookup_mode == 2
    yi, idx = plan(xi, extrap=0.25, return_index=True)
    yo, io = oracle.interp1(xg, yg, xi, extrap=0.25, nthreads=8)
    assert same_bits(yi, yo) and np.array_equal(idx, io)
    yg2 = rng.standard_normal(xg.size).astype(dt)
    plan.set_values(yg2)                                    # a new coarse profile on the same knots
    assert same_bits(plan(xi, extrap=0.25), oracle.interp1(xg, yg2, xi, extrap=0.25, want_idx=False, nthreads=8))


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("shape", [(513, 384, 300_001), (64, 50, 2047), (64, 50, 4097), (300, 200, 5), (1000, 37, 1_000_003)])
def test_interp2_banded_pipeline_same_bits(b200, oracle, dt, shape):
    """The L2-banded scattered pipeline (partition by column band -> interpolate band by band ->
    un-permute; B200_INTERP2_FORCE_BANDS) is a re-ordering of the same arithmetic: same bits as the
    oracle, including NaN / out-of-range queries in either coordinate, ragged tails and infinite extrap."""
    import torch
    nx, ny, nq = shape
    rng = np.random.default_rng(18)
    x = np.unique(np.cumsum(0.5 + rng.random(nx)).astype(dt)); y = np.linspace(-2, 3, ny).astype(dt)
    z = rng.standard_normal((y.size, x.size)).astype(dt)
    plan = b200.Interp2Plan(x, y, z, flags=b200.Interp2Plan.FORCE_CELLS | b200.Interp2Plan.FORCE_BANDS)
    xq = rng.uniform(x[0] - 1, x[-1] + 1, nq).astype(dt); yq = rng.uniform(-2.1, 3.1, nq).astype(dt)
    xq[:5] = [x[0], x[-1], np.nan, x[3], x[-1]]; yq[:5] = [y[0], y[-1], 0.0, np.nan, y[0]]
    for extrap in (np.nan, 2.25, np.inf):
        zq = plan.scattered(torch.from_numpy(xq).cuda(), torch.from_numpy(yq).cuda(), extrap=extrap)
        torch.cuda.synchronize()
        assert same_bits(zq.cpu().numpy(), oracle.interp2_scattered(x, y, z, xq, yq, extrap=extrap, nthreads=8))
    # unaligned device buffers take the scalar load/store path of the same kernels
    tx = torch.from_numpy(xq).cuda()[1:]; ty = torch.from_numpy(yq).cuda()[1:]
    out = torch.empty(nq, dtype=tx.dtype, device="cuda")[1:]
    plan.scattered(tx, ty, extrap=0.5, out=out)
    torch.cuda.synchronize()
    assert same_bits(out.cpu().numpy(), oracle.interp2_scattered(x, y, z, xq[1:], yq[1:], extrap=0.5, nthreads=8))


def test_interp2_affine_axes_same_bits(b200, oracle):
    """linspace-style knots (x0 + j*step with two roundings, verified knot by knot at plan time) are
    recomputed in the kernel instead of loaded; with one knot of each axis moved by one ulp the axes are
    not affine and the same queries take the tables.  Same bits."""
    rng = np.random.default_rng(19)
    x = np.linspace(-1.0, 2.0, 1500); y = np.linspace(0.0, 1.0, 700)
    xp = x.copy(); xp[500] = np.nextafter(xp[500], 5.0)
    yp = y.copy(); yp[300] = np.nextafter(yp[300], 5.0)
    z = rng.standard_normal((y.size, x.size))
    xq = rng.uniform(-1.1, 2.1, 400_003); yq = rng.uniform(-0.1, 1.1, 400_003)
    xq[:6] = [x[0], x[-1], np.nan, x[3], x[-2], np.nextafter(x[-1], 5.0)]; yq[:6] = [y[0], y[-1], 0.0, np.nan, y[-1], 0.5]
    for kx, ky in ((x, y), (xp, yp)):
        ref = oracle.interp2_scattered(kx, ky, z, xq, yq, extrap=-4.0, nthreads=8)
        for flags in (0, b200.Interp2Plan.FORCE_CELLS, b200.Interp2Plan.NO_CELLS):
            assert same_bits(b200.Interp2Plan(kx, ky, z, flags=flags).scattered(xq, yq, extrap=-4.0), ref)


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("shape", [(513, 384), (4, 4), (2, 2), (3, 7), (10, 5), (301, 299)])
def test_interp2_tile_layout_same_bits(b200, oracle, dt, shape):
    """Overlapping 4x4 tiles (B200_INTERP2_FORCE_TILES): every cell's corners in one 128-byte line.
    Grid sizes around the tile stride (3) exercise the clamped last row / column of tiles."""
    nx, ny = shape
    rng = np.random.default_rng(20)
    x = np.unique(np.cumsum(0.5 + rng.random(nx)).astype(dt)); y = np.linspace(-2, 3, ny).astype(dt)
    z = rng.standard_normal((y.size, x.size)).astype(dt)
    plan = b200.Interp2Plan(x, y, z, flags=b200.Interp2Plan.FORCE_TILES)
    nq = 200_003
    xq = rng.uniform(x[0] - 0.5, x[-1] + 0.5, nq).astype(dt); yq = rng.uniform(-2.1, 3.1, nq).astype(dt)
    xq[:5] = [x[0], x[-1], np.nan, x[1], x[-1]]; yq[:5] = [y[0], y[-1], 0.0, np.nan, y[0]]
    xq[5:5 + x.size] = x; yq[5:5 + x.size] = y[-1]              # every x knot on the last row
    xq[1000:1000 + y.size] = x[-1]; yq[1000:1000 + y.size] = y   # every y knot on the last column
    for extrap in (np.nan, -1.5):
        assert same_bits(plan.scattered(xq, yq, extrap=extrap), oracle.interp2_scattered(x, y, z, xq, yq, extrap=extrap, nthreads=8))


def test_affine_detection_is_exact(b200, oracle):
    """One knot moved by one ulp makes an axis non-affine (the plan-time check is knot by knot, bit by bit):
    the table path must then be taken and give the oracle's bits; so must the affine path on the clean axis."""
    rng = np.random.default_rng(21)
    for n in (1000, 8000):                       # shared-memory interp1 path / also large enough for tiles etc.
        x = np.linspace(-1.0, 1.0, n); xp = x.copy(); xp[n // 3] = np.nextafter(xp[n // 3], 2.0)
        y = rng.standard_normal(n)
        xi = rng.uniform(-1.05, 1.05, 300_001); xi[:4] = [x[0], x[-1], xp[n // 3], x[n // 3]]
        for knots in (x, xp):
            yi, idx = b200.Interp1Plan(knots, y)(xi, extrap=0.5, return_index=True)
            yo, io = oracle.interp1(knots, y, xi, extrap=0.5, nthreads=8)
            assert same_bits(yi, yo) and np.array_equal(idx, io)
    x = np.linspace(0.0, 3.0, 257); xp = x.copy(); xp[5] = np.nextafter(xp[5], 0.0)
    yk = np.linspace(-1.0, 0.0, 129)
    z = rng.standard_normal((129, 257))
    xq = rng.uniform(-0.1, 3.1, 200_000); yq = rng.uniform(-1.1, 0.1, 200_000)
    for knots in (x, xp):
        for flags in (0, b200.Interp2Plan.FORCE_TILES, b200.Interp2Plan.NO_CELLS | b200.Interp2Plan.NO_TILES):
            got = b200.Interp2Plan(knots, yk, z, flags=flags).scattered(xq, yq, extrap=9.0)
            assert same_bits(got, oracle.interp2_scattered(knots, yk, z, xq, yq, extrap=9.0, nthreads=8))


def test_branch_free_divide_matches_ieee(b200):
    """The headline interp2 kernel divides with the fast path of the IEEE divide minus its range check
    (interp2.cu: div_rn_fast); inside its contract it must give __ddiv_rn's bits on every operand pair."""
    import ctypes as C
    from armadillocudalinearinterpolation_b200 import _lib
    bad = C.c_ulonglong(123)
    for seed in (1, 2, 3):
        _lib.check(_lib.lib().b200_selftest_div_fast(C.c_ulonglong(400_000_000), C.c_ulonglong(seed), C.byref(bad)))
        assert bad.value == 0


@pytest.mark.parametrize("y_first", [False, True])
def test_interp2_fast_kernel_special_queries(b200, oracle, y_first):
    """The straight-line kernel (both axes affine, tile layout, double) hands every query outside its common case
    to the generic path: out of range in either coordinate, NaN, knot hits, the last row / column, the first bin."""
    rng = np.random.default_rng(41)
    n = 600
    x = np.linspace(-1.0, 2.0, n); y = np.linspace(0.0, 1.0, n + 7)
    z = rng.standard_normal((y.size, x.size))
    nq = 400_003
    xq = rng.uniform(-1.2, 2.2, nq); yq = rng.uniform(-0.1, 1.1, nq)
    xq[:8] = [x[0], x[-1], np.nan, x[5], x[-1], x[0], np.nextafter(x[-1], 0), x[-2]]
    yq[:8] = [y[0], y[-1], 0.3, np.nan, y[0], y[-1], np.nextafter(y[-1], 0), y[-2]]
    xq[100:100 + n] = x; yq[100:100 + n] = rng.uniform(0, 1, n)          # every x knot
    xq[1000:1000 + y.size] = rng.uniform(-1, 2, y.size); yq[1000:1000 + y.size] = y   # every y knot
    flags = b200.Interp2Plan.FORCE_TILES | (b200.Interp2Plan.ORDER_YX if y_first else 0)
    plan = b200.Interp2Plan(x, y, z, flags=flags)
    for extrap in (np.nan, 4.5):
        ref = oracle.interp2_scattered(x, y, z, xq, yq, extrap=extrap, nthreads=8, y_first=y_first)
        assert same_bits(plan.scattered(xq, yq, extrap=extrap), ref)


@pytest.mark.parametrize("y_first", [False, True])
def test_interp2_locality_probe_both_kernels_same_bits(b200, oracle, y_first):
    """Large device-buffer batches on an affine/tile plan are served by one of two kernels, chosen on the device by a
    locality probe (cell-sorted queries -> the straight-line kernel, random queries -> the generic one): both choices
    give the oracle's bits — including special queries in the sorted stream."""
    import torch
    rng = np.random.default_rng(43)
    n = 1300
    x = np.linspace(0.0, 1.0, n); y = np.linspace(-1.0, 1.0, n)
    z = rng.standard_normal((n, n))
    nq = 2_000_003
    xq = rng.uniform(-0.01, 1.01, nq); yq = rng.uniform(-1.02, 1.02, nq)
    xq[:6] = [x[0], x[-1], np.nan, x[7], x[-1], 0.5]; yq[:6] = [y[0], y[-1], 0.1, np.nan, y[3], y[-1]]
    cell = np.clip((xq * (n - 1)).astype(np.int64), 0, n - 1) * n + np.clip(((yq + 1) / 2 * (n - 1)).astype(np.int64), 0, n - 1)
    order = np.argsort(np.nan_to_num(cell), kind="stable")
    flags = b200.Interp2Plan.FORCE_TILES | (b200.Interp2Plan.ORDER_YX if y_first else 0)
    ref = oracle.interp2_scattered(x, y, z, xq, yq, extrap=2.5, nthreads=8, y_first=y_first)
    plan = b200.Interp2Plan(x, y, z, flags=flags)
    for idx in (np.arange(nq), order):
        tx, ty = torch.from_numpy(xq[idx]).cuda(), torch.from_numpy(yq[idx]).cuda()
        zq = plan.scattered(tx, ty, extrap=2.5)
        torch.cuda.synchronize()
        assert same_bits(zq.cpu().numpy(), ref[idx])


def test_plans_run_on_their_own_device_and_restore_the_callers(b200, oracle):
    """A plan lives on the device that was current when it was created; host-buffer calls made while ANOTHER device is
    current still run there (same bits) and hand the caller's current device back."""
    import torch
    if b200.device_count() < 2:
        pytest.skip("needs at least two GPUs in this process")
    rng = np.random.default_rng(31)
    x = np.sort(rng.random(300)); y = np.sort(rng.random(200)); z = rng.standard_normal((200, 300))
    xq = rng.random(50_000) * 1.1 - 0.05; yq = rng.random(50_000) * 1.1 - 0.05
    torch.cuda.set_device(0)
    p2 = b200.Interp2Plan(x, y, z)
    p1 = b200.Interp1Plan(x, z[0])
    ref2 = oracle.interp2_scattered(x, y, z, xq, yq, extrap=3.0)
    ref1 = oracle.interp1(x, z[0], xq, extrap=3.0, want_idx=False)
    last = b200.device_count() - 1
    torch.cuda.set_device(last)
    try:
        assert same_bits(p2.scattered(xq, yq, extrap=3.0), ref2)
        assert torch.cuda.current_device() == last
        assert same_bits(p1(xq, extrap=3.0), ref1)
        assert torch.cuda.current_device() == last
        zi = p2.grid(xq[:64].copy(), yq[:32].copy(), extrap=3.0)
        assert same_bits(zi, oracle.interp2_grid(x, y, z, xq[:64], yq[:32], extrap=3.0))
        p1.close(); p2.close()
        assert torch.cuda.current_device() == last
    finally:
        torch.cuda.set_device(0)


def test_device_paths_capture_into_a_cuda_graph(b200, oracle):
    """The device-pointer entry points make no host round trip and allocate nothing after a first call of the same
    shape, so a caller can capture them into a CUDA graph (torch.cuda.CUDAGraph) and replay it on new data:
    interp1 (programmatic dependent launch), interp2 scattered (both kernels of the locality decision) and the
    tensor grid; every replay is bitwise the direct call."""
    import torch
    rng = np.random.default_rng(77)
    n = 1 << 21                                                   # >= 2^20: the scattered call launches both kernels
    x = np.linspace(0.0, 1.0, 700); y = np.linspace(-1.0, 1.0, 500); z = rng.standard_normal((500, 700))
    xg = np.sort(rng.random(5000)); yg = rng.standard_normal(5000)
    p2 = b200.Interp2Plan(x, y, z); p1 = b200.Interp1Plan(xg, yg)
    xq = torch.rand(n, device="cuda", dtype=torch.float64); yq = torch.rand(n, device="cuda", dtype=torch.float64) * 2 - 1
    q1 = torch.rand(n, device="cuda", dtype=torch.float64)
    xi = torch.rand(96, device="cuda", dtype=torch.float64).sort().values
    yi = (torch.rand(64, device="cuda", dtype=torch.float64) * 2 - 1).sort().values
    zq = torch.empty_like(xq); y1 = torch.empty_like(q1)
    for _ in range(2):                                            # first calls: allocations, function attributes
        p2.scattered(xq, yq, out=zq); p1(q1, out=y1); zi = p2.grid(xi, yi)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        p2.scattered(xq, yq, out=zq)
        p1(q1, out=y1)
        p1(q1, out=y1)                                            # back to back: the programmatic edge
        zi = p2.grid(xi, yi)
    for seed in (1, 2):
        gen = torch.Generator(device="cuda").manual_seed(seed)
        xq.copy_(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64))
        yq.copy_(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * 2 - 1)
        q1.copy_(torch.rand(n, generator=gen, device="cuda", dtype=torch.float64))
        if seed == 2:                                             # sorted by cell: the replay takes the other kernel
            o = ((xq * 699).floor() * 500 + ((yq + 1) / 2 * 499).floor()).argsort()
            xq.copy_(xq[o]); yq.copy_(yq[o])
        g.replay()
        torch.cuda.synchronize()
        assert same_bits(zq.cpu().numpy(), oracle.interp2_scattered(x, y, z, xq.cpu().numpy(), yq.cpu().numpy(), nthreads=8))
        assert same_bits(y1.cpu().numpy(), oracle.interp1(xg, yg, q1.cpu().numpy(), want_idx=False, nthreads=8))
        assert same_bits(zi.cpu().numpy(), oracle.interp2_grid(x, y, z, xi.cpu().numpy(), yi.cpu().numpy()))
