"""Derivatives of tensor-grid interp2: b200_interp2_grid_grad(_dev), b200_interp2_grid_adjoint(_dev), the C++
Interp2Plan::GridGrad / GridAdjoint and the Python grid_grad / grid_adjoint / grid_torch.

Every rule is the scattered rule applied to the mesh: output (i, j) is query k = j*nyi + i at (XI[j], YI[i]).  So the
GPU results are compared bit for bit (on integer views) with the CPU oracle of tests/interp2_grad_oracle.c run on the
mesh, and the grid adjoint with the scattered adjoint on the mesh.  A plain-Python restatement of the separable order
the grid adjoint's node kernel walks is checked against the oracle on the CPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_interp2_grad import GradOracle, ragged, same_as_oracle, same_ints, special_z, torch_same_ints, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="session")
def mesh_oracle(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("grid_grad_oracle") / "libgradoracle.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-std=c11", "-shared",
                           "-o", so, os.path.join(HERE, "interp2_grad_oracle.c"), "-lm"])
    return GradOracle(so)


def mesh(XI, YI):
    """The scattered queries of the grid XI x YI: k = j*nyi + i at (XI[j], YI[i])."""
    return np.repeat(XI, YI.size), np.tile(YI, XI.size)


def on_grid(a, nxi, nyi):
    """Mesh order -> (nyi, nxi), Fortran order."""
    return np.asfortranarray(a.reshape(nxi, nyi).T)


def oracle_grid_grad(goracle, x, y, z, XI, YI, extrap, y_first):
    xq, yq = mesh(XI, YI)
    return tuple(on_grid(a, XI.size, YI.size) for a in goracle.grad(x, y, z, xq, yq, extrap=extrap, y_first=y_first))


def oracle_grid_adjoint(goracle, x, y, XI, YI, g):
    """g (nyi, nxi) -> G (ny, nx) of the scattered oracle on the mesh."""
    xq, yq = mesh(XI, YI)
    return goracle.adjoint(x, y, xq, yq, np.asfortranarray(g).reshape(-1, order="F"))


def axis_queries(rng, knots, n, dt):
    """Unsorted entries with duplicates, every interior knot and the last, and out-of-range / NaN entries."""
    q = rng.uniform(knots[0] - 0.3, knots[-1] + 0.3, n).astype(dt)
    m = min(knots.size, n // 3)
    q[:m] = knots[rng.permutation(knots.size)[:m]]
    q[m:m + 6] = [knots[-1], knots[0], np.nan, knots[-1] + 1, knots[0] - 1, knots[1]]
    q[m + 6:m + 10] = q[m + 2:m + 6]                                  # duplicates
    q[-1] = knots[-1]
    return q


# ---- CPU: the separable order the grid adjoint implements ----

def separable_adjoint(x, y, XI, YI, g):
    """G = W^T g summed the way the node kernel walks it: a stable list of (entry, weight) per bracket and axis; node
    (i, j) starts at +0 and visits the cells (j-1, i-1), (j-1, i), (j, i-1), (j, i) as (cx, cy) in that (key) order, in
    each cell 'for j' in xlist(cx), for i' in ylist(cy)' (ascending mesh index j'*nyi + i'), and adds the terms of the
    roles whose corner it is, in role order 00, 10, 01, 11."""
    dt = g.dtype.type
    nx, ny = x.size, y.size

    def lists(knots, q):
        L = [[] for _ in range(knots.size)]
        for e, v in enumerate(q):
            if knots[0] <= v <= knots[-1]:
                a, _, w = weights(knots, v)
                L[a].append((e, w))
        return L

    LX, LY = lists(x, XI), lists(y, YI)
    G = np.zeros((ny, nx), g.dtype, order="F")
    with np.errstate(all="ignore"):
        for j in range(nx):
            for i in range(ny):
                acc = dt(0)
                for q in range(4):
                    cx, cy = j - 1 + (q >> 1), i - 1 + (q & 1)
                    if cx < 0 or cy < 0:
                        continue
                    bxc, byc = min(cx + 1, nx - 1), min(cy + 1, ny - 1)
                    mask = (cy == i and cx == j) | (byc == i and cx == j) << 1 | (cy == i and bxc == j) << 2 | \
                        (byc == i and bxc == j) << 3
                    for jj, wx in LX[cx]:
                        omx = dt(1) - wx
                        for ii, wy in LY[cy]:
                            omy = dt(1) - wy
                            gk = g[ii, jj]
                            if mask & 1:
                                acc = acc + (omx * omy) * gk
                            if mask & 2:
                                acc = acc + (omx * wy) * gk
                            if mask & 4:
                                acc = acc + (wx * omy) * gk
                            if mask & 8:
                                acc = acc + (wx * wy) * gk
                G[i, j] = acc
    return G


@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("affine", [False, True])
def test_separable_order_equals_the_scattered_oracle_on_the_mesh(mesh_oracle, dt, affine):
    rng = np.random.default_rng(7 + affine)
    if affine:
        x = np.linspace(-1.0, 2.0, 9).astype(dt); y = np.linspace(0.0, 5.0, 7).astype(dt)
    else:
        x = ragged(rng, 9, dt); y = ragged(rng, 7, dt)
    XI = axis_queries(rng, x, 41, dt)
    YI = axis_queries(rng, y, 33, dt)
    # the corner (nx-1, ny-1) and queries on the last knots of both axes
    XI[-2] = x[-1]; YI[-2] = y[-1]
    g = rng.standard_normal((YI.size, XI.size)).astype(dt)
    g[3, 5] = np.inf; g[4, 6] = -np.inf; g[7, 1] = -0.0; g[0, :] = 0.0
    want = oracle_grid_adjoint(mesh_oracle, x, y, XI, YI, g)
    assert same_as_oracle(separable_adjoint(x, y, XI, YI, g), want)
    # nodes with many terms: a 2 x 2 grid under a 30 x 30 query grid
    x2 = np.array([0.0, 1.0], dt); y2 = np.array([-1.0, 3.0], dt)
    XI2 = axis_queries(rng, x2, 30, dt); YI2 = axis_queries(rng, y2, 30, dt)
    g2 = rng.standard_normal((YI2.size, XI2.size)).astype(dt)
    assert same_as_oracle(separable_adjoint(x2, y2, XI2, YI2, g2), oracle_grid_adjoint(mesh_oracle, x2, y2, XI2, YI2, g2))


def test_new_entry_points_are_exported_and_reject_null_without_a_gpu(b200):
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    for name in ("b200_interp2_grid_grad", "b200_interp2_grid_grad_dev", "b200_interp2_grid_adjoint_workspace",
                 "b200_interp2_grid_adjoint_dev", "b200_interp2_grid_adjoint"):
        assert getattr(lib, name) is not None
    n = C.c_size_t(16)
    assert lib.b200_interp2_grid_grad(None, None, n, None, n, None, None, None, C.c_double(0.0)) == -1
    assert lib.b200_interp2_grid_grad_dev(None, None, n, None, n, None, None, None, C.c_double(0.0), None) == -1
    bytes_ = C.c_size_t()
    assert lib.b200_interp2_grid_adjoint_workspace(None, n, n, C.byref(bytes_)) == -1
    assert lib.b200_interp2_grid_adjoint_dev(None, None, n, None, n, None, n, 0, None, n, 0, None, n, None) == -1
    assert lib.b200_interp2_grid_adjoint(None, None, n, None, n, None, None) == -1
    assert b"NULL" in lib.b200_last_error()


# ---- GPU: gradient ----

def _p(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def grid_case(rng, nx, ny, dt, affine):
    if affine:
        return np.linspace(-1.0, 2.0, nx).astype(dt), np.linspace(0.0, 5.0, ny).astype(dt)
    return ragged(rng, nx, dt), np.unique(np.sort(rng.uniform(-3.0, 4.0, ny)).astype(dt))


def axis_specials(rng, knots, n, dt):
    q = axis_queries(rng, knots, n, dt)
    q[-3:] = [np.inf, -np.inf, knots[-1]]
    return q


@pytest.mark.gpu
@pytest.mark.parametrize("nyi", [64, 66, 67])            # V = 4, 2, 1
@pytest.mark.parametrize("shape,affine", [((3, 2), True), ((70, 50), False), ((20000, 7), False)])
@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_gradient_matches_oracle_on_the_mesh(b200, mesh_oracle, dt, y_first, shape, affine, nyi):
    """Both pass orders, axes staged in shared memory and (20000 knots) not, every V build; host and device buffers,
    and outputs misaligned by one element (the V = 1 build).  zi has the bits of grid()."""
    import torch
    nx, ny = shape
    rng = np.random.default_rng(nx + ny + nyi)
    P = b200.Interp2Plan
    x, y = grid_case(rng, nx, ny, dt, affine)
    z = special_z(rng.standard_normal((y.size, x.size)).astype(dt), rng)
    XI = axis_specials(rng, x, 301, dt)
    YI = axis_specials(rng, y, nyi, dt)
    plan = P(x, y, z, flags=P.ORDER_YX if y_first else 0)
    want = oracle_grid_grad(mesh_oracle, x, y, z, XI, YI, 1.25, y_first)
    host = plan.grid_grad(XI, YI, extrap=1.25)
    for got, ref in zip(host, want):
        assert got.flags.f_contiguous and same_as_oracle(got, ref)
    assert same_ints(host[0], plan.grid(XI, YI, extrap=1.25))
    tx, ty = torch.from_numpy(XI).cuda(), torch.from_numpy(YI).cuda()
    dev = plan.grid_grad(tx, ty, extrap=1.25)
    zv = plan.grid(tx, ty, extrap=1.25)
    torch.cuda.synchronize()
    for got, ref in zip(dev, host):
        assert got.shape == (YI.size, XI.size) and got.stride() == (1, YI.size)
        assert same_ints(np.asfortranarray(got.cpu().numpy()), ref)
    assert torch_same_ints(dev[0], zv)
    # outputs one element past an aligned start: the one-row-per-thread build
    n = XI.size * YI.size
    buf = torch.empty(3 * n + 3, dtype=tx.dtype, device="cuda")
    outs = [buf[1 + s * (n + 1):1 + s * (n + 1) + n] for s in range(3)]
    from armadillocudalinearinterpolation_b200 import _lib
    assert _lib.lib().b200_interp2_grid_grad_dev(plan._h, _p(tx), C.c_size_t(XI.size), _p(ty), C.c_size_t(YI.size),
                                                 *(_p(o) for o in outs), C.c_double(1.25), _stream()) == 0
    torch.cuda.synchronize()
    for got, ref in zip(outs, host):
        assert same_ints(got.cpu().numpy().reshape(XI.size, YI.size).T, ref)
    plan.close()


@pytest.mark.gpu
def test_gradient_across_two_launches_and_one_column_per_host_block(b200, mesh_oracle):
    """nxi > 65535*32 columns (two launches of the column-block loop) with a small nyi, and a host call whose slots
    hold one column of the three outputs each."""
    import torch
    rng = np.random.default_rng(5)
    x = ragged(rng, 40); y = np.linspace(0.0, 1.0, 9)
    z = rng.standard_normal((y.size, x.size))
    plan = b200.Interp2Plan(x, y, z)
    XI = np.sort(rng.uniform(x[0] - 0.1, x[-1] + 0.1, 65535 * 32 + 1000)); YI = axis_queries(rng, y, 16, np.float64)
    want = oracle_grid_grad(mesh_oracle, x, y, z, XI, YI, -1.0, False)
    dev = plan.grid_grad(torch.from_numpy(XI).cuda(), torch.from_numpy(YI).cuda(), extrap=-1.0)
    for got, ref in zip(dev, want):
        assert same_as_oracle(np.asfortranarray(got.cpu().numpy()), ref)
    XI2 = axis_queries(rng, x, 16, np.float64); YI2 = np.sort(rng.uniform(y[0] - 0.1, y[-1] + 0.1, (32 << 20) // 24 + 5))
    want = oracle_grid_grad(mesh_oracle, x, y, z, XI2, YI2, -1.0, False)
    for got, ref in zip(plan.grid_grad(XI2, YI2, extrap=-1.0), want):
        assert same_as_oracle(got, ref)
    plan.close()


# ---- GPU: adjoint ----

def adjoint_dev(lib, plan, tx, ty, g, ldg, g_row_major, G, ld, row_major, ws=None, ws_bytes=None):
    import torch
    need = C.c_size_t()
    assert lib.b200_interp2_grid_adjoint_workspace(plan._h, C.c_size_t(tx.numel()), C.c_size_t(ty.numel()),
                                                   C.byref(need)) == 0
    if ws is None:
        ws = torch.empty(max(need.value, 1), dtype=torch.uint8, device="cuda")
    return lib.b200_interp2_grid_adjoint_dev(plan._h, _p(tx), C.c_size_t(tx.numel()), _p(ty), C.c_size_t(ty.numel()),
                                             _p(g) if g is not None else None, C.c_size_t(ldg), g_row_major, _p(G),
                                             C.c_size_t(ld), row_major, _p(ws),
                                             C.c_size_t(need.value if ws_bytes is None else ws_bytes), _stream())


def g_in_layout(torch, g, row_major, pad):
    """g (nyi, nxi) stored column-major (row_major 0) or row-major with ld = minimum + pad: (storage, ld)."""
    nyi, nxi = g.shape
    if row_major:
        ld = nxi + pad
        buf = torch.full((nyi, ld), 5.5, dtype=g.dtype, device=g.device)
        buf[:, :nxi] = g
    else:
        ld = nyi + pad
        buf = torch.full((nxi, ld), 5.5, dtype=g.dtype, device=g.device)
        buf[:, :nyi] = g.t()
    return buf, ld


def G_from(buf, ld, row_major, nx, ny):
    b = buf.cpu().numpy()
    if row_major:
        M = b[:ny * ld].reshape(ny, ld)
        assert (M[:, nx:] == 7.5).all()
        return np.ascontiguousarray(M[:, :nx])
    M = b[:nx * ld].reshape(nx, ld)
    assert (M[:, ny:] == 7.5).all()
    return np.ascontiguousarray(M[:, :ny].T)


def check_against_scattered(b200, torch, plan, x, y, tx, ty, g):
    """grid_adjoint in all four (g layout, G layout) pairs with ld above its minimum equals scattered_adjoint on the
    mesh, GPU against GPU: the same bits, and NaN at the same nodes (a NaN's payload may come from either operand of an
    add)."""
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    nxi, nyi = tx.numel(), ty.numel()
    xq = tx.repeat_interleave(nyi); yq = ty.repeat(nxi)
    want = plan.scattered_adjoint(xq, yq, g.t().contiguous().reshape(-1)).cpu().numpy()
    del xq, yq
    for g_row_major in (0, 1):
        gs, ldg = g_in_layout(torch, g, g_row_major, 3)
        for row_major in (0, 1):
            ld = (x.size + 5) if row_major else (y.size + 3)
            G = torch.full(((x.size + y.size) * ld,), 7.5, dtype=g.dtype, device="cuda")
            assert adjoint_dev(lib, plan, tx, ty, gs, ldg, g_row_major, G, ld, row_major) == 0
            torch.cuda.synchronize()
            assert same_as_oracle(G_from(G, ld, row_major, x.size, y.size), want)
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_adjoint_matches_oracle_and_the_scattered_adjoint(b200, mesh_oracle, dt):
    import torch
    rng = np.random.default_rng(21)
    for (nx, ny), affine, (nxi, nyi) in (((3, 2), True, (50, 40)), ((70, 50), False, (301, 203)),
                                         ((257, 1001), True, (97, 1500)), ((2, 2), True, (1000, 1000))):
        x, y = grid_case(rng, nx, ny, dt, affine)
        z = rng.standard_normal((y.size, x.size)).astype(dt)
        XI = axis_specials(rng, x, nxi, dt); YI = axis_specials(rng, y, nyi, dt)
        g = rng.standard_normal((nyi, nxi)).astype(dt)
        g[:2, :6] = [[np.inf, -np.inf, np.nan, -0.0, 0.0, np.finfo(dt).smallest_subnormal], [1e30, -1e-30, 2, 3, 4, 5]]
        plan = b200.Interp2Plan(x, y, z)
        want = oracle_grid_adjoint(mesh_oracle, x, y, XI, YI, g)
        host = plan.grid_adjoint(XI, YI, g)
        assert host.flags.f_contiguous and same_as_oracle(host, want)
        tx, ty, tg = (torch.from_numpy(a).cuda() for a in (XI, YI, g))
        dZ = plan.grid_adjoint(tx, ty, tg)
        dZt = plan.grid_adjoint(tx, ty, tg.t().contiguous().t())
        torch.cuda.synchronize()
        assert dZ.is_contiguous() and same_ints(dZ.cpu().numpy(), np.ascontiguousarray(host))
        assert torch_same_ints(dZ, dZt)
        assert same_as_oracle(check_against_scattered(b200, torch, plan, x, y, tx, ty, tg), np.ascontiguousarray(host))
        plan.close()


@pytest.mark.gpu
def test_adjoint_edge_cases(b200):
    import torch
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    x = np.linspace(0, 1, 40); y = np.linspace(0, 1, 30)
    plan = b200.Interp2Plan(x, y, np.zeros((30, 40)))
    # every entry out of range (or NaN) on one axis: all +0
    tx = torch.tensor([-1.0, 2.0, float("nan"), 5.0], dtype=torch.float64, device="cuda")
    ty = torch.linspace(0, 1, 7, dtype=torch.float64, device="cuda")
    g = torch.randn(7, 4, dtype=torch.float64, device="cuda")
    dZ = plan.grid_adjoint(tx, ty, g)
    torch.cuda.synchronize()
    assert not bool(torch.signbit(dZ).any()) and bool((dZ == 0).all())
    # empty axes: an all-+0 G written over whatever was there
    e = torch.empty(0, dtype=torch.float64, device="cuda")
    for a, b in ((e, ty), (tx, e)):
        G = torch.full((30, 40), 3.0, dtype=torch.float64, device="cuda")
        assert adjoint_dev(lib, plan, a, b, torch.zeros(1, dtype=torch.float64, device="cuda"), 7, 0, G, 40, 1) == 0
        torch.cuda.synchronize()
        assert bool((G == 0).all()) and not bool(torch.signbit(G).any())
    assert (plan.grid_adjoint(np.zeros(0), np.zeros(5), np.zeros((5, 0))) == 0).all()
    zi = plan.grid_grad(tx, e)
    assert all(t.shape == (0, 4) for t in zi)
    # rejections before any device work: G stays untouched
    G = torch.full((30, 40), 3.0, dtype=torch.float64, device="cuda")
    need = C.c_size_t()
    assert lib.b200_interp2_grid_adjoint_workspace(plan._h, C.c_size_t(4), C.c_size_t(7), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    assert adjoint_dev(lib, plan, tx, ty, g, 7, 0, G, 30, 0, ws, need.value - 1) == -1
    assert b"workspace" in lib.b200_last_error()
    assert adjoint_dev(lib, plan, tx, ty, g, 6, 0, G, 30, 0) == -1 and b"ldg" in lib.b200_last_error()
    assert adjoint_dev(lib, plan, tx, ty, g, 3, 1, G, 30, 0) == -1
    assert adjoint_dev(lib, plan, tx, ty, g, 7, 0, G, 29, 0) == -1 and b"below" in lib.b200_last_error()
    assert adjoint_dev(lib, plan, tx, ty, g, 7, 0, G, 39, 1) == -1
    assert adjoint_dev(lib, plan, tx, ty, None, 7, 0, G, 30, 0) == -1 and b"NULL" in lib.b200_last_error()
    big = C.c_size_t(1 << 31)
    assert lib.b200_interp2_grid_adjoint_workspace(plan._h, big, C.c_size_t(4), C.byref(need)) == -6
    torch.cuda.synchronize()
    assert bool((G == 3.0).all())
    with pytest.raises(ValueError):
        plan.grid_adjoint(tx, ty, g.t())
    with pytest.raises(TypeError):
        plan.grid_adjoint(tx, ty, g.float())
    plan.close()


@pytest.mark.gpu
def test_benchmark_shape_adjoint_equals_scattered_deterministic_on_a_stream_and_in_a_graph(b200):
    """4096^2 f64 (the benchmark plan), 1e4 x 1e4 sorted outputs: grid_adjoint equals scattered_adjoint on the 1e8-query
    mesh in all four layout pairs; the same bits from a second call, another stream and graph replays of the captured
    _dev calls (capture succeeds: they allocate nothing)."""
    import torch
    import bench
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    x, y, z = bench.make_grid()
    plan = b200.Interp2Plan(x, y, z)
    gen = torch.Generator(device="cuda").manual_seed(3)
    tx = torch.sort(torch.rand(10_000, generator=gen, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0])[0]
    ty = torch.sort(torch.rand(10_000, generator=gen, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0])[0]
    g = torch.randn(10_000, 10_000, generator=gen, device="cuda", dtype=torch.float64)
    check_against_scattered(b200, torch, plan, x, y, tx, ty, g)
    a = plan.grid_adjoint(tx, ty, g)
    b = plan.grid_adjoint(tx, ty, g)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = plan.grid_adjoint(tx, ty, g)
    s.synchronize()
    torch.cuda.synchronize()
    assert torch_same_ints(a, b) and torch_same_ints(a, c)
    need = C.c_size_t()
    assert lib.b200_interp2_grid_adjoint_workspace(plan._h, C.c_size_t(10_000), C.c_size_t(10_000), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    G = torch.empty((y.size, x.size), dtype=torch.float64, device="cuda")
    ZI, DX, DY = (torch.empty((10_000, 10_000), dtype=torch.float64, device="cuda") for _ in range(3))

    def run():
        assert adjoint_dev(lib, plan, tx, ty, g, 10_000, 1, G, x.size, 1, ws) == 0
        assert lib.b200_interp2_grid_grad_dev(plan._h, _p(tx), C.c_size_t(10_000), _p(ty), C.c_size_t(10_000), _p(ZI),
                                              _p(DX), _p(DY), C.c_double(0.0), _stream()) == 0
    run()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    G.zero_(); ZI.zero_(); DX.zero_(); DY.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch_same_ints(G, a)
    zr, dxr, dyr = plan.grid_grad(tx, ty, extrap=0.0)
    torch.cuda.synchronize()
    # (ZI of the plan's call is column-major: the captured buffers hold its transpose's storage)
    assert torch_same_ints(ZI.view(-1), zr.t().contiguous().view(-1)) and torch_same_ints(DX.view(-1), dxr.t().contiguous().view(-1))
    assert torch_same_ints(DY.view(-1), dyr.t().contiguous().view(-1))
    assert torch_same_ints(zr, plan.grid(tx, ty, extrap=0.0))
    g.copy_(torch.randn(10_000, 10_000, device="cuda", dtype=torch.float64))
    graph.replay()
    torch.cuda.synchronize()
    assert torch_same_ints(G, plan.grid_adjoint(tx, ty, g))
    plan.close()


# ---- GPU: autograd ----

@pytest.mark.gpu
def test_autograd_gradcheck_and_bits(b200):
    import torch
    rng = np.random.default_rng(41)
    x = ragged(rng, 9); y = np.linspace(-1.0, 1.0, 7)
    z = rng.standard_normal((y.size, x.size))
    plan = b200.Interp2Plan(x, y, z)

    def mids(k, n):
        i = rng.integers(0, k.size - 1, n)
        return k[i] + (0.2 + 0.6 * rng.random(n)) * (k[i + 1] - k[i])

    XI = torch.from_numpy(mids(x, 6)).cuda().requires_grad_()
    YI = torch.from_numpy(mids(y, 5)).cuda().requires_grad_()
    Z = torch.from_numpy(z).cuda().requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b, c: plan.grid_torch(a, b, c), (XI, YI, Z), eps=1e-6, atol=1e-7)
    # backward bits equal the hand-built combination; a set_values between forward and backward changes nothing
    g = torch.randn(6, 5, dtype=torch.float64, device="cuda").t()   # (the layout of the output)
    XI.grad = YI.grad = Z.grad = None
    out = plan.grid_torch(XI, YI, Z)
    plan.set_values(np.zeros_like(z))
    out.backward(g)
    plan.set_values(z)
    zi, dx, dy = plan.grid_grad(XI.detach(), YI.detach())
    dZ = plan.grid_adjoint(XI.detach(), YI.detach(), g)
    torch.cuda.synchronize()
    assert torch_same_ints(out.detach(), zi)
    assert torch_same_ints(XI.grad, (g * dx).sum(0)) and torch_same_ints(YI.grad, (g * dy).sum(1))
    assert torch_same_ints(Z.grad, dZ)
    # axes that need no gradient: the value call serves the forward pass, and only Z gets a gradient
    Z.grad = None

    def no_grad_call(*a, **k):
        raise AssertionError("the gradient call ran")
    plan.grid_grad = no_grad_call
    out2 = plan.grid_torch(XI.detach(), YI.detach(), Z)
    out2.backward(g)
    del plan.grid_grad
    torch.cuda.synchronize()
    assert torch_same_ints(out2.detach(), zi) and torch_same_ints(Z.grad, dZ)
    plan.close()


# ---- C++ ----

@pytest.fixture(scope="module")
def host():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "host"), "-j4"],
                          stdout=subprocess.DEVNULL)
    lib = C.CDLL(os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "lib", "libb200host.so"))
    lib.b200_host_last_error.restype = C.c_char_p
    return lib


def _dp(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.gpu
def test_cpp_grid_grad_and_adjoint(b200, host):
    rng = np.random.default_rng(51)
    x = ragged(rng, 57); y = np.linspace(0.0, 2.0, 43)
    z = np.asfortranarray(special_z(rng.standard_normal((y.size, x.size)), rng))
    XI = axis_specials(rng, x, 120, np.float64); YI = axis_specials(rng, y, 90, np.float64)
    nx, ny, nxi, nyi = x.size, y.size, XI.size, YI.size
    plan = b200.Interp2Plan(x, y, z)
    outs = [np.empty((nyi, nxi), order="F") for _ in range(3)]
    rc = host.b200_host_interp2_grid_grad(_dp(x), nx, _dp(y), ny, _dp(z), _dp(XI), nxi, _dp(YI), nyi,
                                          *(_dp(o) for o in outs), C.c_double(-2.0))
    assert rc == 0, host.b200_host_last_error()
    for got, ref in zip(outs, plan.grid_grad(XI, YI, extrap=-2.0)):
        assert same_ints(got, ref)
    g = np.asfortranarray(rng.standard_normal((nyi, nxi)))
    dz = np.empty((ny, nx), order="F")
    rc = host.b200_host_interp2_grid_adjoint(_dp(x), nx, _dp(y), ny, _dp(z), _dp(XI), nxi, _dp(YI), nyi, _dp(g), nyi,
                                             nxi, _dp(dz))
    assert rc == 0, host.b200_host_last_error()
    assert same_ints(dz, plan.grid_adjoint(XI, YI, g))
    rc = host.b200_host_interp2_grid_adjoint(_dp(x), nx, _dp(y), ny, _dp(z), _dp(XI), nxi, _dp(YI), nyi, _dp(g), nxi,
                                             nyi, _dp(dz))
    assert rc == -1 and b"GridAdjoint: G must be YI.n_elem x XI.n_elem" in host.b200_host_last_error()
    plan.close()
