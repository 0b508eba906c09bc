"""Derivatives of scattered interp2: b200_interp2_scattered_grad(_dev), b200_interp2_scattered_adjoint(_dev), the C++
Interp2Plan::ScatteredGrad / ScatteredAdjoint and the Python scattered_grad / scattered_adjoint / scattered_torch.
GPU results are compared bit for bit (on integer views) with the CPU oracle of tests/interp2_grad_oracle.c, which
itself is checked here against central differences, the dense transpose W^T g and a plain-Python restatement of the
adjoint's summation order."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))


def ints(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def same_ints(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(ints(a), ints(b))


def same_as_oracle(a, ref):
    """Equal bits wherever the oracle is not NaN (-0.0 counts), NaN at the same places."""
    a, ref = np.ascontiguousarray(a), np.ascontiguousarray(ref)
    na, nr = np.isnan(a), np.isnan(ref)
    return a.shape == ref.shape and a.dtype == ref.dtype and np.array_equal(na, nr) and \
        np.array_equal(ints(a)[~na], ints(ref)[~nr])


def torch_same_ints(a, b):
    import torch
    it = torch.int64 if a.dtype == torch.float64 else torch.int32
    return a.shape == b.shape and torch.equal(a.view(it), b.view(it))


# ---- the oracle ----

class GradOracle:
    def __init__(self, so):
        self.lib = C.CDLL(so)

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(C.c_void_p)

    def grad(self, x, y, z, xq, yq, extrap=np.nan, y_first=False):
        dt = np.dtype(z.dtype)
        sfx, creal = ("f64", C.c_double) if dt == np.float64 else ("f32", C.c_float)
        self.lib.grad_oracle_set_order(int(bool(y_first)))
        x, y = np.ascontiguousarray(x, dt), np.ascontiguousarray(y, dt)
        xq, yq = np.ascontiguousarray(xq, dt), np.ascontiguousarray(yq, dt)
        zf = np.asfortranarray(z, dt)
        zq, dx, dy = (np.empty(xq.shape, dt) for _ in range(3))
        f = getattr(self.lib, "grad_oracle_scattered_" + sfx)
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                      C.c_void_p, C.c_void_p, C.c_void_p, creal]
        assert f(self._p(x), x.size, self._p(y), y.size, self._p(zf), self._p(xq), self._p(yq), xq.size, self._p(zq),
                 self._p(dx), self._p(dy), extrap) == 0
        return zq, dx, dy

    def adjoint(self, x, y, xq, yq, g):
        """G (ny, nx), Fortran order."""
        dt = np.dtype(g.dtype)
        sfx = "f64" if dt == np.float64 else "f32"
        x, y = np.ascontiguousarray(x, dt), np.ascontiguousarray(y, dt)
        xq, yq, g = (np.ascontiguousarray(a, dt) for a in (xq, yq, g))
        G = np.empty((y.size, x.size), dt, order="F")
        f = getattr(self.lib, "grad_oracle_adjoint_" + sfx)
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                      C.c_void_p]
        assert f(self._p(x), x.size, self._p(y), y.size, self._p(xq), self._p(yq), self._p(g), xq.size, self._p(G)) == 0
        return G


@pytest.fixture(scope="session")
def goracle(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("grad_oracle") / "libgradoracle.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-std=c11", "-shared",
                           "-o", so, os.path.join(HERE, "interp2_grad_oracle.c"), "-lm"])
    return GradOracle(so)


def weights(g, q):
    """(a, b, w) of in-range, non-NaN q on knots g: the bracket rule, in numpy."""
    a = min(np.searchsorted(g, q, side="right") - 1, g.size - 1)
    b = min(a + 1, g.size - 1)
    ae, be = abs(g[a] - q), abs(g[b] - q)
    w = ae / (ae + be) if ae > 0 else g.dtype.type(0)
    return a, b, w


def dense_W(x, y, xq, yq):
    """W (nq x ny*nx, column-major node index j*ny + i) of in-range queries, in float64."""
    W = np.zeros((xq.size, x.size * y.size))
    for k in range(xq.size):
        if not (x[0] <= xq[k] <= x[-1] and y[0] <= yq[k] <= y[-1]):
            continue
        ax, bx, wx = weights(x, xq[k])
        ay, by, wy = weights(y, yq[k])
        for (j, i, c) in ((ax, ay, (1 - wx) * (1 - wy)), (ax, by, (1 - wx) * wy), (bx, ay, wx * (1 - wy)), (bx, by, wx * wy)):
            W[k, j * y.size + i] += c
    return W


def ragged(rng, n, dt=np.float64):
    return np.unique(np.cumsum(0.3 + rng.random(n)).astype(dt))


# ---- CPU: the oracle against independent restatements ----

def test_oracle_gradient_matches_central_differences(goracle):
    from oracle import oracle_py
    rng = np.random.default_rng(1)
    x, y = ragged(rng, 23), ragged(rng, 17)
    z = rng.standard_normal((y.size, x.size))
    # queries well inside open cells: midpoints jittered by at most a quarter cell
    ix = rng.integers(0, x.size - 1, 2000); iy = rng.integers(0, y.size - 1, 2000)
    xq = x[ix] + (0.25 + 0.5 * rng.random(2000)) * (x[ix + 1] - x[ix])
    yq = y[iy] + (0.25 + 0.5 * rng.random(2000)) * (y[iy + 1] - y[iy])
    for y_first in (False, True):
        zq, dx, dy = goracle.grad(x, y, z, xq, yq, y_first=y_first)
        assert same_ints(zq, oracle_py.interp2_scattered(x, y, z, xq, yq, y_first=y_first))
        h = 1e-6
        fd_x = (oracle_py.interp2_scattered(x, y, z, xq + h, yq) - oracle_py.interp2_scattered(x, y, z, xq - h, yq)) / (2 * h)
        fd_y = (oracle_py.interp2_scattered(x, y, z, xq, yq + h) - oracle_py.interp2_scattered(x, y, z, xq, yq - h)) / (2 * h)
        scale = np.abs(z).max()
        assert np.allclose(dx, fd_x, rtol=1e-7, atol=1e-7 * scale)
        assert np.allclose(dy, fd_y, rtol=1e-7, atol=1e-7 * scale)


def test_oracle_gradient_one_sided_rules(goracle):
    x = np.array([0.0, 1.0, 3.0]); y = np.array([0.0, 2.0, 3.0])
    z = np.array([[0.0, 1.0, 5.0],    # row y = 0
                  [2.0, 4.0, 13.0],   # row y = 2
                  [3.0, 7.0, 30.0]])  # row y = 3
    # interior knot x = 1 at y = 0: the slope of the cell to the right, (5 - 1) / 2
    _, dx, dy = goracle.grad(x, y, z, np.array([1.0]), np.array([0.0]))
    assert dx[0] == 2.0 and dy[0] == (4.0 - 1.0) / 2.0
    # last knot x = 3 at y = 0: the slope of the last cell, from the left, (5 - 1) / 2; dz/dy on the last column
    _, dx, dy = goracle.grad(x, y, z, np.array([3.0]), np.array([0.0]))
    assert dx[0] == 2.0 and dy[0] == (13.0 - 5.0) / 2.0
    # last knots of both axes: (30 - 7) / 2 and (30 - 13) / 1
    zq, dx, dy = goracle.grad(x, y, z, np.array([3.0]), np.array([3.0]))
    assert zq[0] == 30.0 and dx[0] == 11.5 and dy[0] == 17.0
    # last y knot inside an x cell: dz/dx blends row 3 only ((1 - wy) = 1, wy = 0); dz/dy from the last y cell
    _, dx, dy = goracle.grad(x, y, z, np.array([0.5]), np.array([3.0]))
    assert dx[0] == (7.0 - 3.0) / 1.0 and dy[0] == 0.5 * (3.0 - 2.0) + 0.5 * (7.0 - 4.0)
    # outside -> +0 and extrap; NaN -> NaN
    zq, dx, dy = goracle.grad(x, y, z, np.array([-1.0, np.nan, 3.5, np.nan]), np.array([1.0, 1.0, np.nan, 9.0]), extrap=7.0)
    assert zq[0] == 7.0 and ints(dx[:1])[0] == 0 and ints(dy[:1])[0] == 0
    assert np.isnan(dx[1:]).all() and np.isnan(dy[1:]).all()


def _adjoint_reference(x, y, xq, yq, g):
    """The normative order restated in plain Python: a stable sort by cell key, then one addition per term."""
    dt = g.dtype.type
    nx, ny = x.size, y.size
    terms = []
    for k in range(xq.size):
        if not (x[0] <= xq[k] <= x[-1] and y[0] <= yq[k] <= y[-1]):
            continue
        ax, bx, wx = weights(x, xq[k])
        ay, by, wy = weights(y, yq[k])
        omx, omy = dt(1) - wx, dt(1) - wy
        cs = (omx * omy, omx * wy, wx * omy, wx * wy)
        nodes = ((ay, ax), (by, ax), (ay, bx), (by, bx))
        terms.append((ax * ny + ay, k, [(nodes[r], cs[r] * g[k]) for r in range(4)]))
    G = np.zeros((ny, nx), g.dtype, order="F")
    with np.errstate(all="ignore"):
        for _, _, ts in sorted(terms, key=lambda t: (t[0], t[1])):
            for (i, j), t in ts:
                G[i, j] = G[i, j] + t
    return G


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_oracle_adjoint_matches_dense_transpose_and_the_normative_order(goracle, dt):
    rng = np.random.default_rng(2)
    x, y = ragged(rng, 13, dt), ragged(rng, 9, dt)
    nq = 3000
    xq = rng.uniform(x[0] - 0.5, x[-1] + 0.5, nq).astype(dt); yq = rng.uniform(y[0] - 0.5, y[-1] + 0.5, nq).astype(dt)
    xq[:6] = [x[-1], x[-1], x[3], x[0], np.nan, x[2]]; yq[:6] = [y[-1], y[2], y[-1], y[0], y[1], np.nan]
    xq[100:400] = xq[99]; yq[100:400] = yq[99]                                   # many queries in one cell
    g = rng.standard_normal(nq).astype(dt)
    G = goracle.adjoint(x, y, xq, yq, g)
    W = dense_W(x.astype(np.float64), y.astype(np.float64), xq.astype(np.float64), yq.astype(np.float64))
    want = (W.T @ g.astype(np.float64)).reshape(x.size, y.size).T
    tol = 1e-12 if dt == np.float64 else 1e-4
    assert np.allclose(G, want, rtol=tol, atol=tol * np.abs(g).sum())
    assert same_ints(np.asfortranarray(G), _adjoint_reference(x, y, xq, yq, g))
    # special values in g propagate through every term: 0 * inf = NaN
    g2 = g.copy(); g2[7] = np.inf; g2[8] = -np.inf; g2[9] = np.nan; g2[10] = -0.0
    assert same_as_oracle(goracle.adjoint(x, y, xq, yq, g2), _adjoint_reference(x, y, xq, yq, g2))


def test_oracle_dot_product_identity(goracle):
    """<W^T g, V> = <g, W V>: the adjoint is the transpose of the scattered call."""
    from oracle import oracle_py
    rng = np.random.default_rng(3)
    x, y = ragged(rng, 31), ragged(rng, 19)
    nq = 5000
    xq = rng.uniform(x[0] - 0.2, x[-1] + 0.2, nq); yq = rng.uniform(y[0] - 0.2, y[-1] + 0.2, nq)
    g = rng.standard_normal(nq)
    V = rng.standard_normal((y.size, x.size))
    WV = oracle_py.interp2_scattered(x, y, V, xq, yq, extrap=0.0)
    lhs = np.sum(goracle.adjoint(x, y, xq, yq, g) * V)
    assert abs(lhs - np.dot(g, WV)) <= 1e-12 * np.sum(np.abs(g)) * np.abs(V).max()


def test_new_entry_points_reject_null_without_a_gpu(b200):
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    n = C.c_size_t(16)
    assert lib.b200_interp2_scattered_grad(None, None, None, n, None, None, None, C.c_double(0.0)) == -1
    assert lib.b200_interp2_scattered_grad_dev(None, None, None, n, None, None, None, C.c_double(0.0), None) == -1
    bytes_ = C.c_size_t()
    assert lib.b200_interp2_scattered_adjoint_workspace(None, n, C.byref(bytes_)) == -1
    assert lib.b200_interp2_scattered_adjoint_dev(None, None, None, None, n, None, n, 0, None, n, None) == -1
    assert lib.b200_interp2_scattered_adjoint(None, None, None, None, n, None) == -1
    assert b"NULL" in lib.b200_last_error()


# ---- GPU ----

LAYOUTS = ["NO_CELLS|NO_TILES", "FORCE_CELLS", "FORCE_TILES", "default", "FORCE_CELLS|FORCE_BANDS"]


def _flags(P, layout):
    f = 0
    for name in layout.split("|"):
        f |= 0 if name == "default" else getattr(P, name)
    return f


def special_z(z, rng):
    z = z.copy()
    tiny = np.finfo(z.dtype).smallest_subnormal
    flat = z.reshape(-1)
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, tiny, -3 * tiny, 7 * tiny], dtype=z.dtype)
    pos = rng.choice(flat.size, size=min(flat.size, 3 * specials.size), replace=False)
    flat[pos] = np.resize(specials, pos.size)
    z[-1, -1] = -0.0; z[-1, 0] = tiny; z[0, -1] = np.inf
    return z


def grid_case(rng, nx, ny, dt, affine):
    if affine:
        x = np.linspace(-1.0, 2.0, nx).astype(dt); y = np.linspace(0.0, 5.0, ny).astype(dt)
    else:
        x = ragged(rng, nx, dt); y = np.sort(rng.uniform(-3.0, 4.0, ny)).astype(dt)
        y = np.unique(y)
    return x, y


def queries(rng, x, y, nq, dt):
    xq = rng.uniform(x[0] - 0.3, x[-1] + 0.3, nq).astype(dt); yq = rng.uniform(y[0] - 0.3, y[-1] + 0.3, nq).astype(dt)
    xq[:8] = [x[0], x[-1], np.nan, x[1], x[-1], x[-1], np.nan, 1e30]; yq[:8] = [y[0], y[-1], y[1], np.nan, y[0], y[1], np.nan, y[1]]
    k = min(x.size, 3000)
    xq[20:20 + k] = x[:k]; yq[20:20 + k] = y[-1]                       # knots on the last row
    m = min(y.size, 3000)
    xq[4000:4000 + m] = x[-1]; yq[4000:4000 + m] = y[:m]                # ... and on the last column
    xq[8000:8000 + k] = x[:k]; yq[8000:8000 + k] = y[np.arange(k) % y.size]   # interior knots
    return xq, yq


@pytest.mark.gpu
@pytest.mark.parametrize("shape,affine", [((3, 2), True), ((70, 50), False), ((1001, 257), True), ((300, 301), False)])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_gradient_matches_oracle(b200, goracle, dt, y_first, layout, shape, affine):
    import torch
    nx, ny = shape
    rng = np.random.default_rng(nx * 7 + ny)
    P = b200.Interp2Plan
    x, y = grid_case(rng, nx, ny, dt, affine)
    z = special_z(rng.standard_normal((y.size, x.size)).astype(dt), rng)
    xq, yq = queries(rng, x, y, 20_003, dt)
    plan = P(x, y, z, flags=_flags(P, layout) | (P.ORDER_YX if y_first else 0))
    want = goracle.grad(x, y, z, xq, yq, extrap=1.25, y_first=y_first)
    host = plan.scattered_grad(xq, yq, extrap=1.25)
    for got, ref in zip(host, want):
        assert same_as_oracle(got, ref)
    assert same_ints(host[0], plan.scattered(xq, yq, extrap=1.25))
    tx, ty = torch.from_numpy(xq).cuda(), torch.from_numpy(yq).cuda()
    dev = plan.scattered_grad(tx, ty, extrap=1.25)
    zv = plan.scattered(tx, ty, extrap=1.25)
    torch.cuda.synchronize()
    for got, ref in zip(dev, host):
        assert same_ints(got.cpu().numpy(), ref)
    assert torch_same_ints(dev[0], zv)
    # unaligned device buffers: the one-query-per-thread path
    dev1 = plan.scattered_grad(tx[1:], ty[1:], extrap=1.25)
    torch.cuda.synchronize()
    for got, ref in zip(dev1, host):
        assert same_ints(got.cpu().numpy(), ref[1:])
    plan.close()


@pytest.mark.gpu
def test_gradient_axes_beyond_shared_memory_and_pageable_staging(b200, goracle):
    """Knot vectors too long to stage in shared memory (the global-memory search), and pageable host buffers above the
    staging threshold (the pinned ring with five arrays)."""
    rng = np.random.default_rng(11)
    x = ragged(rng, 20000); y = ragged(rng, 7)
    z = rng.standard_normal((y.size, x.size))
    xq, yq = queries(rng, x, y, (1 << 21) + 77, np.float64)
    plan = b200.Interp2Plan(x, y, z)
    got = plan.scattered_grad(xq, yq, extrap=-3.0)
    want = goracle.grad(x, y, z, xq, yq, extrap=-3.0)
    for g_, w_ in zip(got, want):
        assert same_as_oracle(g_, w_)
    x2 = np.linspace(0.0, 1.0, 300); y2 = np.linspace(0.0, 1.0, 200); z2 = rng.standard_normal((200, 300))
    xq2, yq2 = queries(rng, x2, y2, (1 << 21) + 5, np.float64)
    p2 = b200.Interp2Plan(x2, y2, z2)
    got = p2.scattered_grad(xq2, yq2)
    want = goracle.grad(x2, y2, z2, xq2, yq2)
    for g_, w_ in zip(got, want):
        assert same_as_oracle(g_, w_)


def _headline_queries(torch, x, y, nq, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = x.size
    xq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0]
    yq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0]
    cell = ((xq - x[0]) / (x[-1] - x[0]) * (n - 1)).floor() * n + ((yq - y[0]) / (y[-1] - y[0]) * (y.size - 1)).floor()
    o = cell.argsort()
    return (xq, yq), (xq[o].contiguous(), yq[o].contiguous())


@pytest.mark.gpu
def test_headline_gradient_values_equal_the_value_call(b200):
    """4096^2 f64, linspace axes, tiles: zq of the gradient call has the bits of b200_interp2_scattered_dev (which may
    be served by the straight-line kernel), for uniformly random and cell-sorted queries."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    plan = b200.Interp2Plan(x, y, z)
    for qx, qy in _headline_queries(torch, x, y, 1 << 22, 5):
        zq, dx, dy = plan.scattered_grad(qx, qy)
        zv = plan.scattered(qx, qy)
        torch.cuda.synchronize()
        assert torch_same_ints(zq, zv)
        assert bool(torch.isfinite(dx).all()) and bool(torch.isfinite(dy).all())
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["NO_CELLS|NO_TILES", "FORCE_CELLS", "FORCE_TILES"])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_adjoint_matches_oracle(b200, goracle, dt, layout):
    import torch
    rng = np.random.default_rng(21)
    P = b200.Interp2Plan
    for (nx, ny), affine in (((3, 2), True), ((70, 50), False), ((257, 1001), True)):
        x, y = grid_case(rng, nx, ny, dt, affine)
        z = rng.standard_normal((y.size, x.size)).astype(dt)
        xq, yq = queries(rng, x, y, 30_011, dt)
        xq[12000:16000] = xq[11999]; yq[12000:16000] = yq[11999]         # many queries in one cell
        g = rng.standard_normal(xq.size).astype(dt)
        g[:12] = [np.inf, -np.inf, np.nan, -0.0, 0.0, np.finfo(dt).smallest_subnormal, 1e30, -1e-30, 2, 3, 4, 5]
        plan = P(x, y, z, flags=_flags(P, layout))
        want = goracle.adjoint(x, y, xq, yq, g)
        got = plan.scattered_adjoint(xq, yq, g)
        assert got.flags.f_contiguous and same_as_oracle(np.asfortranarray(got), want)
        tx, ty, tg = (torch.from_numpy(a).cuda() for a in (xq, yq, g))
        dZ = plan.scattered_adjoint(tx, ty, tg)
        torch.cuda.synchronize()
        assert dZ.is_contiguous() and same_ints(dZ.cpu().numpy(), np.ascontiguousarray(got))
        # column- and row-major G with ld above its minimum, through the C-ABI; the padding stays untouched
        from armadillocudalinearinterpolation_b200 import _lib
        lib = _lib.lib()
        need = C.c_size_t()
        assert lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(xq.size), C.byref(need)) == 0
        ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for row_major, ld in ((0, y.size + 3), (1, x.size + 5)):
            buf = torch.full(((x.size + y.size) * ld,), 7.5, dtype=tg.dtype, device="cuda")
            assert lib.b200_interp2_scattered_adjoint_dev(plan._h, C.c_void_p(tx.data_ptr()), C.c_void_p(ty.data_ptr()),
                                                          C.c_void_p(tg.data_ptr()), C.c_size_t(xq.size),
                                                          C.c_void_p(buf.data_ptr()), C.c_size_t(ld), row_major,
                                                          C.c_void_p(ws.data_ptr()), C.c_size_t(need.value), stream) == 0
            torch.cuda.synchronize()
            b = buf.cpu().numpy()
            if row_major:
                M = b[:y.size * ld].reshape(y.size, ld)
                assert same_ints(np.ascontiguousarray(M[:, :x.size]), np.ascontiguousarray(got))
                assert (M[:, x.size:] == 7.5).all()
            else:
                M = b[:x.size * ld].reshape(x.size, ld)
                assert same_ints(np.ascontiguousarray(M[:, :y.size]), np.ascontiguousarray(got.T))
                assert (M[:, y.size:] == 7.5).all()
        plan.close()


@pytest.mark.gpu
def test_adjoint_rejections(b200):
    import torch
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    x = np.linspace(0, 1, 40); y = np.linspace(0, 1, 30)
    plan = b200.Interp2Plan(x, y, np.zeros((30, 40)))
    t = torch.zeros(100, dtype=torch.float64, device="cuda")
    G = torch.zeros(1200, dtype=torch.float64, device="cuda")
    need = C.c_size_t()
    assert lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(100), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = C.c_void_p(t.data_ptr())
    call = lambda ld, rm, wsb, nq=100: lib.b200_interp2_scattered_adjoint_dev(
        plan._h, p, p, p, C.c_size_t(nq), C.c_void_p(G.data_ptr()), C.c_size_t(ld), rm, C.c_void_p(ws.data_ptr()),
        C.c_size_t(wsb), s)
    assert call(30, 0, need.value - 1) == -1 and b"workspace" in lib.b200_last_error()
    assert call(29, 0, need.value) == -1 and b"below" in lib.b200_last_error()
    assert call(39, 1, need.value) == -1
    assert call(30, 0, need.value, nq=(1 << 31)) == -1
    assert lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(1 << 31), C.byref(need)) == -1
    assert call(30, 0, 1 << 40) == 0 and call(40, 1, 1 << 40) == 0
    torch.cuda.synchronize()
    with pytest.raises(TypeError):
        plan.scattered_grad(t, t.float())
    with pytest.raises(TypeError):
        plan.scattered_adjoint(t, t, t[::2])
    with pytest.raises(ValueError):
        plan.scattered_adjoint(t, t, t[:50])
    with pytest.raises(ValueError):
        plan.scattered_grad(np.zeros(3), np.zeros(4))


@pytest.mark.gpu
def test_headline_adjoint_matches_oracle_deterministic_on_a_stream_and_in_a_graph(b200, goracle):
    """4096^2 f64 tiles, 1e7 random queries: the oracle's bits, the same bits from a second call, from a non-default
    stream, and from replays of a captured CUDA graph."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    plan = b200.Interp2Plan(x, y, z)
    nq = 10_000_000
    (xq, yq), _ = _headline_queries(torch, x, y, nq, 31)
    g = torch.randn(nq, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(32))
    a = plan.scattered_adjoint(xq, yq, g)
    b = plan.scattered_adjoint(xq, yq, g)
    torch.cuda.synchronize()
    assert torch_same_ints(a, b)
    want = goracle.adjoint(x, y, xq.cpu().numpy(), yq.cpu().numpy(), g.cpu().numpy())
    assert same_as_oracle(a.cpu().numpy(), np.ascontiguousarray(want))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = plan.scattered_adjoint(xq, yq, g)
    s.synchronize()
    assert torch_same_ints(a, c)
    # graph capture and replay (workspace and output static)
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    need = C.c_size_t()
    assert lib.b200_interp2_scattered_adjoint_workspace(plan._h, C.c_size_t(nq), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    G = torch.empty((y.size, x.size), dtype=torch.float64, device="cuda")

    def run():
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        assert lib.b200_interp2_scattered_adjoint_dev(plan._h, C.c_void_p(xq.data_ptr()), C.c_void_p(yq.data_ptr()),
                                                      C.c_void_p(g.data_ptr()), C.c_size_t(nq), C.c_void_p(G.data_ptr()),
                                                      C.c_size_t(x.size), 1, C.c_void_p(ws.data_ptr()),
                                                      C.c_size_t(need.value), st) == 0
    run()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    G.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch_same_ints(G, a)
    g2 = torch.randn(nq, dtype=torch.float64, device="cuda")
    g.copy_(g2)
    graph.replay()
    torch.cuda.synchronize()
    assert torch_same_ints(G, plan.scattered_adjoint(xq, yq, g2))
    # the degenerate case: every query in one cell (correct, serial on four nodes)
    n1 = 200_000
    xs = torch.full((n1,), float(x[100] + 0.3 * (x[101] - x[100])), dtype=torch.float64, device="cuda")
    ys = torch.full((n1,), float(y[7] + 0.6 * (y[8] - y[7])), dtype=torch.float64, device="cuda")
    g1 = g[:n1].contiguous()
    d1 = plan.scattered_adjoint(xs, ys, g1).cpu().numpy()
    w1 = goracle.adjoint(x, y, xs.cpu().numpy(), ys.cpu().numpy(), g1.cpu().numpy())
    assert same_ints(d1, np.ascontiguousarray(w1))
    plan.close()


@pytest.mark.gpu
def test_autograd_gradcheck_and_bits(b200):
    import torch
    rng = np.random.default_rng(41)
    x = ragged(rng, 9); y = np.linspace(-1.0, 1.0, 7)
    z = rng.standard_normal((y.size, x.size))
    plan = b200.Interp2Plan(x, y, z)
    n = 64
    ix = rng.integers(0, x.size - 1, n); iy = rng.integers(0, y.size - 1, n)
    xq0 = x[ix] + (0.2 + 0.6 * rng.random(n)) * (x[ix + 1] - x[ix])
    yq0 = y[iy] + (0.2 + 0.6 * rng.random(n)) * (y[iy + 1] - y[iy])
    XQ = torch.from_numpy(xq0).cuda().requires_grad_()
    YQ = torch.from_numpy(yq0).cuda().requires_grad_()
    Z = torch.from_numpy(z).cuda().requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b, c: plan.scattered_torch(a, b, c), (XQ, YQ, Z), eps=1e-6, atol=1e-7)
    # backward bits equal the direct outputs; a set_values between forward and backward changes nothing
    g = torch.randn(n, dtype=torch.float64, device="cuda")
    out = plan.scattered_torch(XQ, YQ, Z)
    plan.set_values(np.zeros_like(z))
    out.backward(g)
    plan.set_values(z)
    zq, dx, dy = plan.scattered_grad(XQ.detach(), YQ.detach())
    dZ = plan.scattered_adjoint(XQ.detach(), YQ.detach(), g)
    torch.cuda.synchronize()
    assert torch_same_ints(out.detach(), zq)
    assert torch_same_ints(XQ.grad, g * dx) and torch_same_ints(YQ.grad, g * dy)
    assert torch_same_ints(Z.grad, dZ)
    # without Z and with queries that need no gradient: the value call, no gradient flows
    XQ.grad = None
    YQ.grad = None
    out2 = plan.scattered_torch(XQ.detach(), YQ)
    out2.sum().backward()
    torch.cuda.synchronize()
    assert XQ.grad is None and torch_same_ints(YQ.grad, dy)
    assert torch_same_ints(out2.detach(), zq)
    plan.close()


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
def test_cpp_scattered_grad_and_adjoint(b200, goracle, host):
    rng = np.random.default_rng(51)
    x = ragged(rng, 57); y = np.linspace(0.0, 2.0, 43)
    z = np.asfortranarray(special_z(rng.standard_normal((y.size, x.size)), rng))
    xq, yq = queries(rng, x, y, 30_000, np.float64)
    nx, ny, nq = x.size, y.size, xq.size
    zq, dx, dy = np.empty(nq), np.empty(nq), np.empty(nq)
    rc = host.b200_host_interp2_scattered_grad(_dp(x), nx, _dp(y), ny, _dp(z), _dp(xq), nq, _dp(yq), nq, _dp(zq), _dp(dx),
                                               _dp(dy), C.c_double(-2.0))
    assert rc == 0, host.b200_host_last_error()
    for got, ref in zip((zq, dx, dy), goracle.grad(x, y, z, xq, yq, extrap=-2.0)):
        assert same_as_oracle(got, ref)
    g = rng.standard_normal(nq)
    dz = np.empty((ny, nx), order="F")
    rc = host.b200_host_interp2_scattered_adjoint(_dp(x), nx, _dp(y), ny, _dp(z), _dp(xq), nq, _dp(yq), nq, _dp(g), nq,
                                                  _dp(dz))
    assert rc == 0, host.b200_host_last_error()
    assert same_ints(dz, goracle.adjoint(x, y, xq, yq, g))
    rc = host.b200_host_interp2_scattered_grad(_dp(x), nx, _dp(y), ny, _dp(z), _dp(xq), nq, _dp(yq), nq - 1, _dp(zq),
                                               _dp(dx), _dp(dy), C.c_double(-2.0))
    assert rc == -1 and b"ScatteredGrad: XQ and YQ" in host.b200_host_last_error()
    rc = host.b200_host_interp2_scattered_adjoint(_dp(x), nx, _dp(y), ny, _dp(z), _dp(xq), nq, _dp(yq), nq, _dp(g), nq - 1,
                                                  _dp(dz))
    assert rc == -1 and b"ScatteredAdjoint: XQ, YQ and G" in host.b200_host_last_error()
