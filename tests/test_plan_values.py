"""Plan values updated in place: b200_interp1_plan_set_values_dev, b200_interp2_plan_set_values(_dev), the C++
Interp2Plan::SetValues and the Python set_values methods.  After an update a plan must give, bit for bit, what a plan
created with the new values gives (and the oracle), whichever way the values arrive: host array, device column-major
or row-major, with or without a leading dimension beyond the minimum.  Bits are compared on integer views, so NaN
payloads and -0.0 count."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ints(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def same_ints(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(ints(a), ints(b))


def same_as_oracle(a, ref):
    """Equal bits wherever the oracle is not NaN (-0.0 counts), NaN at the same places (payloads may differ
    between the host and the device)."""
    a, ref = np.ascontiguousarray(a), np.ascontiguousarray(ref)
    na, nr = np.isnan(a), np.isnan(ref)
    return a.shape == ref.shape and np.array_equal(na, nr) and np.array_equal(ints(a)[~na], ints(ref)[~nr])


def torch_same_ints(a, b):
    import torch
    it = torch.int64 if a.dtype == torch.float64 else torch.int32
    return a.shape == b.shape and torch.equal(a.view(it), b.view(it))


def special_values(z, rng):
    """z with NaN, +-inf, -0.0 and subnormals, some of them on the last row / column (the clamped table entries)."""
    z = z.copy()
    ny, nx = z.shape
    tiny = np.finfo(z.dtype).smallest_subnormal
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, tiny, -3 * tiny, 7 * tiny], dtype=z.dtype)
    flat = z.reshape(-1)
    pos = rng.choice(flat.size, size=min(flat.size, 3 * specials.size), replace=False)
    flat[pos] = np.resize(specials, pos.size)
    z[-1, -1] = -0.0
    z[-1, 0] = tiny
    z[0, -1] = np.nan if nx * ny > 4 else z[0, -1]
    return z


# ---- CPU: argument checks come before any device work ----

def test_new_entry_points_reject_null_without_a_gpu(b200):
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    assert lib.b200_interp1_plan_set_values_dev(None, None, None) == -1
    assert lib.b200_interp2_plan_set_values(None, None) == -1
    assert lib.b200_interp2_plan_set_values_dev(None, None, C.c_size_t(16), 0, None) == -1
    assert lib.b200_interp2_plan_set_values_dev(None, None, C.c_size_t(16), 1, None) == -1
    assert b"NULL" in lib.b200_last_error()


# ---- GPU ----

def _dev_col(torch, z):
    t = torch.from_numpy(np.ascontiguousarray(z.T)).cuda().t()          # (ny, nx), strides (1, ny)
    assert t.stride() == (1, z.shape[0])
    return t


def _dev_col_ld(torch, z):
    ny, nx = z.shape
    big = np.full((ny + 5, nx + 2), np.nan, dtype=z.dtype)
    big[0, :] = 1e30; big[-1, :] = -1e30
    big[2:2 + ny, 1:1 + nx] = z
    t = torch.from_numpy(np.ascontiguousarray(big.T)).cuda().t()[2:2 + ny, 1:1 + nx]   # column block, ld = ny + 5
    assert t.stride() == (1, ny + 5)
    return t


def _dev_row(torch, z):
    t = torch.from_numpy(np.ascontiguousarray(z)).cuda()
    assert t.stride() == (z.shape[1], 1)
    return t


def _dev_row_ld(torch, z):
    ny, nx = z.shape
    big = np.full((ny + 3, nx + 7), -np.inf, dtype=z.dtype)
    big[1:1 + ny, 3:3 + nx] = z
    t = torch.from_numpy(big).cuda()[1:1 + ny, 3:3 + nx]                # row slice, ld = nx + 7
    assert t.stride() == (nx + 7, 1)
    return t


WAYS = {"host": None, "dev_col": _dev_col, "dev_col_ld": _dev_col_ld, "dev_row": _dev_row, "dev_row_ld": _dev_row_ld}


def _set(plan, z, way):
    import torch
    if WAYS[way] is None:
        plan.set_values(z)
    else:
        plan.set_values(WAYS[way](torch, z))
        torch.cuda.synchronize()


LAYOUTS = ["default", "FORCE_CELLS", "FORCE_TILES", "NO_CELLS|NO_TILES", "FORCE_CELLS|FORCE_BANDS"]


def _flags(P, layout):
    f = 0
    for name in layout.split("|"):
        f |= 0 if name == "default" else getattr(P, name)
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 2), (3, 7), (70, 50), (1001, 257)])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_interp2_set_values_equals_fresh_plan(b200, oracle, dt, y_first, layout, shape):
    import torch
    nx, ny = shape
    rng = np.random.default_rng(nx * 1000 + ny)
    P = b200.Interp2Plan
    flags = _flags(P, layout) | (P.ORDER_YX if y_first else 0)
    x = np.unique(np.cumsum(0.5 + rng.random(nx)).astype(dt))
    y = np.linspace(-2, 3, ny).astype(dt)
    assert x.size == nx
    z1 = rng.standard_normal((ny, nx)).astype(dt)
    z2 = special_values(rng.standard_normal((ny, nx)).astype(dt), rng)
    nq = 20_003
    xq = rng.uniform(x[0] - 0.5, x[-1] + 0.5, nq).astype(dt); yq = rng.uniform(-2.1, 3.1, nq).astype(dt)
    xq[:5] = [x[0], x[-1], np.nan, x[1], x[-1]]; yq[:5] = [y[0], y[-1], 0.0, np.nan, y[0]]
    k = min(nx, 4000)
    xq[10:10 + k] = x[:k]; yq[10:10 + k] = y[-1]                     # knots on the last row
    xq[5000:5000 + min(ny, 4000)] = x[-1]; yq[5000:5000 + min(ny, 4000)] = y[:4000]   # ... and the last column
    xi = np.sort(rng.uniform(x[0] - 0.2, x[-1] + 0.2, 61)).astype(dt)
    yi = np.sort(rng.uniform(-2.1, 3.1, 47)).astype(dt)
    tx, ty = torch.from_numpy(xq).cuda(), torch.from_numpy(yq).cuda()

    fresh = P(x, y, z2, flags=flags)
    want_s = fresh.scattered(xq, yq, extrap=1.25)
    want_d = fresh.scattered(tx, ty, extrap=1.25)
    torch.cuda.synchronize()
    want_d = want_d.cpu().numpy()
    want_g = fresh.grid(xi, yi, extrap=-0.5)
    fresh.close()
    assert same_ints(want_d, want_s)
    assert same_as_oracle(want_s, oracle.interp2_scattered(x, y, z2, xq, yq, extrap=1.25, nthreads=8, y_first=y_first))
    assert same_as_oracle(want_g, oracle.interp2_grid(x, y, z2, xi, yi, extrap=-0.5, y_first=y_first))

    plan = P(x, y, z1, flags=flags)
    before = plan.scattered(xq, yq, extrap=1.25)
    for way in WAYS:
        _set(plan, z2, way)
        assert same_ints(plan.scattered(xq, yq, extrap=1.25), want_s), way
        got_d = plan.scattered(tx, ty, extrap=1.25)                      # the banded pipeline serves device buffers
        torch.cuda.synchronize()
        assert same_ints(got_d.cpu().numpy(), want_d), way
        assert same_ints(plan.grid(xi, yi, extrap=-0.5), want_g), way
        plan.set_values(z1)                                              # back to Z1 before the next way
        assert same_ints(plan.scattered(xq, yq, extrap=1.25), before), way
    plan.close()


@pytest.mark.gpu
def test_headline_plan_row_major_update_equals_fresh_plan(b200):
    """The headline shape: 4096^2 f64, linspace axes, tiles.  Uniformly random and cell-sorted batches of 2^20 device
    queries (the device-side locality probe sends them to the generic and to the straight-line kernel) after a
    row-major set_values from a torch tensor."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    n = x.size
    z2 = np.random.default_rng(91).standard_normal((y.size, x.size))
    plan = b200.Interp2Plan(x, y, z)
    plan.set_values(torch.from_numpy(z2).cuda())
    fresh = b200.Interp2Plan(x, y, z2)
    g = torch.Generator(device="cuda").manual_seed(92)
    nq = 1 << 20
    xq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64) * (x[-1] - x[0]) + x[0]
    yq = torch.rand(nq, generator=g, device="cuda", dtype=torch.float64) * (y[-1] - y[0]) + y[0]
    cell = ((xq - x[0]) / (x[-1] - x[0]) * (n - 1)).floor() * n + ((yq - y[0]) / (y[-1] - y[0]) * (y.size - 1)).floor()
    o = cell.argsort()
    for qx, qy in ((xq, yq), (xq[o].contiguous(), yq[o].contiguous())):
        a = plan.scattered(qx, qy)
        b = fresh.scattered(qx, qy)
        torch.cuda.synchronize()
        assert torch_same_ints(a, b)
    plan.close(); fresh.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float64, np.float32])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_interp1_set_values_dev_equals_fresh_plan(b200, oracle, dt, mode):
    import torch
    rng = np.random.default_rng(100 + mode)
    if mode == 0:
        xg = np.arange(50001, dtype=np.float64) / 262144.0              # exactly uniform: index arithmetic
    elif mode == 1:
        xg = np.cumsum(0.5 + rng.random(50001))                         # bucket table
    else:
        xg = np.cumsum(0.5 + rng.random(1000))                          # staged in shared memory
    xg = np.unique(xg.astype(dt))
    y1 = rng.standard_normal(xg.size).astype(dt)
    y2 = special_values(rng.standard_normal(xg.size).astype(dt).reshape(1, -1), rng).reshape(-1)
    xi = rng.uniform(xg[0] - 1, xg[-1] + 1, 1_000_003).astype(dt)
    xi[:4] = [xg[0], xg[-1], np.nan, xg[17]]
    xi[100:100 + min(xg.size, 5000)] = xg[:5000]
    plan = b200.Interp1Plan(xg, y1)
    assert plan.lookup_mode == mode
    plan.set_values(torch.from_numpy(y2).cuda())
    torch.cuda.synchronize()
    fresh = b200.Interp1Plan(xg, y2)
    yi, idx = plan(xi, extrap=0.75, return_index=True)
    yf, idf = fresh(xi, extrap=0.75, return_index=True)
    assert same_ints(yi, yf) and np.array_equal(idx, idf)
    yo, io = oracle.interp1(xg, y2, xi, extrap=0.75, nthreads=8)
    assert same_as_oracle(yi, yo) and np.array_equal(idx, io)
    td = torch.from_numpy(xi).cuda()                                    # device queries too
    yd, idd = plan(td, extrap=0.75, return_index=True)
    torch.cuda.synchronize()
    assert same_ints(yd.cpu().numpy(), yf) and np.array_equal(idd.cpu().numpy(), idf)
    plan.set_values(y1)                                                 # the host path still works after it
    assert same_ints(plan(xi, extrap=0.75), b200.Interp1Plan(xg, y1)(xi, extrap=0.75))


@pytest.mark.gpu
def test_updates_are_ordered_on_the_callers_stream(b200):
    """scattered(Z1), set_values(Z2), scattered, set_values(Z3 row-major), scattered — queued on a non-default stream
    with no synchronisation in between; each batch sees exactly the values set before it.  Same for interp1."""
    import torch
    rng = np.random.default_rng(7)
    nx, ny = 1024, 768
    x = np.linspace(0.0, 1.0, nx); y = np.linspace(-1.0, 1.0, ny)
    zs = [rng.standard_normal((ny, nx)) for _ in range(3)]
    xg = np.sort(rng.random(5000)); ys = [rng.standard_normal(5000) for _ in range(3)]
    nq = 1 << 24
    xq = torch.rand(nq, device="cuda", dtype=torch.float64); yq = torch.rand(nq, device="cuda", dtype=torch.float64) * 2 - 1
    z2 = _dev_col(torch, zs[1]); z3 = _dev_row(torch, zs[2])
    y2 = torch.from_numpy(ys[1]).cuda(); y3 = torch.from_numpy(ys[2]).cuda()
    p2 = b200.Interp2Plan(x, y, zs[0]); p1 = b200.Interp1Plan(xg, ys[0])
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        o = [p2.scattered(xq, yq)]
        p2.set_values(z2); o.append(p2.scattered(xq, yq))
        p2.set_values(z3); o.append(p2.scattered(xq, yq))
        o1 = [p1(xq)]
        p1.set_values(y2); o1.append(p1(xq))
        p1.set_values(y3); o1.append(p1(xq))
    s.synchronize()
    for k in range(3):
        fresh = b200.Interp2Plan(x, y, zs[k])
        assert torch_same_ints(o[k], fresh.scattered(xq, yq)), k
        assert torch_same_ints(o1[k], b200.Interp1Plan(xg, ys[k])(xq)), k
        torch.cuda.synchronize()


@pytest.mark.gpu
def test_set_values_dev_captures_into_a_cuda_graph(b200):
    """set_values from a static tensor followed by scattered queries, captured with torch.cuda.graph (default capture
    mode) and replayed with two different contents of the static tensor: each replay equals its fresh plan."""
    import torch
    rng = np.random.default_rng(8)
    nx, ny = 700, 500
    x = np.linspace(0.0, 1.0, nx); y = np.linspace(-1.0, 1.0, ny)
    zs = [rng.standard_normal((ny, nx)) for _ in range(3)]
    xg = np.sort(rng.random(3000)); ys = [rng.standard_normal(3000) for _ in range(3)]
    n = 1 << 21
    xq = torch.rand(n, device="cuda", dtype=torch.float64); yq = torch.rand(n, device="cuda", dtype=torch.float64) * 2 - 1
    p2 = b200.Interp2Plan(x, y, zs[0], flags=b200.Interp2Plan.FORCE_TILES); p1 = b200.Interp1Plan(xg, ys[0])
    z_static = torch.from_numpy(zs[0]).cuda(); y_static = torch.from_numpy(ys[0]).cuda()
    zq = torch.empty_like(xq); y1 = torch.empty_like(xq)
    for _ in range(2):                                                 # first calls: function attributes
        p2.set_values(z_static); p2.scattered(xq, yq, out=zq)
        p1.set_values(y_static); p1(xq, out=y1)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        p2.set_values(z_static)
        p2.scattered(xq, yq, out=zq)
        p1.set_values(y_static)
        p1(xq, out=y1)
    for k in (1, 2):
        z_static.copy_(torch.from_numpy(zs[k]))
        y_static.copy_(torch.from_numpy(ys[k]))
        g.replay()
        torch.cuda.synchronize()
        want = b200.Interp2Plan(x, y, zs[k], flags=b200.Interp2Plan.FORCE_TILES).scattered(xq, yq)
        want1 = b200.Interp1Plan(xg, ys[k])(xq)
        torch.cuda.synchronize()
        assert torch_same_ints(zq, want), k
        assert torch_same_ints(y1, want1), k


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
def test_cpp_interp2_plan_set_values(b200, oracle, host):
    rng = np.random.default_rng(9)
    nx, ny, nq = 57, 43, 30_000
    x = np.cumsum(0.5 + rng.random(nx)); y = np.linspace(0.0, 2.0, ny)
    z1 = np.asfortranarray(rng.standard_normal((ny, nx)))
    z2 = np.asfortranarray(special_values(rng.standard_normal((ny, nx)), rng))
    xq = rng.uniform(x[0] - 1, x[-1] + 1, nq); yq = rng.uniform(-0.1, 2.1, nq)
    got = np.empty(nq); want = np.empty(nq)
    rc = host.b200_host_interp2_set_values(_dp(x), nx, _dp(y), ny, _dp(z1), _dp(z2), ny, nx, _dp(xq), _dp(yq), nq,
                                           _dp(got), C.c_double(-2.0))
    assert rc == 0, host.b200_host_last_error()
    rc = host.b200_host_interp2(_dp(x), nx, _dp(y), ny, _dp(z2), _dp(xq), nq, _dp(yq), nq, _dp(want), C.c_double(-2.0), 2)
    assert rc == 0, host.b200_host_last_error()
    assert same_ints(got, want)
    assert same_as_oracle(got, oracle.interp2_scattered(x, y, z2, xq, yq, extrap=-2.0))
    # a wrongly shaped arma::mat is rejected with the constructor's message
    bad = np.zeros((ny + 1) * nx)
    rc = host.b200_host_interp2_set_values(_dp(x), nx, _dp(y), ny, _dp(z1), _dp(bad), ny + 1, nx, _dp(xq), _dp(yq), nq,
                                           _dp(got), C.c_double(-2.0))
    assert rc == -1
    assert host.b200_host_last_error() == \
        b"b200::Interp2Plan: X.n_elem must equal Z.n_cols and Y.n_elem must equal Z.n_rows"


@pytest.mark.gpu
def test_python_rejections_leave_the_plan_unchanged(b200):
    import torch
    from armadillocudalinearinterpolation_b200 import _lib
    rng = np.random.default_rng(10)
    nx, ny = 40, 30
    x = np.linspace(0, 1, nx); y = np.linspace(0, 1, ny); z = rng.standard_normal((ny, nx))
    xq = rng.random(1000); yq = rng.random(1000)
    plan = b200.Interp2Plan(x, y, z)
    before = plan.scattered(xq, yq)
    with pytest.raises(ValueError):
        plan.set_values(np.zeros((nx, ny)))
    with pytest.raises(ValueError):
        plan.set_values(torch.zeros((ny, nx + 1), dtype=torch.float64, device="cuda"))
    with pytest.raises(TypeError):
        plan.set_values(torch.zeros((ny, nx), dtype=torch.float32, device="cuda"))
    with pytest.raises(TypeError):
        plan.set_values(np.zeros((ny, nx), dtype=np.complex128))
    # ld below its minimum, straight through the C-ABI: rejected before any device work
    t = torch.zeros((ny, nx), dtype=torch.float64, device="cuda")
    lib = _lib.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.b200_interp2_plan_set_values_dev(plan._h, C.c_void_p(t.data_ptr()), C.c_size_t(ny - 1), 0, stream) == -1
    assert lib.b200_interp2_plan_set_values_dev(plan._h, C.c_void_p(t.data_ptr()), C.c_size_t(nx - 1), 1, stream) == -1
    assert b"below" in lib.b200_last_error()
    assert lib.b200_interp2_plan_set_values_dev(plan._h, None, C.c_size_t(ny), 0, stream) == -1
    assert lib.b200_interp2_plan_set_values(plan._h, None) == -1
    torch.cuda.synchronize()
    assert same_ints(plan.scattered(xq, yq), before)
    # interp1
    p1 = b200.Interp1Plan(x, z[0])
    b1 = p1(xq)
    with pytest.raises(ValueError):
        p1.set_values(np.zeros(nx + 1))
    with pytest.raises(ValueError):
        p1.set_values(torch.zeros(nx - 1, dtype=torch.float64, device="cuda"))
    with pytest.raises(TypeError):
        p1.set_values(torch.zeros(nx, dtype=torch.float32, device="cuda"))
    with pytest.raises(TypeError):
        p1.set_values(torch.zeros(2 * nx, dtype=torch.float64, device="cuda")[::2])
    assert lib.b200_interp1_plan_set_values_dev(p1._h, None, stream) == -1
    assert same_ints(p1(xq), b1)
