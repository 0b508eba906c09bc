"""Derivatives of interp1: b200_interp1_grad(_dev), b200_interp1_adjoint(_dev), the C++ Interp1Plan::Grad / Adjoint and
the Python grad / adjoint / interp_torch.  GPU results are compared bit for bit (on integer views) with the CPU oracle of
tests/interp1_grad_oracle.c, which itself is checked here against central differences, the dense transpose W^T g and a
plain-Python restatement of the adjoint's blocked sum."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
B = 256   # B200_INTERP1_ADJOINT_BLOCK (checked against the header by test_oracle_block_is_the_header_constant)


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

class Grad1Oracle:
    def __init__(self, so):
        self.lib = C.CDLL(so)
        self.lib.grad1_oracle_block.restype = C.c_size_t

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(C.c_void_p)

    def grad(self, x, y, xi, extrap=np.nan):
        dt = np.dtype(y.dtype)
        sfx, creal = ("f64", C.c_double) if dt == np.float64 else ("f32", C.c_float)
        x, y, xi = (np.ascontiguousarray(a, dt) for a in (x, y, xi))
        yi, dy = np.empty(xi.shape, dt), np.empty(xi.shape, dt)
        f = getattr(self.lib, "grad1_oracle_" + sfx)
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, creal]
        assert f(self._p(x), self._p(y), x.size, self._p(xi), xi.size, self._p(yi), self._p(dy), extrap) == 0
        return yi, dy

    def adjoint(self, x, xi, g):
        dt = np.dtype(g.dtype)
        sfx = "f64" if dt == np.float64 else "f32"
        x, xi, g = (np.ascontiguousarray(a, dt) for a in (x, xi, g))
        G = np.empty(x.size, dt)
        f = getattr(self.lib, "adj1_oracle_" + sfx)
        f.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        assert f(self._p(x), x.size, self._p(xi), self._p(g), xi.size, self._p(G)) == 0
        return G


@pytest.fixture(scope="session")
def g1oracle(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("grad1_oracle") / "libgrad1oracle.so")
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wno-unknown-pragmas",
                           "-std=c11", "-shared", "-o", so, os.path.join(HERE, "interp1_grad_oracle.c"), "-lm"])
    return Grad1Oracle(so)


def ragged(rng, n, dt=np.float64):
    return np.unique(np.cumsum(0.3 + rng.random(n)).astype(dt))


def weight(x, q):
    """(a, b, w) of in-range, non-NaN q: the bracket rule, in numpy."""
    a = min(np.searchsorted(x, q, side="right") - 1, x.size - 1)
    b = min(a + 1, x.size - 1)
    ae, be = abs(x[a] - q), abs(x[b] - q)
    w = ae / (ae + be) if ae > 0 else x.dtype.type(0)
    return a, b, w


def dense_W(x, xi):
    W = np.zeros((xi.size, x.size))
    for k in range(xi.size):
        if not (x[0] <= xi[k] <= x[-1]):
            continue
        a, b, w = weight(x, xi[k])
        W[k, a] += 1 - w
        W[k, b] += w
    return W


def blocked_sum(t, dt):
    """R of include/b200_interp.h in plain Python."""
    if len(t) <= B:
        acc = dt(0)
        for v in t:
            acc = dt(acc + v)
        return acc
    return blocked_sum([blocked_sum(t[i:i + B], dt) for i in range(0, len(t), B)], dt)


def adjoint_reference(x, xi, g):
    """The normative order restated: terms in ascending (segment, query index, role) order per node, then R."""
    dt = g.dtype.type
    lists = [[] for _ in range(x.size)]
    with np.errstate(all="ignore"):
        for k in sorted((k for k in range(xi.size) if x[0] <= xi[k] <= x[-1]), key=lambda k: (weight(x, xi[k])[0], k)):
            a, b, w = weight(x, xi[k])
            lists[a].append(dt(dt(1) - w) * g[k])
            lists[b].append(w * g[k])
        return np.array([blocked_sum(l, dt) for l in lists], dtype=g.dtype)


# ---- CPU: the oracle against independent restatements ----

def test_oracle_block_is_the_header_constant(g1oracle):
    assert g1oracle.lib.grad1_oracle_block() == B


def test_oracle_slopes_match_central_differences(g1oracle):
    from oracle import oracle_py
    rng = np.random.default_rng(1)
    x = ragged(rng, 41)
    y = rng.standard_normal(x.size)
    i = rng.integers(0, x.size - 1, 3000)
    xi = x[i] + (0.25 + 0.5 * rng.random(i.size)) * (x[i + 1] - x[i])
    yi, dy = g1oracle.grad(x, y, xi)
    assert same_ints(yi, oracle_py.interp1(x, y, xi)[0])
    h = 1e-6
    fd = (oracle_py.interp1(x, y, xi + h)[0] - oracle_py.interp1(x, y, xi - h)[0]) / (2 * h)
    assert np.allclose(dy, fd, rtol=1e-7, atol=1e-7 * np.abs(y).max())


def test_oracle_one_sided_rules(g1oracle):
    x = np.array([0.0, 1.0, 3.0, 4.0])
    y = np.array([2.0, 3.0, 9.0, 5.0])
    xi = np.array([0.0, 1.0, 3.0, 4.0, 0.5, -np.inf, np.inf, -1.0, 5.0, np.nan])
    yi, dy = g1oracle.grad(x, y, xi, extrap=7.0)
    assert dy[0] == 1.0                 # first knot: the segment to the right
    assert dy[1] == 3.0                 # interior knot: the segment to the right, (9 - 3) / 2
    assert dy[2] == -4.0                # interior knot 3: (5 - 9) / 1
    assert dy[3] == -4.0                # last knot: the last segment, from the left
    assert dy[4] == 1.0
    assert (ints(dy[5:9]) == 0).all() and (yi[5:9] == 7.0).all()   # out of range, +-inf included: +0
    assert np.isnan(dy[9]) and np.isnan(yi[9])


@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_oracle_adjoint_matches_dense_transpose_and_the_blocked_sum(g1oracle, dt):
    rng = np.random.default_rng(2)
    x = ragged(rng, 17, dt)
    ni = 4000
    xi = rng.uniform(x[0] - 0.5, x[-1] + 0.5, ni).astype(dt)
    xi[:5] = [x[-1], x[0], x[3], np.nan, x[-1]]
    xi[100:1100] = xi[99]                                   # 1000 queries in one segment: two levels of R
    g = rng.standard_normal(ni).astype(dt)
    G = g1oracle.adjoint(x, xi, g)
    want = dense_W(x.astype(np.float64), xi.astype(np.float64)).T @ g.astype(np.float64)
    tol = 1e-12 if dt == np.float64 else 1e-4
    assert np.allclose(G, want, rtol=tol, atol=tol * np.abs(g).sum())
    assert same_ints(G, adjoint_reference(x, xi, g))
    g2 = g.copy(); g2[7] = np.inf; g2[8] = -np.inf; g2[9] = np.nan; g2[10] = -0.0
    assert same_as_oracle(g1oracle.adjoint(x, xi, g2), adjoint_reference(x, xi, g2))


def test_oracle_adjoint_three_levels(g1oracle):
    """70 000 queries in one segment: more than B^2 terms on each of its nodes, so R has three levels."""
    rng = np.random.default_rng(3)
    x = np.linspace(0.0, 1.0, 11)
    xi = rng.uniform(x[4], x[5], 70_000)
    g = rng.standard_normal(xi.size) * 1e3
    G = g1oracle.adjoint(x, xi, g)
    assert same_ints(G, adjoint_reference(x, xi, g))
    # and not the one-at-a-time sum on those nodes (the blocked sum is a different order)
    a, b, w = zip(*(weight(x, q) for q in xi))
    seq = np.float64(0)
    for wk, gk in zip(w, g):
        seq = seq + (1 - wk) * gk
    assert np.isclose(G[4], seq, rtol=1e-12)


def test_oracle_dot_product_identity(g1oracle):
    from oracle import oracle_py
    rng = np.random.default_rng(4)
    x = ragged(rng, 53)
    xi = rng.uniform(x[0] - 0.3, x[-1] + 0.3, 6000)
    g = rng.standard_normal(xi.size)
    v = rng.standard_normal(x.size)
    Wv = oracle_py.interp1(x, v, xi, extrap=0.0)[0]
    lhs = np.dot(g1oracle.adjoint(x, xi, g), v)
    assert abs(lhs - np.dot(g, Wv)) <= 1e-12 * np.sum(np.abs(g)) * np.abs(v).max()


def test_new_entry_points_reject_null_without_a_gpu(b200):
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    n = C.c_size_t(16)
    assert lib.b200_interp1_grad(None, None, n, None, None, C.c_double(0.0)) == -1
    assert lib.b200_interp1_grad_dev(None, None, n, None, None, C.c_double(0.0), None) == -1
    bytes_ = C.c_size_t()
    assert lib.b200_interp1_adjoint_workspace(None, n, C.byref(bytes_)) == -1
    assert lib.b200_interp1_adjoint_dev(None, None, None, n, None, None, n, None) == -1
    assert lib.b200_interp1_adjoint(None, None, None, n, None) == -1
    assert b"NULL" in lib.b200_last_error()


# ---- GPU ----

def knots(rng, kind, n, dt):
    if kind == "linspace":
        return np.linspace(-1.0, 2.0, n).astype(dt)
    if kind == "quasi":   # uniform-ish but not affine: lookup mode 0 through the stored knots
        x = np.linspace(-1.0, 2.0, n)
        x[1:-1] += (rng.random(n - 2) - 0.5) * 1e-3 * (x[1] - x[0])
        return x.astype(dt)
    return ragged(rng, n, dt)


def special_y(y, rng):
    y = y.copy()
    tiny = np.finfo(y.dtype).smallest_subnormal
    sp = np.array([np.nan, np.inf, -np.inf, -0.0, tiny, -3 * tiny], dtype=y.dtype)
    pos = rng.choice(y.size, size=min(y.size, sp.size), replace=False)
    y[pos] = sp[:pos.size]
    y[-1] = -0.0
    return y


def queries(rng, x, ni, dt):
    xi = rng.uniform(x[0] - 0.3 * (x[-1] - x[0]), x[-1] + 0.3 * (x[-1] - x[0]), ni).astype(dt)
    xi[:8] = [x[0], x[-1], np.nan, np.inf, -np.inf, x[-1], x[min(1, x.size - 1)], np.nan]
    k = min(x.size, 3000)
    xi[20:20 + k] = x[:k]                      # knots
    xi[4000:4000 + k] = x[-k:]
    return xi


# (knots, ng, lookup mode): grids that fit in shared memory take mode 2 whatever their knots
MODES = [("linspace", 2, 2), ("linspace", 3, 2), ("ragged", 257, 2), ("linspace", 6000, 2), ("ragged", 5000, 2),
         ("quasi", 20_000, 0), ("linspace", 1_000_000, 0), ("ragged", 1_000_000, 1)]


def check_mode(plan, mode, dt):
    """f32 knot vectors may round to another (quasi-)uniform classification: only the path family is fixed there"""
    if dt == np.float64 or mode == 2:
        assert plan.lookup_mode == mode
    else:
        assert plan.lookup_mode in (0, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,mode", MODES)
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_gradient_matches_oracle(b200, g1oracle, dt, kind, n, mode):
    import torch
    rng = np.random.default_rng(n + (7 if dt == np.float32 else 0))
    x = knots(rng, kind, n, dt)
    y = special_y(rng.standard_normal(x.size).astype(dt), rng)
    xi = queries(rng, x, 200_003, dt)
    plan = b200.Interp1Plan(x, y)
    check_mode(plan, mode, dt)
    want = g1oracle.grad(x, y, xi, extrap=1.25)
    host = plan.grad(xi, extrap=1.25)
    for got, ref in zip(host, want):
        assert same_as_oracle(got, ref)
    assert same_ints(host[0], plan(xi, extrap=1.25))
    t = torch.from_numpy(xi).cuda()
    yi, dy = plan.grad(t, extrap=1.25)
    yv = plan(t, extrap=1.25)
    torch.cuda.synchronize()
    assert same_ints(yi.cpu().numpy(), host[0]) and same_ints(dy.cpu().numpy(), host[1])
    assert torch_same_ints(yi, yv)
    yi1, dy1 = plan.grad(t[1:], extrap=1.25)     # unaligned: the scalar kernel
    torch.cuda.synchronize()
    assert same_ints(yi1.cpu().numpy(), host[0][1:]) and same_ints(dy1.cpu().numpy(), host[1][1:])
    plan.close()


@pytest.mark.gpu
def test_gradient_host_paths_pinned_and_pageable(b200, g1oracle):
    """>= 2^21 queries from pageable numpy memory (the pinned ring) and from pinned memory (the two-slot pipeline)."""
    import torch
    rng = np.random.default_rng(11)
    x = ragged(rng, 20_000)
    y = rng.standard_normal(x.size)
    xi = queries(rng, x, (1 << 21) + 77, np.float64)
    plan = b200.Interp1Plan(x, y)
    want = g1oracle.grad(x, y, xi, extrap=-3.0)
    for got, ref in zip(plan.grad(xi, extrap=-3.0), want):
        assert same_as_oracle(got, ref)
    # every buffer pinned: the two-slot pipeline
    from armadillocudalinearinterpolation_b200 import _lib
    pin = [torch.empty(xi.size, dtype=torch.float64).pin_memory() for _ in range(3)]
    pin[0].copy_(torch.from_numpy(xi))
    assert _lib.lib().b200_interp1_grad(plan._h, C.c_void_p(pin[0].data_ptr()), C.c_size_t(xi.size),
                                        C.c_void_p(pin[1].data_ptr()), C.c_void_p(pin[2].data_ptr()),
                                        C.c_double(-3.0)) == 0
    assert same_as_oracle(pin[1].numpy(), want[0]) and same_as_oracle(pin[2].numpy(), want[1])
    plan.close()


@pytest.mark.gpu
def test_gradient_config1_every_query(b200, g1oracle):
    """BASELINE config 1: 1e6 knots x 1e7 queries, every query against the oracle."""
    import torch
    rng = np.random.default_rng(12)
    x = np.linspace(0.0, 1.0, 1_000_000)
    y = np.sin(7 * x) + rng.standard_normal(x.size) * 1e-3
    plan = b200.Interp1Plan(x, y)
    assert plan.lookup_mode == 0
    xi = rng.uniform(-0.01, 1.01, 10_000_000)
    yi, dy = plan.grad(torch.from_numpy(xi).cuda())
    want = g1oracle.grad(x, y, xi)
    assert same_as_oracle(yi.cpu().numpy(), want[0]) and same_as_oracle(dy.cpu().numpy(), want[1])
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,mode", [("linspace", 2, 2), ("ragged", 257, 2), ("linspace", 6000, 2),
                                         ("quasi", 1_000_000, 0), ("ragged", 1_000_000, 1)])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_adjoint_matches_oracle(b200, g1oracle, dt, kind, n, mode):
    import torch
    rng = np.random.default_rng(21 + n)
    x = knots(rng, kind, n, dt)
    plan = b200.Interp1Plan(x, rng.standard_normal(x.size).astype(dt))
    check_mode(plan, mode, dt)
    xi = queries(rng, x, 300_011, dt)
    seg = min(x.size - 2, 1)
    xi[12000:82000] = rng.uniform(x[seg], x[seg + 1], 70_000).astype(dt)   # > B^2 terms on two nodes
    g = rng.standard_normal(xi.size).astype(dt)
    g[:12] = [np.inf, -np.inf, np.nan, -0.0, 0.0, np.finfo(dt).smallest_subnormal, 1e30, -1e-30, 2, 3, 4, 5]
    want = g1oracle.adjoint(x, xi, g)
    assert same_as_oracle(plan.adjoint(xi, g), want)
    tx, tg = torch.from_numpy(xi).cuda(), torch.from_numpy(g).cuda()
    d = plan.adjoint(tx, tg)
    torch.cuda.synchronize()
    assert same_as_oracle(d.cpu().numpy(), want)
    for m in (0, 1, 2, 300):
        assert same_as_oracle(plan.adjoint(xi[:m], g[:m]), g1oracle.adjoint(x, xi[:m], g[:m]))
    plan.close()


@pytest.mark.gpu
def test_adjoint_rejections(b200):
    import torch
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    plan = b200.Interp1Plan(np.linspace(0, 1, 40), np.zeros(40))
    t = torch.zeros(100, dtype=torch.float64, device="cuda")
    G = torch.zeros(40, dtype=torch.float64, device="cuda")
    need = C.c_size_t()
    assert lib.b200_interp1_adjoint_workspace(plan._h, C.c_size_t(100), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = C.c_void_p(t.data_ptr())
    call = lambda wsb, ni=100: lib.b200_interp1_adjoint_dev(plan._h, p, p, C.c_size_t(ni), C.c_void_p(G.data_ptr()),
                                                            C.c_void_p(ws.data_ptr()), C.c_size_t(wsb), s)
    assert call(need.value - 1) == -1 and b"workspace" in lib.b200_last_error()
    assert call(need.value, ni=1 << 31) == -1
    assert lib.b200_interp1_adjoint_workspace(plan._h, C.c_size_t(1 << 31), C.byref(need)) == -1
    assert call(1 << 40) == 0
    torch.cuda.synchronize()
    with pytest.raises(TypeError):
        plan.adjoint(t, t.float())
    with pytest.raises(ValueError):
        plan.adjoint(t, t[:50])
    with pytest.raises(ValueError):
        plan.adjoint(np.zeros(3), np.zeros(4))


@pytest.mark.gpu
def test_adjoint_deterministic_on_a_stream_in_a_graph_and_in_one_segment(b200, g1oracle):
    """1e6 knots, 1e7 random queries: the oracle's bits, the same bits from a second call, from a non-default stream and
    from replays of a captured CUDA graph with new g; then 1e7 queries in one segment."""
    import torch
    from armadillocudalinearinterpolation_b200 import _lib
    lib = _lib.lib()
    x = np.linspace(0.0, 1.0, 1_000_000)
    plan = b200.Interp1Plan(x, np.cos(x))
    ni = 10_000_000
    gen = torch.Generator(device="cuda").manual_seed(31)
    xi = torch.rand(ni, generator=gen, device="cuda", dtype=torch.float64) * 1.02 - 0.01
    g = torch.randn(ni, generator=gen, device="cuda", dtype=torch.float64)
    a = plan.adjoint(xi, g)
    b = plan.adjoint(xi, g)
    torch.cuda.synchronize()
    assert torch_same_ints(a, b)
    assert same_as_oracle(a.cpu().numpy(), g1oracle.adjoint(x, xi.cpu().numpy(), g.cpu().numpy()))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = plan.adjoint(xi, g)
    s.synchronize()
    assert torch_same_ints(a, c)
    need = C.c_size_t()
    assert lib.b200_interp1_adjoint_workspace(plan._h, C.c_size_t(ni), C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device="cuda")
    G = torch.empty(x.size, dtype=torch.float64, device="cuda")

    def run():
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        assert lib.b200_interp1_adjoint_dev(plan._h, C.c_void_p(xi.data_ptr()), C.c_void_p(g.data_ptr()),
                                            C.c_size_t(ni), C.c_void_p(G.data_ptr()), C.c_void_p(ws.data_ptr()),
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
    g.copy_(torch.randn(ni, device="cuda", dtype=torch.float64))
    graph.replay()
    torch.cuda.synchronize()
    assert torch_same_ints(G, plan.adjoint(xi, g))
    # every query in one segment: two nodes of 1e7 terms each (three levels of R)
    x1 = float(x[1234] + 0.3 * (x[1235] - x[1234]))
    xs = torch.full((ni,), x1, dtype=torch.float64, device="cuda") + torch.rand(ni, generator=gen, device="cuda",
                                                                                 dtype=torch.float64) * 1e-7
    d1 = plan.adjoint(xs, g).cpu().numpy()
    assert same_ints(d1, g1oracle.adjoint(x, xs.cpu().numpy(), g.cpu().numpy()))
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [9, 3000])
def test_autograd_gradcheck_and_bits(b200, n):
    import torch
    rng = np.random.default_rng(41)
    x = ragged(rng, n)
    y = rng.standard_normal(x.size)
    plan = b200.Interp1Plan(x, y)
    m = 64
    i = rng.integers(0, x.size - 1, m)
    xi0 = x[i] + (0.2 + 0.6 * rng.random(m)) * (x[i + 1] - x[i])
    XI = torch.from_numpy(xi0).cuda().requires_grad_()
    Y = torch.from_numpy(y).cuda().requires_grad_()
    assert torch.autograd.gradcheck(lambda a, b: plan.interp_torch(a, b), (XI, Y), eps=1e-6, atol=1e-7)
    g = torch.randn(m, dtype=torch.float64, device="cuda")
    out = plan.interp_torch(XI, Y)
    plan.set_values(np.zeros_like(y))
    out.backward(g)
    plan.set_values(y)
    yi, dy = plan.grad(XI.detach())
    dY = plan.adjoint(XI.detach(), g)
    torch.cuda.synchronize()
    assert torch_same_ints(out.detach(), yi)
    assert torch_same_ints(XI.grad, g * dy) and torch_same_ints(Y.grad, dY)
    XI.grad = None
    out2 = plan.interp_torch(XI.detach())     # queries that need no gradient: the value call
    assert not out2.requires_grad
    out3 = plan.interp_torch(XI)
    out3.sum().backward()
    torch.cuda.synchronize()
    assert torch_same_ints(out2, yi) and torch_same_ints(XI.grad, dy)
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
def test_cpp_grad_and_adjoint(b200, g1oracle, host):
    rng = np.random.default_rng(51)
    x = ragged(rng, 571)
    y = special_y(rng.standard_normal(x.size), rng)
    xi = queries(rng, x, 30_000, np.float64)
    n, ni = x.size, xi.size
    yi, dy = np.empty(ni), np.empty(ni)
    rc = host.b200_host_interp1_grad(_dp(x), n, _dp(y), n, _dp(xi), ni, _dp(yi), _dp(dy), C.c_double(-2.0))
    assert rc == 0, host.b200_host_last_error()
    for got, ref in zip((yi, dy), g1oracle.grad(x, y, xi, extrap=-2.0)):
        assert same_as_oracle(got, ref)
    g = rng.standard_normal(ni)
    d = np.empty(n)
    rc = host.b200_host_interp1_adjoint(_dp(x), _dp(y), n, _dp(xi), ni, _dp(g), ni, _dp(d))
    assert rc == 0, host.b200_host_last_error()
    assert same_ints(d, g1oracle.adjoint(x, xi, g))
    rc = host.b200_host_interp1_grad(_dp(x), n, _dp(y), n - 1, _dp(xi), ni, _dp(yi), _dp(dy), C.c_double(-2.0))
    assert rc == -1 and b"X and Y must have the same number" in host.b200_host_last_error()
    rc = host.b200_host_interp1_adjoint(_dp(x), _dp(y), n, _dp(xi), ni, _dp(g), ni - 1, _dp(d))
    assert rc == -1 and b"Adjoint: XI and G" in host.b200_host_last_error()
