"""Host-buffer calls of the interpolation plans (host_run in csrc/host_staging.cuh, and the synchronous host adjoint)
against the device-buffer calls on the same inputs, bit for bit: pinned buffers over several 2^22-query pipeline chunks,
calls of different kinds alternating on one plan as the batch grows and shrinks, and the adjoint from host arrays."""
import ctypes as C

import numpy as np
import pytest

N_CHUNKS = 3 * (1 << 22) + 5   # four pipeline chunks: both slots used twice, and an odd tail
EXTRAP = -2.5


def ints(a):
    a = np.ascontiguousarray(a)
    return a.view({8: np.int64, 4: np.int32}[a.dtype.itemsize])


def same(host, dev):
    """host: a (pinned) CPU tensor or numpy array; dev: a CUDA tensor.  Equal bits."""
    h = host.numpy() if hasattr(host, "numpy") else host
    return h.shape == tuple(dev.shape) and np.array_equal(ints(h), ints(dev.cpu().numpy()))


def pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.from_numpy(a).dtype).pin_memory()
    t.copy_(torch.from_numpy(a))
    return t


def empty_pinned(n, like):
    import torch
    return torch.empty(n, dtype=like).pin_memory()


def ptr(t):
    return C.c_void_p(t.data_ptr())


def ragged(rng, n, dt=np.float64):
    return np.cumsum(0.25 + rng.random(n)).astype(dt)


def spread(rng, x, n, dt):
    """queries over the grid and 10 % beyond it on either side, with NaNs and the end knots among them"""
    w = x[-1] - x[0]
    q = rng.uniform(x[0] - 0.1 * w, x[-1] + 0.1 * w, n).astype(dt)
    k = min(n, 4)
    q[:k] = np.array([x[0], x[-1], np.nan, x[1]], dt)[:k]
    return q


@pytest.fixture(scope="module")
def lib(b200):
    from armadillocudalinearinterpolation_b200 import _lib
    return _lib.lib()


def make_plan1(b200, ng, dt, seed=1):
    rng = np.random.default_rng(seed)
    x = ragged(rng, ng, dt)
    return b200.Interp1Plan(x, rng.standard_normal(ng).astype(dt)), x


def make_plan2(b200, seed=2):
    rng = np.random.default_rng(seed)
    x = ragged(rng, 700)
    y = np.linspace(-1.0, 3.0, 500)
    return b200.Interp2Plan(x, y, rng.standard_normal((y.size, x.size))), x, y


def interp1_host(lib, plan, kind, hx, n, outs):
    """b200_interp1_exec (kind 'value' / 'idx') or b200_interp1_grad on the first n entries of pinned buffers"""
    if kind == "grad":
        return lib.b200_interp1_grad(plan._h, ptr(hx), C.c_size_t(n), ptr(outs[0]), ptr(outs[2]), C.c_double(EXTRAP))
    return lib.b200_interp1_exec(plan._h, ptr(hx), C.c_size_t(n), ptr(outs[0]), ptr(outs[1]) if kind == "idx" else None,
                                 C.c_double(EXTRAP))


def check_interp1(plan, kind, dx, n, outs):
    if kind == "grad":
        yi, dy = plan.grad(dx[:n], EXTRAP)
        return same(outs[0][:n], yi) and same(outs[2][:n], dy)
    if kind == "idx":
        yi, idx = plan(dx[:n], EXTRAP, return_index=True)
        return same(outs[0][:n], yi) and same(outs[1][:n], idx)
    return same(outs[0][:n], plan(dx[:n], EXTRAP))


@pytest.mark.gpu
@pytest.mark.parametrize("ng", [1000, 20_000])   # the shared-memory kernels, the global-table kernels
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_interp1_pinned_buffers_over_several_chunks(b200, lib, dt, ng):
    import torch
    plan, x = make_plan1(b200, ng, dt)
    xi = spread(np.random.default_rng(3), x, N_CHUNKS, dt)
    hx = pinned(xi)
    dx = hx.cuda()
    outs = [empty_pinned(N_CHUNKS, hx.dtype), empty_pinned(N_CHUNKS, torch.int32), empty_pinned(N_CHUNKS, hx.dtype)]
    for kind in ("value", "idx", "grad"):
        assert interp1_host(lib, plan, kind, hx, N_CHUNKS, outs) == 0
        assert check_interp1(plan, kind, dx, N_CHUNKS, outs), kind
    plan.close()


@pytest.mark.gpu
def test_interp2_pinned_buffers_over_several_chunks(b200, lib):
    plan, x, y = make_plan2(b200)
    rng = np.random.default_rng(4)
    hx, hy = pinned(spread(rng, x, N_CHUNKS, np.float64)), pinned(spread(rng, y, N_CHUNKS, np.float64))
    dx, dy = hx.cuda(), hy.cuda()
    hz, hdx, hdy = (empty_pinned(N_CHUNKS, hx.dtype) for _ in range(3))
    n = C.c_size_t(N_CHUNKS)
    assert lib.b200_interp2_scattered(plan._h, ptr(hx), ptr(hy), n, ptr(hz), C.c_double(EXTRAP)) == 0
    assert same(hz, plan.scattered(dx, dy, EXTRAP))
    assert lib.b200_interp2_scattered_grad(plan._h, ptr(hx), ptr(hy), n, ptr(hz), ptr(hdx), ptr(hdy),
                                           C.c_double(EXTRAP)) == 0
    zq, gx, gy = plan.scattered_grad(dx, dy, EXTRAP)
    assert same(hz, zq) and same(hdx, gx) and same(hdy, gy)
    plan.close()


# batch sizes of the alternating calls, in pipeline chunks: one, two, four, two, one
SIZES = [1000, (1 << 21) + (1 << 22) + 3, N_CHUNKS, (1 << 22) + 1, 777]


@pytest.mark.gpu
def test_interp1_alternating_calls_on_one_plan(b200, lib):
    """value + index, gradient, value, gradient at every size while the batch grows and then shrinks: the pipeline's
    buffers serve every array list of the plan"""
    import torch
    plan, x = make_plan1(b200, 20_000, np.float64, seed=5)
    hx = pinned(spread(np.random.default_rng(6), x, N_CHUNKS, np.float64))
    dx = hx.cuda()
    outs = [empty_pinned(N_CHUNKS, hx.dtype), empty_pinned(N_CHUNKS, torch.int32), empty_pinned(N_CHUNKS, hx.dtype)]
    for n in SIZES:
        for kind in ("idx", "grad", "value", "grad"):
            for o in outs:
                o.fill_(0)
            assert interp1_host(lib, plan, kind, hx, n, outs) == 0
            assert check_interp1(plan, kind, dx, n, outs), (n, kind)
    plan.close()


@pytest.mark.gpu
def test_interp2_alternating_calls_on_one_plan(b200, lib):
    plan, x, y = make_plan2(b200, seed=7)
    rng = np.random.default_rng(8)
    hx, hy = pinned(spread(rng, x, N_CHUNKS, np.float64)), pinned(spread(rng, y, N_CHUNKS, np.float64))
    dx, dy = hx.cuda(), hy.cuda()
    hz, hdx, hdy = (empty_pinned(N_CHUNKS, hx.dtype) for _ in range(3))
    for n in SIZES:
        for grad in (False, True, False, True):
            hz.fill_(0)
            if grad:
                assert lib.b200_interp2_scattered_grad(plan._h, ptr(hx), ptr(hy), C.c_size_t(n), ptr(hz), ptr(hdx),
                                                       ptr(hdy), C.c_double(EXTRAP)) == 0
                zq, gx, gy = plan.scattered_grad(dx[:n], dy[:n], EXTRAP)
                assert same(hz[:n], zq) and same(hdx[:n], gx) and same(hdy[:n], gy), n
            else:
                assert lib.b200_interp2_scattered(plan._h, ptr(hx), ptr(hy), C.c_size_t(n), ptr(hz),
                                                  C.c_double(EXTRAP)) == 0
                assert same(hz[:n], plan.scattered(dx[:n], dy[:n], EXTRAP)), n
    plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 3_000_001])
def test_host_adjoint_equals_device_adjoint(b200, n):
    import torch
    rng = np.random.default_rng(9 + n)
    p1, x = make_plan1(b200, 20_000, np.float64, seed=10)
    xi, g = spread(rng, x, n, np.float64), rng.standard_normal(n)
    assert same(p1.adjoint(xi, g), p1.adjoint(torch.from_numpy(xi).cuda(), torch.from_numpy(g).cuda()))
    p2, x, y = make_plan2(b200, seed=11)
    xq, yq = spread(rng, x, n, np.float64), spread(rng, y, n, np.float64)
    dev = p2.scattered_adjoint(*(torch.from_numpy(a).cuda() for a in (xq, yq, g)))
    assert same(p2.scattered_adjoint(xq, yq, g), dev)
    p1.close()
    p2.close()
