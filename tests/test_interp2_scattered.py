"""Scattered interp2 (b200_interp2_scattered_dev, b200_interp2_scattered) against the CPU oracle: every build of the
value kernels, reached by a restatement of the launcher's route; the straight-line kernel of the headline path on the
queries it hands to its slow path and on the benchmark's 1e8 cell-sorted queries; the on-device locality probe that
picks between it and the generic kernel, at its threshold and at every gate in front of it; the range limits of the
branch-free divide in every f64 path (interp1 included); the host pipelines' chunking; the banded pipeline's two
chunk sizes and its slab boundary.

Bits are compared on integer views, so -0.0 counts; NaN is compared by position only (payloads may differ between the
host and the device).  Device outputs are written into a buffer filled with a sentinel, which must survive outside
the nq outputs and be gone inside them: a kernel pair whose probes disagree, or a tail nobody writes, leaves it
behind."""
import ctypes as C
import os

import numpy as np
import pytest

from armadillocudalinearinterpolation_b200 import _lib

pytestmark = pytest.mark.gpu

SENTINEL = -1234.5678
NT = os.cpu_count() or 8
EXTRAPS = (np.nan, -0.0, 2.5, np.inf)
GATE = 1 << 20                      # plan2_scattered_launch: the straight-line kernel is launched from 2^20 queries on
PROBE_PAIRS, PROBE_THRESHOLD = 1024, 640      # queries_are_local (interp2.cu)
BAND_SLAB = 1 << 27                 # kBandSlab: the banded pipeline runs in slabs of this many queries
NO_CELLS, FORCE_CELLS, NO_BANDS, FORCE_BANDS, NO_TILES, FORCE_TILES, ORDER_YX = 1, 2, 4, 8, 16, 32, 64
MiB = 1 << 20


def ints(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def same_as_oracle(a, ref, chunk=1 << 24):
    """Equal bits wherever the oracle is not NaN, NaN at the same places (in chunks: no copy of 1e8 outputs)."""
    a, ref = np.asarray(a).ravel(), np.asarray(ref).ravel()
    if a.shape != ref.shape or a.dtype != ref.dtype:
        return False
    for s in range(0, a.size, chunk):
        x, r = a[s:s + chunk], ref[s:s + chunk]
        nx, nr = np.isnan(x), np.isnan(r)
        if not (np.array_equal(nx, nr) and np.array_equal(ints(x)[~nx], ints(r)[~nr])):
            return False
    return True


def sentinel_bits(dt):
    return ints(np.array([SENTINEL], dt))[0]


# ---- restatement of the launcher's route (interp_common.cuh: axis_create; interp2.cu: table_layout, plan2_create,
#      plan2_scattered_launch, queries_are_local) ----

def c_int(t):
    """(int)t as the device converts (cvt.rzi.s32): toward zero, saturating, NaN -> 0"""
    t = np.asarray(t, np.float64)
    t = np.where(np.isnan(t), 0.0, t)
    return np.clip(np.trunc(np.clip(t, -2.0 ** 31, 2.0 ** 31 - 1)), -2 ** 31, 2 ** 31 - 1).astype(np.int64)


class Axis:
    """axis_create: lookup mode, bucket count, inv_w, step and the affine flag, in the knots' own precision"""

    def __init__(self, k):
        k = np.ascontiguousarray(k)
        T = k.dtype.type
        n = k.size
        self.n, self.x0, self.xmax = n, k[0], k[-1]
        with np.errstate(all="ignore"):
            span = T(k[-1] - k[0])
            self.nb, self.inv_w = n - 1, T(n - 1) / span
            self.step = span / T(n - 1)
            b = np.clip(c_int((k - k[0]) * self.inv_w), 0, n - 2)
            uniform = bool(np.all(np.abs(b - np.arange(n)) <= 1))
            j = np.arange(n - 1).astype(T)
            knots_affine = bool(np.all(k[:-1] == j * self.step + k[0]))
        finite_step = bool(np.isfinite(self.step) and self.step > 0)
        self.affine = finite_step and knots_affine
        self.mode = 0
        if not np.isfinite(self.inv_w) or not uniform:
            self.mode, self.nb = 1, n
            with np.errstate(all="ignore"):
                self.inv_w = T(n) / span
            if not np.isfinite(self.inv_w):
                self.inv_w = T(0)

    def smem_bytes(self, esz):
        pad16 = lambda b: (b + 15) & ~15
        if self.affine:
            return 0
        return pad16(esz * self.n) + (pad16(4 * (self.nb + 1)) if self.mode else 0)

    def safe(self):
        """the straight-line kernel's range rule for one axis"""
        lo, hi = 2.0 ** -400, 2.0 ** 400
        return bool(self.affine and self.mode == 0 and self.n >= 3 and lo <= self.step <= hi and lo <= self.inv_w <= hi)


class PlanInfo:
    """What plan2_create decides for (x, y, flags): shared-memory axes, table layout, banded pipeline"""

    def __init__(self, x, y, flags=0):
        x, y = np.asarray(x), np.asarray(y)
        self.f64 = x.dtype == np.float64
        self.t = "f64" if self.f64 else "f32"
        esz = x.dtype.itemsize
        self.V = 32 // esz
        self.X, self.Y = Axis(x), Axis(y)
        self.yfirst = bool(flags & ORDER_YX)
        self.use_smem = 16 + self.X.smem_bytes(esz) + self.Y.smem_bytes(esz) <= 110 * 1024
        zbytes = x.size * y.size * esz
        tiles = bool(flags & FORCE_TILES) or (not (flags & (NO_TILES | FORCE_CELLS | NO_CELLS)) and self.f64 and
                                               12 * MiB < zbytes < 180 * MiB)
        by_size = (zbytes <= 12 * MiB or zbytes >= 180 * MiB) if self.f64 else (zbytes <= 10 * MiB or zbytes >= 200 * MiB)
        records = bool(flags & (FORCE_CELLS | FORCE_BANDS)) or (not tiles and not (flags & NO_CELLS) and by_size)
        self.records = records and self.use_smem and 4 * zbytes <= 32 << 30
        self.tiles = tiles and self.use_smem and not (self.records and (flags & FORCE_CELLS))
        self.band_K, self.band_rounds = 0, 0
        ax_b = 16 + self.X.smem_bytes(esz)
        if (flags & FORCE_BANDS) and not (flags & NO_BANDS) and self.records and x.size * y.size < 0xfffffffe and \
                ax_b + 2048 * 2 * esz + 1024 <= 200 * 1024:
            rounds = 2 if ax_b + 2 * 2048 * 2 * esz + 1024 <= 110 * 1024 else 1
            nx, col = x.size, y.size * 4 * esz
            s = 0
            while (2 << s) * col <= 32 * MiB and (2 << s) < nx:
                s += 1
            while s > 0 and (nx + (1 << s) - 1) >> s < 4:
                s -= 1
            while (nx + (1 << s) - 1) >> s > 64:
                s += 1
            K = (nx + (1 << s) - 1) >> s
            if K >= 2:
                self.band_K, self.band_rounds = K, rounds

    def straight_line_launched(self, nq, aligned):
        return (self.f64 and aligned and nq // self.V > 0 and self.use_smem and self.tiles and self.X.safe() and
                self.Y.safe() and nq >= GATE)

    def probe_count(self, xq, yq, nq_vec):
        """queries_are_local's count: of the pairs (i, i + 1), i = (nq_vec / 1024) s, those whose tiles
        (cell / 3, cell clamped to [0, n - 2]) are at most 1 apart along X and 2 along Y"""
        return int(np.count_nonzero(self.probe_near(xq, yq, nq_vec)))

    def probe_near(self, xq, yq, nq_vec):
        """the probe's verdict on each of its 1024 sample pairs (none when nq_vec < 2048)"""
        step = nq_vec // PROBE_PAIRS
        if step < 2:
            return np.zeros(PROBE_PAIRS, bool)
        i = step * np.arange(PROBE_PAIRS)

        def tile(A, q):
            with np.errstate(all="ignore"):
                t = (np.asarray(q, np.float64) - np.float64(A.x0)) * np.float64(A.inv_w)
            return np.clip(c_int(t), 0, A.n - 2) // 3

        dx = np.abs(tile(self.X, xq[i]) - tile(self.X, xq[i + 1]))
        dy = np.abs(tile(self.Y, yq[i]) - tile(self.Y, yq[i + 1]))
        return (dx <= 1) & (dy <= 2)

    def route(self, xq, yq, aligned, device=True):
        """The value builds that serve one call of nq = xq.size queries (the banded pipeline only serves device
        buffers; of the straight-line pair, the one the probe picks)"""
        nq = xq.size
        if nq == 0:
            return set()
        if device and self.band_K >= 2:
            return {f"banded<{self.t},{self.band_rounds}>"}
        nvec = nq // self.V if aligned else 0
        out = set()
        if nvec and self.use_smem:
            if self.straight_line_launched(nq, aligned) and \
                    self.probe_count(xq, yq, nvec * self.V) >= PROBE_THRESHOLD:
                out.add(f"affine_tiles<{str(self.yfirst).lower()}>")
            else:
                out.add(f"smem<{self.t},{2 if self.tiles else 1 if self.records else 0}>")
        elif nvec:
            out.add(f"vec<{self.t}>")
        if nvec * self.V < nq:
            out.add(f"scalar<{self.t}>")
        return out


ALL_BUILDS = ({f"smem<{t},{l}>" for t in ("f64", "f32") for l in (0, 1, 2)} | {"affine_tiles<false>", "affine_tiles<true>"} |
              {f"{k}<{t}>" for k in ("vec", "scalar") for t in ("f64", "f32")} |
              {f"banded<{t},{r}>" for t in ("f64", "f32") for r in (1, 2)})


# ---- inputs ----

def ragged(rng, n, dt):
    """strictly ascending, unevenly spaced knots (no affine axis)"""
    x = np.unique(np.cumsum(0.25 + rng.random(n)).astype(dt))
    assert x.size == n
    return x


def special_z(rng, ny, nx, dt):
    """Z with NaN, +-inf, -0.0 and subnormals (some on the last row and column), whole cells of -0.0, an infinite
    column and a row of -inf"""
    z = rng.standard_normal((ny, nx)).astype(dt)
    tiny = np.finfo(dt).smallest_subnormal
    specials = np.array([np.nan, np.inf, -np.inf, -0.0, tiny, -3 * tiny, 7 * tiny], dt)
    k = min(z.size - 4, 3 * specials.size)
    z.reshape(-1)[rng.choice(z.size, k, replace=False)] = np.resize(specials, k)
    z[-1, -1] = -0.0
    z[-1, 0] = tiny
    z[0, -1] = -5 * tiny
    z[-1, nx // 2] = np.inf
    z[ny // 2, -1] = np.nan
    z[ny // 3:ny // 3 + 2, nx // 3:nx // 3 + 2] = -0.0          # a whole cell of -0.0 ...
    z[-2:, -2:] = -0.0                                        # ... and the last cell
    z[:, nx // 5] = np.inf
    z[ny // 5, :] = -np.inf
    return z


def cell_sorted(rng, x, y, n, margin=0.0):
    """n uniform queries over the grid (and `margin` of the span beyond it), ordered by grid cell"""
    dt = x.dtype
    sx, sy = float(x[-1] - x[0]), float(y[-1] - y[0])
    xq = rng.uniform(x[0] - margin * sx, x[-1] + margin * sx, n).astype(dt)
    yq = rng.uniform(y[0] - margin * sy, y[-1] + margin * sy, n).astype(dt)
    cx = np.clip(np.searchsorted(x, xq, "right") - 1, 0, x.size - 1)
    cy = np.clip(np.searchsorted(y, yq, "right") - 1, 0, y.size - 1)
    o = np.argsort(cx * y.size + cy, kind="stable")
    return xq[o], yq[o]


def edge_queries(k, rng, n_other, other, cap=600):
    """every knot of axis k (of a long axis: `cap` of them, both ends included), the neighbours of both ends and the
    non-finite values, each paired with a coordinate of the other axis"""
    dt = k.dtype.type
    lo, hi = k[0], k[-1]
    if k.size > cap:
        k = k[np.unique(np.concatenate([np.linspace(0, k.size - 1, cap).astype(int), [1, 2, k.size - 3, k.size - 2]]))]
    ends = np.array([np.nextafter(lo, dt(-np.inf)), lo, np.nextafter(lo, dt(np.inf)),
                     np.nextafter(hi, dt(-np.inf)), hi, np.nextafter(hi, dt(np.inf)), np.nan, np.inf, -np.inf], dt)
    a = np.concatenate([k, ends, np.full(n_other, hi)])
    b = np.concatenate([rng.uniform(other[0], other[-1], k.size).astype(dt), rng.uniform(other[0], other[-1], ends.size).astype(dt),
                        other[np.linspace(0, other.size - 1, n_other).astype(int)]])
    return a, b


def special_queries(rng, x, y):
    """the straight-line kernel's slow-path queries: every knot of both axes, the last row and column, both
    neighbours of each end, NaN and +-inf in either coordinate, knot hits in both coordinates"""
    ax, ay = edge_queries(x, rng, 40, y)
    by, bx = edge_queries(y, rng, 40, x)
    kx = x[rng.integers(0, x.size, 200)]
    ky = y[rng.integers(0, y.size, 200)]
    return np.concatenate([ax, bx, kx]), np.concatenate([ay, by, ky])


def embed(xq, yq, sx, sy, block_at):
    """sx, sy written into the sorted stream one per group of four queries (at lane m % 4, the other three lanes
    ordinary), never on a probe sample, and once more as one contiguous block from `block_at`"""
    xq, yq = xq.copy(), yq.copy()
    m = np.arange(sx.size)
    pos = 8 + 16 * m + (m % 4)
    assert pos[-1] < block_at
    xq[pos], yq[pos] = sx, sy
    xq[block_at:block_at + sx.size], yq[block_at:block_at + sx.size] = sx, sy
    return xq, yq


# ---- calls ----

def torch_at(a, offset):
    """a as a CUDA tensor starting `offset` elements past a 32-byte (allocation) boundary"""
    import torch
    buf = torch.empty(offset + a.size + 1, dtype=torch.float64 if a.dtype == np.float64 else torch.float32, device="cuda")
    t = buf[offset:offset + a.size]
    t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    return t


def dev_call(plan, tx, ty, extrap, oz=0, tail=37):
    """b200_interp2_scattered_dev with zq `oz` elements into a buffer filled with SENTINEL; asserts the sentinel is
    intact outside zq and gone inside it.  Returns (status, zq, zq's address)."""
    import torch
    n = tx.numel()
    buf = torch.full((oz + n + tail,), SENTINEL, dtype=tx.dtype, device="cuda")
    zq = buf[oz:oz + n]
    rc = _lib.lib().b200_interp2_scattered_dev(plan._h, C.c_void_p(tx.data_ptr()), C.c_void_p(ty.data_ptr()),
                                               C.c_size_t(n), C.c_void_p(zq.data_ptr()), C.c_double(extrap),
                                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    h = buf.cpu().numpy()
    s = sentinel_bits(h.dtype)
    assert np.all(ints(h[:oz]) == s) and np.all(ints(h[oz + n:]) == s), "scattered_dev wrote outside zq"
    out = h[oz:oz + n]
    assert not np.any(ints(out) == s), f"{np.count_nonzero(ints(out) == s)} outputs never written"
    return rc, out, zq.data_ptr()


def aligned(*ptrs):
    return all(p % 32 == 0 for p in ptrs)


def oracle2(oracle, x, y, z, xq, yq, extrap, y_first):
    ref = oracle.interp2_scattered(x, y, z, xq, yq, extrap=extrap, nthreads=NT, y_first=y_first)
    assert not np.any(ints(ref) == sentinel_bits(ref.dtype))
    return ref


# ---- 1. every build, every operand alignment ----

OFFSETS = [(0, 0, 0), (1, 0, 0), (0, 2, 0), (0, 0, 3), (3, 1, 2), (2, 3, 1)]
CASES = [  # name, dtype, flags
    ("records", "f64", 0), ("records", "f32", 0),
    ("column", "f64", NO_CELLS | NO_TILES), ("column", "f32", NO_CELLS | NO_TILES),
    ("tiles", "f64", FORCE_TILES), ("tiles", "f32", FORCE_TILES),
    ("straight_line", "f64", FORCE_TILES),
    ("wide", "f64", 0), ("wide", "f32", 0),
    ("banded2", "f64", FORCE_CELLS | FORCE_BANDS), ("banded2", "f32", FORCE_CELLS | FORCE_BANDS),
    ("banded1", "f64", FORCE_CELLS | FORCE_BANDS), ("banded1", "f32", FORCE_CELLS | FORCE_BANDS),
]


def case_inputs(name, t):
    """axes, Z, the queries (a prefix of them is each call's batch) and the batch sizes of one case"""
    dt = np.float64 if t == "f64" else np.float32
    rng = np.random.default_rng(61)
    V = 32 // np.dtype(dt).itemsize
    if name == "straight_line":
        x, y = np.linspace(-1.0, 2.0, 302), np.linspace(0.0, 1.0, 200)
        n = GATE + 3
    else:
        nx = {"wide": 14500 if t == "f64" else 29000, "banded1": 5000 if t == "f64" else 12000}.get(name, 300)
        x, y = ragged(rng, nx, dt), np.linspace(-2.0, 3.0, 40 if name in ("wide", "banded1") else 200).astype(dt)
        n = 40_000 + 3
    x, y = x.astype(dt), y.astype(dt)
    z = special_z(rng, y.size, x.size, dt)
    xq, yq = cell_sorted(rng, x, y, n, margin=0.02)
    sx, sy = special_queries(rng, x, y)
    xq, yq = embed(xq, yq, sx, sy, n // 2 + 8)
    k = (n - 3) // V
    return x, y, z, xq, yq, [0, 3, k * V, k * V + 1, k * V + 3]


def case_routes(name, t, y_first):
    x, y, _, xq, yq, nqs = case_inputs(name, t)
    flags = dict((c[0], c[2]) for c in CASES if c[1] == t)[name] | (ORDER_YX if y_first else 0)
    info = PlanInfo(x, y, flags)
    return {(offs, nq): info.route(xq[:nq], yq[:nq], offs == (0, 0, 0)) for offs in OFFSETS for nq in nqs}


def test_cases_reach_every_value_build():
    """By the restated route, the cases of test_every_value_build reach all sixteen builds of the value kernels."""
    reached = set()
    for name, t, _ in CASES:
        for y_first in (False, True):
            for r in case_routes(name, t, y_first).values():
                reached |= r
    assert reached == ALL_BUILDS, (ALL_BUILDS - reached, reached - ALL_BUILDS)


@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("name,t,flags", CASES)
def test_every_value_build(b200, oracle, name, t, flags, y_first):
    """Each case's plan, queries cell-sorted with every slow-path query embedded, Z with special values; xq, yq and
    zq 0-3 elements past a 32-byte boundary, nq = 0, 3 and kV + {0, 1, 3}, extrap NaN, -0.0, finite and +inf: the
    outputs equal the oracle's, every one of them is written and nothing else is.  The route restated from the
    plan's inputs and the actual addresses names the build that served each call."""
    x, y, z, xq, yq, nqs = case_inputs(name, t)
    flags |= ORDER_YX if y_first else 0
    info = PlanInfo(x, y, flags)
    intended = case_routes(name, t, y_first)
    plan = b200.Interp2Plan(x, y, z, flags=flags)
    refs = {e: oracle2(oracle, x, y, z, xq, yq, e, y_first) for e in EXTRAPS}
    served = set()
    for offs in OFFSETS:
        tx, ty = torch_at(xq, offs[0]), torch_at(yq, offs[1])
        for nq in nqs:
            for e in EXTRAPS:
                rc, got, zaddr = dev_call(plan, tx[:nq], ty[:nq], e, offs[2])
                r = info.route(xq[:nq], yq[:nq], aligned(tx.data_ptr(), ty.data_ptr(), zaddr))
                case = (offs, nq, e, sorted(r))
                assert rc == 0, case
                assert r == intended[(offs, nq)], case
                assert same_as_oracle(got, refs[e][:nq]), case
                served |= r
    assert served == set().union(*intended.values())
    plan.close()


# ---- 2. the straight-line kernel on its slow-path queries ----

@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("nx,ny", [(301, 200), (302, 201), (303, 199)])
def test_straight_line_kernel_slow_path_queries(b200, oracle, nx, ny, y_first):
    """Affine tile plans with nx - 1 and ny - 1 at every residue mod 3 (the clamped last tile row and column), a
    cell-sorted batch of 2^20 + 3 device queries that the restated probe calls local, with every knot of both axes,
    the last row and column, both neighbours of each end, NaN and +-inf in either coordinate and knot hits in groups
    of four next to ordinary queries; Z with NaN, +-inf, -0.0, subnormals and whole cells of -0.0."""
    rng = np.random.default_rng(62)
    x, y = np.linspace(-1.0, 2.0, nx), np.linspace(0.0, 1.0, ny)
    z = special_z(rng, ny, nx, np.float64)
    n = GATE + 3
    xq, yq = cell_sorted(rng, x, y, n, margin=0.01)
    sx, sy = special_queries(rng, x, y)
    xq, yq = embed(xq, yq, sx, sy, n // 2 + 8)
    flags = FORCE_TILES | (ORDER_YX if y_first else 0)
    info = PlanInfo(x, y, flags)
    assert info.X.safe() and info.Y.safe()
    tx, ty = torch_at(xq, 0), torch_at(yq, 0)
    plan = b200.Interp2Plan(x, y, z, flags=flags)
    for e in EXTRAPS:
        rc, got, zaddr = dev_call(plan, tx, ty, e)
        assert rc == 0
        assert info.route(xq, yq, aligned(tx.data_ptr(), ty.data_ptr(), zaddr)) == \
            {f"affine_tiles<{str(y_first).lower()}>", "scalar<f64>"}
        assert same_as_oracle(got, oracle2(oracle, x, y, z, xq, yq, e, y_first)), e
    plan.close()


def test_headline_plan_cell_sorted_queries_every_output(b200, oracle):
    """The benchmark's headline plan (4096^2 f64, default flags: tiles, affine axes) and its 1e8 queries of seed 2235
    ordered by grid cell as bench.py orders them: the straight-line kernel serves the call, every output is the
    oracle's."""
    import torch
    import bench
    x, y, z = bench.make_grid()
    info = PlanInfo(x, y, 0)
    assert info.tiles and info.X.safe() and info.Y.safe()
    g = torch.Generator(device="cuda").manual_seed(2235)
    xq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
    yq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
    cell = (xq * (bench.NX - 1)).floor().to(torch.int64) * bench.NY + (yq * (bench.NY - 1)).floor().to(torch.int64)
    order = cell.argsort()
    del cell
    xs, ys = xq[order], yq[order]
    del order, xq, yq
    hx, hy = xs.cpu().numpy(), ys.cpu().numpy()
    plan = b200.Interp2Plan(x, y, z)
    rc, got, zaddr = dev_call(plan, xs, ys, np.nan)
    assert rc == 0
    assert info.route(hx, hy, aligned(xs.data_ptr(), ys.data_ptr(), zaddr)) == {"affine_tiles<false>"}
    del xs, ys
    plan.close()
    assert same_as_oracle(got, oracle.interp2_scattered(x, y, z, hx, hy, nthreads=NT))


# ---- 3. the locality probe ----

def probe_plan():
    rng = np.random.default_rng(63)
    x, y = np.linspace(0.0, 1.0, 1201), np.linspace(-1.0, 1.0, 901)
    return x, y, special_z(rng, y.size, x.size, np.float64)


def with_count(info, xq, yq, nq_vec, target):
    """break sample pairs of a cell-sorted batch (the second query of the pair moved half the grid away along X)
    until the probe counts `target` near pairs"""
    xq = xq.copy()
    i = (nq_vec // PROBE_PAIRS) * np.arange(PROBE_PAIRS)
    near = np.flatnonzero(info.probe_near(xq, yq, nq_vec))
    assert near.size >= target
    x0, span = info.X.x0, info.X.xmax - info.X.x0
    for s in near[:near.size - target]:
        xq[i[s] + 1] = x0 + (xq[i[s]] - x0 + span / 2) % span
    assert info.probe_count(xq, yq, nq_vec) == target
    return xq


@pytest.mark.parametrize("y_first", [False, True])
@pytest.mark.parametrize("count", [639, 640, 641])
def test_probe_threshold(b200, oracle, count, y_first):
    """Batches whose probe count is exactly 639, 640 and 641: both kernels of the pair must reach the same decision
    in every CTA (if they disagree, no kernel or both write the outputs).  The restated probe gives the intended
    count and answer, the outputs equal the oracle's and every one of them is written."""
    rng = np.random.default_rng(64)
    x, y, z = probe_plan()
    flags = FORCE_TILES | (ORDER_YX if y_first else 0)
    info = PlanInfo(x, y, flags)
    n = GATE + 4 * 997
    xq, yq = cell_sorted(rng, x, y, n, margin=0.01)
    xq = with_count(info, xq, yq, n, count)
    tx, ty = torch_at(xq, 0), torch_at(yq, 0)
    plan = b200.Interp2Plan(x, y, z, flags=flags)
    rc, got, zaddr = dev_call(plan, tx, ty, 0.5)
    assert rc == 0
    served = info.route(xq, yq, aligned(tx.data_ptr(), ty.data_ptr(), zaddr))
    assert served == ({f"affine_tiles<{str(y_first).lower()}>"} if count >= PROBE_THRESHOLD else {"smem<f64,2>"})
    assert same_as_oracle(got, oracle2(oracle, x, y, z, xq, yq, 0.5, y_first))
    plan.close()


def gate_plan(kind):
    """(x, y, whether the straight-line kernel is eligible) for the probe's gates other than the query count"""
    y = np.linspace(-1.0, 1.0, 257)
    if kind == "n2":
        return np.array([0.0, 1.0]), y, False
    s = {"step_lo_in": 2.0 ** -400, "step_lo_out": np.nextafter(2.0 ** -400, 0.0),
         "step_hi_in": 2.0 ** 400, "step_hi_out": np.nextafter(2.0 ** 400, np.inf)}[kind]
    return np.linspace(0.0, 256 * s, 257), y, kind.endswith("_in")


@pytest.mark.parametrize("kind,nq", [("count", GATE - 1), ("count", GATE), ("count", GATE + 3), ("n2", GATE + 3),
                                     ("step_lo_in", GATE + 3), ("step_lo_out", GATE + 3),
                                     ("step_hi_in", GATE + 3), ("step_hi_out", GATE + 3)])
def test_probe_gates(b200, oracle, kind, nq):
    """Both sides of each gate in front of the probe: nq = 2^20 - 1, 2^20, 2^20 + 3; an axis of two knots; affine
    steps on and just outside 2^-400 and 2^400.  Cell-sorted queries: where the pair is launched the probe picks the
    straight-line kernel.  The restated route agrees, the outputs equal the oracle's."""
    rng = np.random.default_rng(65)
    if kind == "count":
        x, y, z = probe_plan()
        eligible = nq >= GATE
    else:
        x, y, eligible = gate_plan(kind)
        z = special_z(rng, y.size, x.size, np.float64)
    info = PlanInfo(x, y, FORCE_TILES)
    assert info.tiles and info.X.safe() == (kind == "count" or eligible)
    xq, yq = cell_sorted(rng, x, y, nq, margin=0.01)
    tx, ty = torch_at(xq, 0), torch_at(yq, 0)
    plan = b200.Interp2Plan(x, y, z, flags=FORCE_TILES)
    rc, got, zaddr = dev_call(plan, tx, ty, -1.5)
    assert rc == 0
    r = info.route(xq, yq, aligned(tx.data_ptr(), ty.data_ptr(), zaddr))
    assert info.straight_line_launched(nq, True) == eligible
    assert r - {"scalar<f64>"} == ({"affine_tiles<false>"} if eligible else {"smem<f64,2>"})
    assert same_as_oracle(got, oracle2(oracle, x, y, z, xq, yq, -1.5, False))
    plan.close()


# ---- 4. the branch-free divide's range limits ----

def tiny_distances():
    """distances from a knot across every binade from 2^-1074 to 2^-480, 2^-500 and its neighbours"""
    e = np.arange(-1074, -479)
    d = np.concatenate([np.ldexp(m, e) for m in (1.0, 1.25, 1.5, 1.9999999999999998)])
    edge = 2.0 ** -500
    d = np.concatenate([d, [edge, np.nextafter(edge, 0.0), np.nextafter(edge, 1.0), 2.0 ** -1074]])
    return np.unique(d[d > 0])


def tiny_2d_inputs(x, y):
    """queries at tiny distances from the zero knot of x (both sides) and above the zero knot of y, and Z with 0 on
    those knots and 1e300 on their neighbours"""
    rng = np.random.default_rng(66)
    d = tiny_distances()
    jx, jy = int(np.flatnonzero(x == 0)[0]), int(np.flatnonzero(y == 0)[0])
    ry = rng.uniform(y[jy + 1], y[-1], d.size)
    rx = rng.uniform(x[0], x[-1], d.size)
    xq = np.concatenate([d, -d, rx, d, -d])
    yq = np.concatenate([ry, ry, d, d, d])
    z = rng.standard_normal((y.size, x.size))
    z[:, jx] = np.where(np.arange(y.size) % 2, -0.0, 0.0)
    z[:, [jx + 1] + ([jx - 1] if jx else [])] = 1e300
    z[jy, :] = np.where(np.arange(x.size) % 2, 0.0, -0.0)
    z[jy + 1, :] = 1e300
    return xq, yq, z


def check_layouts(b200, oracle, x, y, z, xq, yq, layouts, y_first=False):
    """the queries through each plan layout, aligned and 1 / 3 elements off: the oracle's bits"""
    served = set()
    for flags in layouts:
        flags |= ORDER_YX if y_first else 0
        info = PlanInfo(x, y, flags)
        plan = b200.Interp2Plan(x, y, z, flags=flags)
        for e in (np.nan, 0.75):
            ref = oracle2(oracle, x, y, z, xq, yq, e, y_first)
            for offs in ((0, 0, 0), (1, 3, 1)):
                tx, ty = torch_at(xq, offs[0]), torch_at(yq, offs[1])
                rc, got, zaddr = dev_call(plan, tx, ty, e, offs[2])
                r = info.route(xq, yq, aligned(tx.data_ptr(), ty.data_ptr(), zaddr))
                assert rc == 0 and same_as_oracle(got, ref), (flags, e, offs, sorted(r))
                served |= r
        plan.close()
    return served


def test_divide_range_limits_straight_line_and_generic(b200, oracle):
    """An affine grid whose axes have an exact 0 knot; queries at distances 2^-1074 .. 2^-480 from it (a_err at,
    below and above 2^-500), Z = 0 / -0.0 there and 1e300 on the neighbouring knots, so a weight wrong in its last bit
    changes the output.  Through the straight-line kernel (the queries cell-sorted inside a 2^20-query batch), the
    generic kernel with each table layout, the banded pipeline and the scalar kernel."""
    x, y = np.linspace(-1.0, 1.0, 2049), np.linspace(0.0, 3.0, 1000)
    assert x[1024] == 0.0 and y[0] == 0.0
    xq, yq, z = tiny_2d_inputs(x, y)
    served = check_layouts(b200, oracle, x, y, z, xq, yq,
                           [0, FORCE_CELLS, NO_CELLS | NO_TILES, FORCE_CELLS | FORCE_BANDS])
    assert {"smem<f64,2>", "smem<f64,1>", "smem<f64,0>", "scalar<f64>", "banded<f64,2>"} <= served
    # inside a large cell-sorted batch: the straight-line kernel
    rng = np.random.default_rng(67)
    n = GATE + 8
    bx, by = cell_sorted(rng, x, y, n - xq.size)
    allx, ally = np.concatenate([bx, xq]), np.concatenate([by, yq])
    cx = np.searchsorted(x, allx, "right") - 1
    cy = np.searchsorted(y, ally, "right") - 1
    o = np.argsort(cx * y.size + cy, kind="stable")
    allx, ally = allx[o], ally[o]
    for y_first in (False, True):
        info = PlanInfo(x, y, ORDER_YX if y_first else 0)
        tx, ty = torch_at(allx, 0), torch_at(ally, 0)
        plan = b200.Interp2Plan(x, y, z, flags=ORDER_YX if y_first else 0)
        rc, got, zaddr = dev_call(plan, tx, ty, np.nan)
        assert rc == 0
        assert info.route(allx, ally, aligned(tx.data_ptr(), ty.data_ptr(), zaddr)) == {f"affine_tiles<{str(y_first).lower()}>"}
        assert same_as_oracle(got, oracle2(oracle, x, y, z, allx, ally, np.nan, y_first))
        plan.close()


def test_divide_range_limits_vec_kernel(b200, oracle):
    """The same tiny distances on a ragged X axis too long for shared memory (the global-table kernel), with an exact
    0 knot made by shifting the knots."""
    rng = np.random.default_rng(68)
    x = ragged(rng, 14500, np.float64)
    x = x - x[7000]
    assert np.all(np.diff(x) > 0) and x[7000] == 0.0
    y = np.linspace(0.0, 3.0, 64)
    xq, yq, z = tiny_2d_inputs(x, y)
    assert not PlanInfo(x, y).use_smem
    served = check_layouts(b200, oracle, x, y, z, xq, yq, [0])
    assert served == {"vec<f64>", "scalar<f64>"}


@pytest.mark.parametrize("kind", ["huge_step", "overflowing_span"])
def test_divide_range_limits_large_operands(b200, oracle, kind):
    """Sums above 2^500 (an affine axis with a step of 2^600) and an axis whose span overflows
    ([-1.5e308, 1.5e308]: lookup mode 1, inv_w = 0), queries near both ends, through every table layout."""
    rng = np.random.default_rng(69)
    if kind == "huge_step":
        x = np.linspace(0.0, 256 * 2.0 ** 600, 257)
        info = Axis(x)
        assert info.affine and info.mode == 0 and not info.safe()
    else:
        x = np.linspace(-1.5, 1.5, 7) * 1e308
        info = Axis(x)
        assert info.mode == 1 and info.inv_w == 0 and not info.affine
    y = np.linspace(0.0, 1.0, 50)
    lo, hi, w = x[0], x[-1], x[1] - x[0]
    near = np.array([lo, np.nextafter(lo, np.inf), lo + w * 1e-300, lo + w * 1e-5, lo + w / 3, np.nextafter(x[1], -np.inf),
                     x[1], hi, np.nextafter(hi, -np.inf), hi - w * 1e-300, hi - w * 1e-5, hi - w / 3,
                     np.nextafter(hi, np.inf), np.nextafter(lo, -np.inf)])
    u = rng.random(4000)
    xq = np.concatenate([near, lo * (1 - u) + hi * u, x])         # (no hi - lo: it overflows)
    yq = rng.uniform(-0.05, 1.05, xq.size)
    z = special_z(rng, y.size, x.size, np.float64)
    z[:, 0] = 0.0
    z[:, 1] = 1e300
    z[:, -1] = -0.0
    z[:, -2] = -1e300
    check_layouts(b200, oracle, x, y, z, xq, yq, [0, FORCE_TILES, FORCE_CELLS, NO_CELLS | NO_TILES, FORCE_CELLS | FORCE_BANDS])


def interp1_axis(mode):
    """an axis of interp1 lookup mode `mode` with an exact 0 knot; its spacing is no power of two (a divide by a power
    of two is exact in any implementation)"""
    rng = np.random.default_rng(70)
    if mode == 2:
        return np.linspace(0.0, 3.0, 1000)                        # small enough for shared memory
    if mode == 0:
        return np.linspace(0.0, 3.0, 200_001)                     # uniform, too large for shared memory
    x = ragged(rng, 20_000, np.float64)
    return x - x[9000]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_divide_range_limits_interp1(b200, oracle, mode):
    """interp1 f64 in each lookup mode (0: the straight-line fast path of the record kernel, 1: bucket table,
    2: shared memory) on an axis with an exact 0 knot: queries at tiny distances on both sides of it (below the first
    knot: extrap), values 0 and -0.0 there and +-1e300 on its neighbours; also the huge-step and overflowing-span
    axes."""
    rng = np.random.default_rng(71)
    x = interp1_axis(mode)
    j = int(np.flatnonzero(x == 0)[0])
    y = rng.standard_normal(x.size)
    d = tiny_distances()
    xi = np.concatenate([d, -d, rng.uniform(x[0], x[-1], 20_000)])
    plan = b200.Interp1Plan(x, y)
    assert plan.lookup_mode == mode
    for zero in (0.0, -0.0):
        y[j], y[j + 1] = zero, -1e300
        if j:
            y[j - 1] = 1e300
        plan.set_values(y)
        yi, idx = plan(xi, extrap=0.5, return_index=True)
        yo, io = oracle.interp1(x, y, xi, extrap=0.5, nthreads=NT)
        assert same_as_oracle(yi, yo) and np.array_equal(idx, io), zero
    plan.close()
    for xk in (np.linspace(0.0, 1024 * 2.0 ** 600, 1025), np.linspace(-1.5, 1.5, 1025) * 1e308):
        w = xk[1] - xk[0]
        yk = rng.standard_normal(xk.size)
        yk[0], yk[1], yk[-1], yk[-2] = 0.0, 1e300, -0.0, -1e300
        xi = np.concatenate([xk, [xk[0] + w * 1e-300, xk[-1] - w * 1e-300, np.nextafter(xk[0], np.inf),
                                  np.nextafter(xk[-1], -np.inf)], xk[:-1] + w * rng.random(xk.size - 1)])
        xi = np.concatenate([xi, rng.uniform(0, 1, 20_000) * (xk[-1] / 2) + rng.uniform(0, 1, 20_000) * (xk[0] / 2)])
        p = b200.Interp1Plan(xk, yk)
        yi, idx = p(xi, extrap=0.5, return_index=True)
        yo, io = oracle.interp1(xk, yk, xi, extrap=0.5, nthreads=NT)
        assert same_as_oracle(yi, yo) and np.array_equal(idx, io)
        p.close()


# ---- 5. host routes ----

def host_call(plan, xq, yq, extrap, tail=37, zbuf=None):
    """b200_interp2_scattered into a host buffer (zbuf, or a fresh pageable one) filled with SENTINEL"""
    n = xq.size
    buf = np.empty(n + tail, xq.dtype) if zbuf is None else zbuf
    buf[:] = SENTINEL
    rc = _lib.lib().b200_interp2_scattered(plan._h, C.c_void_p(xq.ctypes.data), C.c_void_p(yq.ctypes.data),
                                           C.c_size_t(n), C.c_void_p(buf.ctypes.data), C.c_double(extrap))
    s = sentinel_bits(buf.dtype)
    assert np.all(ints(buf[n:]) == s), "scattered wrote outside zq"
    assert not np.any(ints(buf[:n]) == s), "outputs never written"
    return rc, buf[:n]


def test_host_pageable_chunks_at_the_gate(b200, oracle):
    """A pageable batch of 3 * 2^20 + 5 cell-sorted queries on a plan where the straight-line kernel is eligible:
    three 2^20-query chunks, each exactly at the gate with its own probe (local), then a 5-query chunk."""
    rng = np.random.default_rng(72)
    x, y, z = probe_plan()
    info = PlanInfo(x, y, FORCE_TILES)
    n = 3 * GATE + 5
    xq, yq = cell_sorted(rng, x, y, n, margin=0.01)
    sx, sy = special_queries(rng, x, y)
    xq, yq = embed(xq, yq, sx, sy, GATE + 8)
    chunks = [info.route(xq[o:o + GATE], yq[o:o + GATE], True, device=False) for o in range(0, n, GATE)]
    assert chunks == [{"affine_tiles<false>"}] * 3 + [{"smem<f64,2>", "scalar<f64>"}]
    plan = b200.Interp2Plan(x, y, z, flags=FORCE_TILES)
    rc, got = host_call(plan, xq, yq, np.inf)
    assert rc == 0
    assert same_as_oracle(got, oracle2(oracle, x, y, z, xq, yq, np.inf, False))
    plan.close()


def test_host_pinned_two_chunks(b200, oracle):
    """A pinned batch of 2^22 + 2^19 + 3 cell-sorted queries: one 2^22-query chunk (straight-line kernel), then one
    under 2^20 (the generic kernel alone), on the two-slot pipeline."""
    import torch
    rng = np.random.default_rng(73)
    x, y, z = probe_plan()
    info = PlanInfo(x, y, FORCE_TILES | ORDER_YX)
    n = (1 << 22) + (1 << 19) + 3
    xs, ys = cell_sorted(rng, x, y, n, margin=0.01)
    sx, sy = special_queries(rng, x, y)
    xs, ys = embed(xs, ys, sx, sy, (1 << 22) + 1000)
    assert [info.route(xs[o:o + (1 << 22)], ys[o:o + (1 << 22)], True, device=False) for o in (0, 1 << 22)] == \
        [{"affine_tiles<true>"}, {"smem<f64,2>", "scalar<f64>"}]
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    xq, yq = pin(xs), pin(ys)
    zbuf = torch.empty(n + 37, dtype=torch.float64).pin_memory().numpy()
    plan = b200.Interp2Plan(x, y, z, flags=FORCE_TILES | ORDER_YX)
    rc, got = host_call(plan, xq, yq, -0.0, zbuf=zbuf)
    assert rc == 0
    assert same_as_oracle(got, oracle2(oracle, x, y, z, xs, ys, -0.0, True))
    plan.close()


# ---- 6. the banded pipeline's slab boundary ----

def test_banded_across_the_slab_boundary(b200, oracle):
    """2^27 + 5 f32 queries through the banded pipeline: one full slab, then a 5-query slab; special queries on both
    sides of the boundary, zq one element off alignment so both slabs store element by element."""
    rng = np.random.default_rng(74)
    x, y = ragged(rng, 300, np.float32), np.linspace(-2.0, 3.0, 200).astype(np.float32)
    z = special_z(rng, y.size, x.size, np.float32)
    info = PlanInfo(x, y, FORCE_CELLS | FORCE_BANDS)
    assert info.band_K >= 2 and info.band_rounds == 2
    n = BAND_SLAB + 5
    xq = rng.uniform(x[0] - 1, x[-1] + 1, n).astype(np.float32)
    yq = rng.uniform(-2.1, 3.1, n).astype(np.float32)
    sx, sy = special_queries(rng, x, y)
    xq[n - sx.size:], yq[n - sx.size:] = sx, sy               # the last of them in the second slab
    plan = b200.Interp2Plan(x, y, z, flags=FORCE_CELLS | FORCE_BANDS)
    tx, ty = torch_at(xq, 0), torch_at(yq, 0)
    ref = oracle2(oracle, x, y, z, xq, yq, 1.25, False)
    for oz in (0, 1):
        rc, got, _ = dev_call(plan, tx, ty, 1.25, oz)
        assert rc == 0
        assert same_as_oracle(got, ref), oz
        del got
    plan.close()
