"""The C++ host layer (armadillocudalinearinterpolation_b200/host): the reference's solver
interfaces re-implemented over the Armadillo shim, and the drop-in map class.  CPU tests drive
NewtonSolver / Stability on analytic problems through host_capi.cpp; GPU tests drive the real
EventDrivenMapB200 through the same solvers and compare with the oracle's Newton trajectory."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "host")
LIBDIR = os.path.join(ROOT, "armadillocudalinearinterpolation_b200", "lib")
Z_DRIVER = np.array([np.float32(0.3310), np.float32(0.6914), np.float32(1.3557)], dtype=np.float64)
BETA = float(np.float32(13.0589))


@pytest.fixture(scope="module")
def host():
    subprocess.check_call(["make", "-C", HOST, "-j4"], stdout=subprocess.DEVNULL)
    lib = C.CDLL(os.path.join(LIBDIR, "libb200host.so"))
    lib.b200_host_last_error.restype = C.c_char_p
    return lib


def dp(a):
    return a.ctypes.data_as(C.c_void_p)


def newton_quadratic(host, guess, tol=1e-10, max_it=20, eps=1e-7, damping=1.0, use_jac=0):
    n = len(guess)
    g = np.array(guess, float); sol = np.zeros(n); hist = np.full(max_it + 1, np.nan)
    nh = C.c_int(); calls = C.c_int(); J = np.zeros((n, n), order="F")
    rc = host.b200_host_newton_quadratic(n, dp(g), C.c_double(tol), max_it, C.c_double(eps), C.c_double(damping),
                                         use_jac, dp(sol), dp(hist), C.byref(nh), C.byref(calls), dp(J))
    assert rc >= 0, host.b200_host_last_error()
    return dict(sol=sol, hist=hist[:nh.value], its=rc // 4, converged=bool(rc & 2), post_once=bool(rc & 1),
                calls=calls.value, J=J)


def test_newton_converges_quadratically_and_counts_calls(host):
    r = newton_quadratic(host, [1.0, 1.0, 1.0])
    assert r["converged"] and r["post_once"]
    u = r["sol"]
    F = u ** 2 - np.arange(2, 5) + 0.1 * np.roll(u, -1)
    assert np.max(np.abs(F)) < 1e-10
    assert len(r["hist"]) == r["its"] + 1 and r["hist"][-1] <= 1e-10        # history trimmed to the iterations done
    assert r["hist"][-1] < r["hist"][-2] ** 1.5                              # super-linear tail
    # reference cost model: 1 + its * (n + 1) evaluations with the solver's own FD loop (NewtonSolver.cpp:67,110,191)
    assert r["calls"] == 1 + r["its"] * 4
    rj = newton_quadratic(host, [1.0, 1.0, 1.0], use_jac=1)                  # user Jacobian: 1 + its evaluations
    assert rj["calls"] == 1 + rj["its"] and np.allclose(rj["sol"], u, atol=1e-9)
    assert np.allclose(rj["J"], r["J"], atol=1e-5)                           # pJacobianExternal hands out the last Jacobian
    # a problem that offers F and dF/dU in one call (AbstractNonlinearProblemFused): one fused call per iterate, no
    # plain ComputeF at all; same iterates, and the Jacobian handed out is still the last one a step was taken with
    rf = newton_quadratic(host, [1.0, 1.0, 1.0], use_jac=2)
    assert rf["calls"] == 1000 * (1 + rf["its"]) and rf["its"] == rj["its"] and rf["post_once"]
    assert np.array_equal(rf["sol"], rj["sol"]) and np.array_equal(rf["hist"], rj["hist"]) and np.array_equal(rf["J"], rj["J"])
    # ... or the Jacobian from the residual in hand: 1 + its plain evaluations, one given-F Jacobian per iteration
    rg = newton_quadratic(host, [1.0, 1.0, 1.0], use_jac=3)
    assert rg["calls"] == (1 + rg["its"]) + 1000000 * rg["its"] and rg["its"] == rj["its"]
    assert np.array_equal(rg["sol"], rj["sol"]) and np.array_equal(rg["hist"], rj["hist"]) and np.array_equal(rg["J"], rj["J"])


def test_newton_not_converged_and_damping(host):
    r = newton_quadratic(host, [1.0, 1.0, 1.0], max_it=2)
    assert not r["converged"] and r["its"] == 2 and len(r["hist"]) == 3 and r["post_once"]
    d = newton_quadratic(host, [1.0, 1.0, 1.0], damping=0.5, max_it=60, tol=1e-8)
    assert d["converged"] and d["its"] > r["its"]


@pytest.mark.parametrize("n", [3, 8, 40, 200])
def test_shim_solve_and_eig_gen_match_numpy(host, n):
    rng = np.random.default_rng(n)
    A = np.asfortranarray(rng.standard_normal((n, n)))
    b = rng.standard_normal(n); x = np.zeros(n)
    assert host.b200_host_solve(n, dp(A), dp(b), dp(x)) == 0
    assert np.allclose(x, np.linalg.solve(A, b), rtol=1e-9, atol=1e-9)
    re = np.zeros(n); im = np.zeros(n)
    cnt = host.b200_host_stability_linear(n, dp(A), 1, C.c_double(1e-6), 1, dp(re), dp(im))
    lam = np.linalg.eigvals(A)
    mine = np.sort_complex(re + 1j * im); ref = np.sort_complex(lam)
    assert np.allclose(mine, ref, rtol=1e-8, atol=1e-8)
    assert cnt == int(np.sum(np.abs(lam) > 1.0))
    assert host.b200_host_solve(2, dp(np.zeros((2, 2), order="F")), dp(np.ones(2)), dp(np.zeros(2))) == 1  # singular


def test_stability_problem_types(host):
    """flow counts Re > 0; map counts |lambda| > 1; equationFree adds I to the FD Jacobian of F = A u - u."""
    A = np.asfortranarray(np.diag([1.5, 0.5, -0.2]) + 0.01 * np.ones((3, 3)))
    re = np.zeros(3); im = np.zeros(3)
    # via the problem: F(u) = A u - u, J = A - I (FD, exact for a linear map up to rounding)
    assert host.b200_host_stability_linear(3, dp(A), 2, C.c_double(1e-6), 0, dp(re), dp(im)) == 1   # eig(A): one > 1
    assert np.allclose(np.sort(re), np.sort(np.linalg.eigvals(A).real), atol=1e-6)
    lamJ = np.linalg.eigvals(A - np.eye(3))
    assert host.b200_host_stability_linear(3, dp(A), 1, C.c_double(1e-6), 0, None, None) == int(np.sum(np.abs(lamJ) > 1)) == 1  # |eig(A - I)| > 1
    assert host.b200_host_stability_linear(3, dp(A), 0, C.c_double(1e-6), 0, None, None) == 1       # Re eig(A - I) > 0: one
    assert host.b200_host_stability_linear(3, dp(A), 0, C.c_double(1e-6), 1, None, None) == 2       # matrix overload on A itself


REF_DRIVER = os.path.join(os.environ.get("B200_REFERENCE_DIR", ""), "Driver.cu")


@pytest.mark.skipif(not os.environ.get("B200_REFERENCE_DIR") or not os.path.exists(REF_DRIVER),
                    reason="B200_REFERENCE_DIR does not name a checkout of the reference project")
def test_reference_driver_compiles_unmodified_against_the_host_layer(tmp_path, host):
    """Drop-in evidence: the reference's own Driver.cu (copied to a temp dir, never into the repo)
    compiles and links against this host layer + compat headers without a single edit."""
    src = tmp_path / "Driver_ref.cpp"
    shutil.copy(REF_DRIVER, src)
    exe = tmp_path / "ref_driver"
    cmd = ["/usr/bin/g++", "-std=c++14", "-O0", f"-I{HOST}/compat", f"-I{HOST}/arma_shim", f"-I{HOST}",
           f"-I{ROOT}/include", str(src)] + [os.path.join(HOST, f) for f in
           ("AbstractNonlinearSolver.cpp", "NewtonSolver.cpp", "Stability.cpp", "EventDrivenMapB200.cpp")] + \
          [f"-L{LIBDIR}", "-lb200edm", f"-Wl,-rpath,{LIBDIR}", "-o", str(exe)]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-3000:]
    assert exe.exists()


@pytest.mark.gpu
def test_edm_newton_through_the_reference_interfaces(host, oracle):
    """NewtonSolver drives EventDrivenMapB200 (a) through ComputeF only — the reference's sequential
    FD loop — and (b) through ComputeDFDU — one batched launch.  Same iterates, bit for bit, and the
    fixed point the oracle's Newton finds (Driver.cu settings: tol 1e-4, eps 1e-2, <= 10 iterations)."""
    R, N, n = 8, 1024, 3
    res = []
    for mode in (0, 1, 3):   # 3: plug-in Jacobian with the reference's call sequence (F, then dF/dU) instead of the fused one
        sol = np.zeros(n); hist = np.full(11, np.nan); nh = C.c_int(); J = np.zeros((n, n), order="F")
        rc = host.b200_host_edm_newton(C.c_double(BETA), R, N, dp(Z_DRIVER), n, C.c_double(1e-4), 10, C.c_double(1e-2),
                                       mode, C.c_double(0.0), dp(sol), dp(hist), C.byref(nh), dp(J))
        assert rc >= 0, host.b200_host_last_error()
        res.append((rc, sol, hist[:nh.value], J))
    assert res[0][0] == 1 and res[1][0] == 1 and res[2][0] == 1
    for other in (res[1], res[2]):
        assert np.array_equal(res[0][1], other[1]) and np.array_equal(res[0][2], other[2]) and np.array_equal(res[0][3], other[3])
    # oracle Newton with the same settings
    cfg = oracle.edm_cfg(R=1, N=N)
    z = Z_DRIVER.copy(); f, _ = oracle.edm_compute_f(cfg, z, aux=False); hist = [np.linalg.norm(f)]
    while hist[-1] > 1e-4 and len(hist) <= 10:
        Jo, f0 = oracle.edm_compute_dfdu(cfg, z, 1e-2)
        z = z + np.linalg.solve(Jo, -f0); f, _ = oracle.edm_compute_f(cfg, z, aux=False); hist.append(np.linalg.norm(f))
    assert len(hist) == len(res[1][2])
    assert np.allclose(res[1][1], z, rtol=0, atol=1e-8)        # FD Jacobians amplify 1e-13 by 1/eps per step
    assert np.allclose(res[1][2], hist, rtol=1e-5, atol=1e-9)
    assert np.max(np.abs(res[1][3] - Jo)) < 1e-7 * np.max(np.abs(Jo))


@pytest.mark.gpu
def test_edm_stability_through_the_reference_interfaces(host, oracle):
    R, N, n = 4, 1024, 3
    u = np.array([0.33144403, 0.69563678, 1.36572108])
    out = []
    for mode in (0, 1):
        re = np.zeros(n); im = np.zeros(n)
        cnt = host.b200_host_edm_stability(C.c_double(BETA), R, N, dp(u), n, C.c_double(1e-2), mode, dp(re), dp(im))
        assert cnt >= 0, host.b200_host_last_error()
        out.append((cnt, re.copy(), im.copy()))
    assert out[0][0] == out[1][0] and np.array_equal(out[0][1], out[1][1])
    Jo, _ = oracle.edm_compute_dfdu(oracle.edm_cfg(R=1, N=N), u, 1e-2)
    lam = np.linalg.eigvals(Jo + np.eye(3))
    assert out[1][0] == int(np.sum(np.abs(lam) > 1.0)) == 1
    assert np.allclose(np.sort(out[1][1]), np.sort(lam.real), atol=1e-6)


@pytest.mark.gpu
def test_continuation_driver_runs(host):
    """examples/driver.cpp — the reference experiment plus the beta-continuation loop the reference
    leaves commented out (Driver.cu:86-112): Newton converges at each beta and the travelling wave has
    exactly one unstable direction (the spectrum pinned in tests/test_oracle_edm.py)."""
    exe = os.path.join(LIBDIR, "driver_b200")
    out = subprocess.run([exe, "2", "16", "1024", "0.1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("beta =")]
    assert len(lines) == 2
    assert all("unstable eigenvalues = 1" in l for l in lines), lines
    assert out.stdout.count("The method converged after") == 2


@pytest.mark.gpu
def test_continuation_trajectory_matches_the_oracle(host, oracle):
    """The beta-continuation of Driver.cu:86-112 (solve -> count unstable eigenvalues -> beta += 0.1 -> reuse the
    solution), run by examples/driver.cpp through NewtonSolver / Stability / EventDrivenMapB200, against the same
    loop on the CPU oracle: every fixed point to 1e-8 and every eigenvalue count."""
    exe = os.path.join(LIBDIR, "driver_b200")
    steps = 3      # (at the fourth step, beta = 13.359, Newton from the previous solution diverges — in the oracle too)
    out = subprocess.run([exe, str(steps), "4", "1024", "0.1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    got = []
    for l in out.stdout.splitlines():
        if l.startswith("beta ="):
            tok = l.split()
            got.append((float(tok[2]), np.array([float(tok[5]), float(tok[6]), float(tok[7])]), int(tok[tok.index("eigenvalues") + 2])))
    assert len(got) == steps
    beta = float(np.float32(13.0589)); z = Z_DRIVER.copy()
    for k in range(steps):
        b32 = float(np.float32(beta))                       # SetParameters(0, (float) beta), Driver.cu:108
        cfg = oracle.edm_cfg(R=1, N=1024, beta=b32 if k else beta)
        f, _ = oracle.edm_compute_f(cfg, z, aux=False); it = 0
        while np.linalg.norm(f) > 1e-4 and it < 10:
            J, f0 = oracle.edm_compute_dfdu(cfg, z, 1e-2)
            z = z + np.linalg.solve(J, -f0); f, _ = oracle.edm_compute_f(cfg, z, aux=False); it += 1
        assert np.linalg.norm(f) <= 1e-4
        J, _ = oracle.edm_compute_dfdu(cfg, z, 1e-2)
        unstable = int(np.sum(np.abs(np.linalg.eigvals(J + np.eye(3))) > 1.0))
        assert abs(got[k][0] - beta) < 1e-9
        assert np.allclose(got[k][1], z, rtol=0, atol=1e-8), (k, got[k][1], z)
        assert got[k][2] == unstable
        beta += 0.1


# ---- the Armadillo-facing interpolation adaptor (host/InterpB200.hpp) ----
def test_interp_adaptor_rejects_what_it_does_not_offer(host):
    """No GPU needed: argument checks of b200::interp1 happen before any device call
    (arma::interp1 raises logic_error for unknown methods and mismatched X / Y too)."""
    x = np.linspace(0, 1, 8); y = x ** 2; xi = np.array([0.5]); yi = np.zeros(1)
    rc = host.b200_host_interp1(dp(x), dp(y), 8, dp(xi), 1, dp(yi), C.c_double(0.0), b"nearest", 0, None)
    assert rc == -1 and b"unsupported interpolation type" in host.b200_host_last_error()
    for name in ("b200_host_interp1", "b200_host_interp2"):
        assert hasattr(host, name)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_interp1_adaptor_matches_oracle(host, oracle, mode):
    rng = np.random.default_rng(31)
    x = np.cumsum(0.5 + rng.random(3000)); y = np.sin(x); y2 = np.cos(x)
    xi = rng.uniform(x[0] - 1, x[-1] + 1, 20001); xi[:3] = [x[0], x[-1], np.nan]
    yi = np.empty_like(xi)
    for method in (b"linear", b"*linear"):
        rc = host.b200_host_interp1(dp(x), dp(y), x.size, dp(xi), xi.size, dp(yi), C.c_double(-2.5), method, mode,
                                    dp(y2) if mode == 1 else None)
        assert rc == 0, host.b200_host_last_error()
        ref = oracle.interp1(x, y2 if mode == 1 else y, xi, extrap=-2.5, want_idx=False)
        assert np.array_equal(np.isnan(yi), np.isnan(ref)) and np.array_equal(yi[~np.isnan(yi)], ref[~np.isnan(ref)])
    xs = x.copy(); xs[5] = xs[4]                                       # not strictly ascending: reported, not sorted
    assert host.b200_host_interp1(dp(xs), dp(y), x.size, dp(xi), xi.size, dp(yi), C.c_double(0.0), b"linear", 0, None) == -1
    assert b"ascending" in host.b200_host_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_interp2_adaptor_matches_oracle(host, oracle, mode):
    rng = np.random.default_rng(32)
    x = np.linspace(0, 1, 70); y = np.cumsum(0.5 + rng.random(50)); z = np.asfortranarray(rng.standard_normal((50, 70)))
    if mode == 2:
        xq = rng.uniform(-0.1, 1.1, 5000); yq = rng.uniform(y[0] - 1, y[-1] + 1, 5000)
        out = np.empty(5000)
        rc = host.b200_host_interp2(dp(x), 70, dp(y), 50, dp(z), dp(xq), 5000, dp(yq), 5000, dp(out), C.c_double(7.0), mode)
        assert rc == 0, host.b200_host_last_error()
        ref = oracle.interp2_scattered(x, y, z, xq, yq, extrap=7.0)
    else:
        xi = np.sort(rng.uniform(-0.1, 1.1, 40)); yi = np.sort(rng.uniform(y[0] - 1, y[-1] + 1, 33))
        out = np.empty((33, 40), order="F")
        rc = host.b200_host_interp2(dp(x), 70, dp(y), 50, dp(z), dp(xi), 40, dp(yi), 33, dp(out), C.c_double(7.0), mode)
        assert rc == 0, host.b200_host_last_error()
        ref = oracle.interp2_grid(x, y, z, xi, yi, extrap=7.0)
    assert out.shape == ref.shape and np.array_equal(out, ref)


@pytest.mark.gpu
def test_interp1_adaptor_fvec(host, oracle):
    rng = np.random.default_rng(33)
    x = np.unique(np.cumsum(0.5 + rng.random(2000)).astype(np.float32)); y = np.sin(x).astype(np.float32)
    xi = rng.uniform(x[0], x[-1], 10001).astype(np.float32)
    yi = np.empty_like(xi)
    assert host.b200_host_interp1_f32(dp(x), dp(y), x.size, dp(xi), xi.size, dp(yi), C.c_float(0.0)) == 0, host.b200_host_last_error()
    assert np.array_equal(yi, oracle.interp1(x, y, xi, extrap=0.0, want_idx=False))


# ---- round 2: the eigen-solve behind arma::eig_gen, and configs 4 / 5 through the C++ classes ----
@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 1000])
def test_eig_gen_backend_matches_numpy(host, n, monkeypatch):
    """arma::eig_gen as Stability.cpp:40,72 calls it: for n >= 256 the shim hands the matrix to
    b200_eig_gen_f64 (cuSOLVER GEEV on the device); same spectrum as numpy (LAPACK dgeev) and as the
    shim's own Hessenberg-QR (B200_SHIM_HOST_EIG=1)."""
    rng = np.random.default_rng(100 + n)
    A = np.asfortranarray(rng.standard_normal((n, n)) / np.sqrt(n) + np.diag(np.linspace(0.2, 1.4, n)))
    lam = np.sort_complex(np.linalg.eigvals(A))
    re = np.zeros(n); im = np.zeros(n); ms = C.c_double()
    for rep in range(2):
        assert host.b200_host_eig_gen(n, dp(A), dp(re), dp(im), C.byref(ms)) == 0, host.b200_host_last_error()
    print(f"eig_gen n={n}: {ms.value:.1f} ms (device backend, second call)")
    got = np.sort_complex(re + 1j * im)
    assert np.allclose(got, lam, rtol=1e-8, atol=1e-8)
    assert int(np.sum(np.abs(got) > 1.0)) == int(np.sum(np.abs(lam) > 1.0))
    if n <= 300:
        monkeypatch.setenv("B200_SHIM_HOST_EIG", "1")
        assert host.b200_host_eig_gen(n, dp(A), dp(re), dp(im), C.byref(ms)) == 0
        assert np.allclose(np.sort_complex(re + 1j * im), lam, rtol=1e-8, atol=1e-8)


def _newton_multi(host, R, N, ndev, mode=1, sigma=0.0):
    n = 3
    sol = np.zeros(n); hist = np.full(11, np.nan); nh = C.c_int(); J = np.zeros((n, n), order="F"); ms = np.zeros(2)
    devs = (C.c_int * max(ndev, 1))(*range(max(ndev, 1)))
    rc = host.b200_host_edm_newton_multi(C.c_double(BETA), R, N, dp(Z_DRIVER), n, C.c_double(1e-4), 10, C.c_double(1e-2),
                                         mode, C.c_double(sigma), ndev, devs, dp(sol), dp(hist), C.byref(nh), dp(J), dp(ms))
    assert rc >= 0, host.b200_host_last_error()
    return rc, sol, hist[:nh.value], J, ms


@pytest.mark.gpu
def test_config4_newton_driver_settings_cpp(host, b200):
    """BASELINE config 4 through the product's own C++ NewtonSolver with the reference driver's settings
    (Driver.cu:28-37: tol 1e-4, <= 10 iterations, eps 1e-2, R = 1000, N = 1024): converges to the fixed point
    pinned in tests/test_oracle_edm.py; with several GPUs in this process (SetDevices -> NCCL all-gather inside
    libb200edm.so) every iterate is bitwise the single-GPU one."""
    rc1, sol1, hist1, J1, ms1 = _newton_multi(host, 1000, 1024, 1)
    assert rc1 == 1
    assert np.allclose(sol1, [0.331444, 0.695637, 1.365721], atol=2e-6) and hist1[-1] < 1e-4
    ndev = b200.device_count()
    if ndev >= 2:
        for sigma in (0.0, 0.3):
            a = _newton_multi(host, 1000, 1024, 1, sigma=sigma)
            b = _newton_multi(host, 1000, 1024, min(ndev, 8), sigma=sigma)
            assert a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])


def _profile_stability(host, R, N, nc, T, u, eps, ndev):
    n = 2 * nc
    ms = np.zeros(3); J = np.zeros((n, n), order="F"); re = np.zeros(n); im = np.zeros(n)
    devs = (C.c_int * max(ndev, 1))(*range(max(ndev, 1)))
    cnt = host.b200_host_profile_stability(C.c_double(BETA), R, N, nc, C.c_double(T), dp(u), C.c_double(eps), ndev, devs,
                                           dp(ms), dp(J), dp(re), dp(im))
    assert cnt > -1000, host.b200_host_last_error()
    return cnt, J, re + 1j * im, ms


@pytest.mark.gpu
def test_config5_profile_stability_cpp(host, b200):
    """BASELINE config 5 (small shape) through Stability::ComputeNumUnstableEigenvalues of the C++ host layer:
    the Jacobian is the Python binding's, bit for bit (columns formed / differenced on the device), the count is
    numpy's on that Jacobian, and several devices give the same bits."""
    nc, R, N, T, eps = 96, 6, 512, 0.5, 1e-3
    u = np.concatenate([0.2 + 0.7 * np.sin(np.linspace(0, np.pi, nc)) ** 2, np.linspace(0.0, 0.4, nc)])
    cnt, J, lam, ms = _profile_stability(host, R, N, nc, T, u, eps, 1)
    m = b200.EventDrivenMap([BETA], R, noNeurons=N)
    m.SetTimeHorizon(T); m.SetProfileMode(nc)
    Jp = m.ComputeDFDU(u, eps)
    assert np.array_equal(J, Jp)
    # the same Jacobian column by column through ComputeF (the callers' own loop, Stability.cpp:95-109)
    f0 = m.ComputeF(u)
    for i in (0, 7, nc, 2 * nc - 1):
        du = u.copy(); du[i] += eps
        assert np.array_equal(J[:, i], (m.ComputeF(du) - f0) * eps ** -1)
    ref = np.linalg.eigvals(J + np.eye(2 * nc))
    assert cnt == int(np.sum(np.abs(ref) > 1.0))
    assert np.allclose(np.sort_complex(lam), np.sort_complex(ref), atol=1e-7)
    ndev = b200.device_count()
    if ndev >= 2:
        cnt2, J2, lam2, ms2 = _profile_stability(host, R, N, nc, T, u, eps, min(ndev, 8))
        assert cnt2 == cnt and np.array_equal(J2, J)


@pytest.mark.gpu
def test_config5_rest_state_known_spectrum_cpp(host, b200):
    """BASELINE config 5 at its full shape (n = 1000 coarse unknowns, N = 1024 neurons) on a state whose answer is
    known in closed form: at rest (v = I below threshold, s = 0) no neuron fires, the map is linear,
        v(T) = v e^-T + I (1 - e^-T) + kappa s,   s(T) = s e^-(beta T),   kappa = e^-T (e^((1-beta) T) - 1) / (1 - beta),
    so with M = restrict o lift (linear interpolation coarse -> fine -> coarse, rows sum to one)
        I + J = [[e^-T M, kappa M], [0, e^-(beta T) M]].
    Checked through Stability::ComputeNumUnstableEigenvalues of the C++ host layer (FD Jacobian on the GPU, eig_gen =
    cuSOLVER GEEV behind the shim): the block relations, the spectrum against the two 500 x 500 blocks, the largest
    eigenvalue e^-T (constant profiles), and zero unstable eigenvalues."""
    nc, N, T, eps = 500, 1024, 1.0, 1e-3
    beta = float(np.float32(13.0589)); I = float(np.float32(0.9))
    u = np.concatenate([np.full(nc, I), np.zeros(nc)])
    cnt, J, lam, ms = _profile_stability(host, 1, N, nc, T, u, eps, 1)
    assert cnt == 0
    A = J + np.eye(2 * nc)
    e1, eb = np.exp(-T), np.exp(-beta * T)
    kappa = e1 * (np.exp((1.0 - beta) * T) - 1.0) / (1.0 - beta)
    M = A[nc:, nc:] / eb
    assert np.allclose(M.sum(axis=1), 1.0, atol=1e-6)                       # interpolation reproduces constants
    assert np.max(np.abs(A[:nc, :nc] - e1 * M)) < 1e-9                      # dv(T)/dv
    assert np.max(np.abs(A[:nc, nc:] - kappa * M)) < 1e-9                   # dv(T)/ds
    assert np.max(np.abs(A[nc:, :nc])) < 1e-9                               # ds(T)/dv = 0
    mu = np.linalg.eigvals(M)
    ref = np.concatenate([e1 * mu, eb * mu])
    assert np.allclose(np.sort(np.abs(lam)), np.sort(np.abs(ref)), atol=1e-8)
    assert abs(np.max(np.abs(lam)) - e1) < 1e-8                             # the constant profile decays like e^-T
    ndev = b200.device_count()
    if ndev >= 2:
        cnt2, J2, lam2, _ = _profile_stability(host, 1, N, nc, T, u, eps, min(ndev, 8))
        assert cnt2 == 0 and np.array_equal(J2, J)


@pytest.mark.gpu
def test_newton_on_the_profile_map_finds_the_rest_state(host, b200):
    """NewtonSolver on the profile map (n = 2 n_coarse unknowns, Jacobian = one batch of evaluations through the
    plug-in).  The travelling wave is not a fixed point of this map in the lab frame (DESIGN section 6); the rest state
    v = I, s = 0 is.  From a smooth sub-threshold perturbation nobody fires, the map is linear and Newton lands on
    the rest state in one step (200 unknowns, Jacobian = 200 evaluations given the residual).  (A perturbation that
    makes neurons fire starts a wave; the event-driven map is then discontinuous in u and Newton from there is a matter
    of luck — the oracle shows both outcomes — so that is not a test.)"""
    nc, N, T = 100, 1024, 0.5
    I = float(np.float32(0.9))
    xs = np.linspace(0.0, 2.0 * np.pi, nc, endpoint=False)
    rest = np.concatenate([np.full(nc, I), np.zeros(nc)])

    def solve(guess, ndev=1):
        sol = np.zeros(2 * nc); hist = np.full(21, np.nan); nh = C.c_int(); ms = np.zeros(1)
        devs = (C.c_int * max(ndev, 1))(*range(max(ndev, 1)))
        rc = host.b200_host_profile_newton(C.c_double(BETA), 2, N, nc, C.c_double(T), dp(guess), C.c_double(1e-9), 20,
                                           C.c_double(1e-4), ndev, devs, dp(sol), dp(hist), C.byref(nh), dp(ms))
        assert rc >= 0, host.b200_host_last_error()
        return rc, sol, hist[:nh.value]

    g = rest + np.concatenate([0.04 * np.sin(xs), 0.01 * (1 + np.cos(2 * xs))])          # max v = 0.94 < vth
    rc, sol, hist = solve(g)
    assert rc == 1 and len(hist) == 2 and hist[0] > 1e-2 and hist[-1] < 1e-9
    assert np.max(np.abs(sol - rest)) < 1e-9
    if b200.device_count() >= 2:
        rc3, sol3, hist3 = solve(g, min(b200.device_count(), 4))
        assert rc3 == rc and np.array_equal(sol3, sol) and np.array_equal(hist3, hist)
