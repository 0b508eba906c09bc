"""The pin against the REAL reference.

tests/golden/ref_b200.npz holds raw outputs of the UNMODIFIED reference (EventDrivenMap.cu, NewtonSolver.cpp,
Stability.cpp compiled for sm_100a by oracle/ref_build/Makefile, run on a B200 by tools/make_ref_golden.py;
report: profiles/r2_reference_run_on_b200.txt).  The reference's device arithmetic is FP32 and it carries the
accept[0] quirk (SURVEY Q1), so:

  * CPU tests (no GPU): the oracle in its FP32 / Q1 mode reproduces the reference's integer outputs exactly
    (initial, last and crossed front cells, accept flags) and its floats to FP32 noise (CUDA expf/powf vs glibc);
    the oracle-side Newton iteration reproduces the reference NewtonSolver's residual history and fixed point.
  * GPU tests: the product's FP32 compatibility mode does the same against the same vectors, and against the
    reference run live on this box (oracle/_ref present) at points that are not in the fixture.

The FP64 product path is then tied to the FP64 oracle (tests/test_edm_gpu.py, 1e-10), and the FP64 oracle to this
FP32 one by sharing every line of oracle/edm_oracle_impl.inc (one template, two arithmetic types).
Recorded deviations of the reference itself (not reproduced by default): Q1 accept[0] bias (quirk flag reproduces
it); the heterogeneous ensemble differs between successive ComputeF calls of one reference object although
ResetSeed() re-applies the seed (the cuRAND offset keeps advancing) — the fixture's sigma > 0 case therefore uses
the ensemble read back from the device.
"""
import os

import numpy as np
import pytest

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_b200.npz"))
CASES = ["A_default_1024", "B_default_512", "C_offguess_1024", "D_sigma05_1024", "E_T2_768"]
BETA = float(np.float32(13.0589))
GUESS = np.array([np.float32(0.3310), np.float32(0.6914), np.float32(1.3557)], np.float64)
FTOL = 2e-5     # FP32 map outputs: CUDA expf/powf vs glibc differ in the last ulp, the event loop amplifies it


def case_cfg(tag):
    beta, R, N, T, sigma, seed = G[f"{tag}_cfg"]
    return float(beta), int(R), int(N), float(T), float(sigma), int(seed)


def mean_of(tag):
    # for the heterogeneous case the arrays are the replay's (the ensemble that was read back)
    return G[f"{tag}_mean_replay"] if case_cfg(tag)[4] > 0 else G[f"{tag}_mean"]


@pytest.mark.parametrize("tag", CASES)
def test_oracle_fp32_reproduces_the_reference_run(oracle, tag):
    beta, R, N, T, sigma, seed = case_cfg(tag)
    z = G[f"{tag}_z"]
    cfg = oracle.edm_cfg(R=R, N=N, beta=beta, sigma=sigma, seed=seed, precision=1, quirks=1, time_horizon=T,
                         beta_ext=(G[f"{tag}_beta"].astype(np.float64) if sigma > 0 else None))
    f, a = oracle.edm_compute_f(cfg, z, nthreads=8)
    assert np.array_equal(a["init_index"], G[f"{tag}_init_index"])                      # EventDrivenMap.cu:361-376
    assert np.array_equal(a["coupling"].astype(np.float32), G[f"{tag}_coupling"])      # :111-129, bit for bit
    lv, ls = G[f"{tag}_lift_v"].astype(np.float64), G[f"{tag}_lift_s"].astype(np.float64)
    assert np.array_equal(np.isnan(lv), np.isnan(a["lift_v"]))                         # Q8: same FP32 overflow NaNs
    ok = ~np.isnan(lv)
    assert np.max(np.abs(lv - a["lift_v"])[ok]) < 5e-6 and np.nanmax(np.abs(ls - a["lift_s"])) < 5e-6   # :505-542
    assert np.array_equal(a["last_index"].T, G[f"{tag}_last_index"])                   # :575-674, every realisation
    assert np.array_equal(a["crossed_index"].T, G[f"{tag}_crossed_index"])
    assert np.array_equal(a["accept"], G[f"{tag}_accept"])
    assert np.max(np.abs(a["last_time"].T - G[f"{tag}_last_time"])) < FTOL
    assert np.max(np.abs(a["crossed_time"].T - G[f"{tag}_crossed_time"])) < FTOL
    assert np.max(np.abs(a["position"].T - G[f"{tag}_position"])) < FTOL               # :769-785
    assert np.max(np.abs(a["mean"] - mean_of(tag))) < FTOL                             # :787-824 incl. the accept[0] quirk
    if sigma == 0:
        assert np.max(np.abs(f - G[f"{tag}_F"])) < 5 * FTOL                            # :239
    # and the intended semantics differ from the reference by exactly the Q1 factor (R-1)/R when all are accepted
    if sigma == 0 and R > 1:
        cfg0 = oracle.edm_cfg(R=1, N=N, beta=beta, precision=1, quirks=0, time_horizon=T)
        _, a0 = oracle.edm_compute_f(cfg0, z)
        assert np.max(np.abs(a0["mean"] * (R - 1) / R - G[f"{tag}_mean"])) < FTOL


def test_oracle_newton_reproduces_the_reference_newton_solver(oracle):
    """NewtonSolver.cpp:40-161 + FD Jacobian :164-197 of the reference, run on the reference map on a B200 with
    the driver's settings (Driver.cu:28-37) at N = 1024, R = 1000: 7 iterations to 3.5e-5.  The oracle-side
    iteration (FP32 map, Q1 mean of 1000 identical realisations) follows the same residual history."""
    def F(z):
        cfg = oracle.edm_cfg(R=1, N=1024, beta=BETA, precision=1)
        _, a = oracle.edm_compute_f(cfg, z)
        pos = a["position"][0].astype(np.float32)
        mean = (pos * np.float32(999)) / np.float32(1000)          # accept[0] quirk at sigma = 0
        zf = z.astype(np.float32).astype(np.float64)               # EventDrivenMap.cu:172
        return -zf[0] * np.array([0.0, zf[1], zf[2]]) - mean.astype(np.float64) + zf[0] * 5.0
    z = GUESS.copy(); f = F(z); hist = [np.linalg.norm(f)]
    while hist[-1] > 1e-4 and len(hist) <= 10:
        J = np.zeros((3, 3))
        for i in range(3):
            du = z.copy(); du[i] += 1e-2
            J[:, i] = (F(du) - f) * 1e-2 ** -1
        z = z + np.linalg.solve(J, -f); f = F(z); hist.append(np.linalg.norm(f))
    ref_hist = G["N_hist"][G["N_hist"] > 0]
    assert int(G["N_flag"][0]) == 0 and len(ref_hist) == len(hist) == 8
    assert np.allclose(hist, ref_hist, rtol=0.06, atol=2e-6)       # FP32 noise through 7 FD-Newton steps
    assert np.allclose(z, G["N_z"], atol=2e-5)
    assert np.allclose(J, G["N_jac"], atol=2e-3)
    lam = np.linalg.eigvals(G["N_jac"] + np.eye(3))
    assert int(np.sum(np.abs(lam) > 1)) == int(G["N_unstable"][0]) == 1       # Stability.cpp:22-36 on the reference map
    # N = 512 (the state the committed Driver.cu is left in, :68-71): the reference's FD Jacobian goes singular at
    # the third iterate and arma::solve throws — recorded, not a target
    assert int(G["N512_flag"][0]) == -2


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["A_default_1024", "B_default_512", "C_offguess_1024", "E_T2_768"])
def test_product_fp32_mode_reproduces_the_reference_run(b200, tag):
    beta, R, N, T, sigma, seed = case_cfg(tag)
    m = b200.EventDrivenMap([beta], R, noNeurons=N, precision="f32")
    m.SetModel(time_horizon=T, quirks=b200.QUIRK_ACCEPT0_BIAS)
    m.SetDebugFlag(True)
    f = m.ComputeF(G[f"{tag}_z"])
    assert np.array_equal(m.DebugFetch("init_index")[0], G[f"{tag}_init_index"])
    assert np.array_equal(m.DebugFetch("last_index")[0].T, G[f"{tag}_last_index"])
    assert np.array_equal(m.DebugFetch("crossed_index")[0].T, G[f"{tag}_crossed_index"])
    assert np.array_equal(m.DebugFetch("accept")[0], G[f"{tag}_accept"])
    assert np.max(np.abs(m.DebugFetch("position")[0].T - G[f"{tag}_position"])) < FTOL
    assert np.max(np.abs(m.DebugFetch("mean")[0] - G[f"{tag}_mean"])) < FTOL
    assert np.max(np.abs(f - G[f"{tag}_F"])) < 5 * FTOL
    lv = G[f"{tag}_lift_v"].astype(np.float64); mine = m.DebugFetch("lift_v")[0]
    ok = ~np.isnan(lv) & ~np.isnan(mine)
    assert ok.sum() >= np.sum(~np.isnan(lv)) and np.max(np.abs(lv - mine)[ok]) < 5e-6   # (no FP32-overflow NaNs here: Q8)
    assert np.max(np.abs(m.DebugFetch("coupling").astype(np.float32) - G[f"{tag}_coupling"])) < 1e-7
    # the FP64 product path sits within FP32 resolution of the reference once the Q1 factor is applied
    d = b200.EventDrivenMap([beta], R, noNeurons=N)
    d.SetModel(time_horizon=T, quirks=b200.QUIRK_ACCEPT0_BIAS)
    assert np.max(np.abs(d.ComputeF(G[f"{tag}_z"]) - G[f"{tag}_F"])) < 2e-4


@pytest.mark.gpu
def test_product_against_the_reference_live(b200, oracle):
    """The reference itself, run here (oracle/_ref/libedm_ref.so), at points that are not in the fixture:
    same front cells as the product's FP32 mode and the FP32 oracle, F to FP32 noise."""
    from oracle import ref_py
    if not ref_py.available():
        pytest.skip("oracle/_ref was not built (needs B200_REFERENCE_DIR at build time)")
    rng = np.random.default_rng(5)
    for k in range(4):
        z = GUESS * (1 + 0.03 * rng.standard_normal(3))
        N = [1024, 512, 768, 1000][k]; R = 6
        f_ref, a = ref_py.run(z, BETA, R, N)
        m = b200.EventDrivenMap([BETA], R, noNeurons=N, precision="f32")
        m.SetModel(quirks=b200.QUIRK_ACCEPT0_BIAS); m.SetDebugFlag(True)
        f = m.ComputeF(z)
        assert np.array_equal(m.DebugFetch("last_index")[0].T, a["last_index"])
        assert np.array_equal(m.DebugFetch("crossed_index")[0].T, a["crossed_index"])
        assert np.max(np.abs(m.DebugFetch("position")[0].T - a["position"])) < FTOL
        assert np.max(np.abs(f - f_ref)) < 5 * FTOL
        fo, ao = oracle.edm_compute_f(oracle.edm_cfg(R=R, N=N, beta=BETA, precision=1, quirks=1), z)
        assert np.array_equal(ao["last_index"].T, a["last_index"]) and np.max(np.abs(fo - f_ref)) < 5 * FTOL
