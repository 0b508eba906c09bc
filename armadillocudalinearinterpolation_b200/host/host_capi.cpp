// host_capi.cpp — a few C entry points over the C++ host layer so that the test-suite (pytest,
// ctypes) can drive NewtonSolver / Stability / EventDrivenMapB200 exactly as a C++ user would.
#include <chrono>
#include <cmath>
#include <cstring>
#include <sstream>
#include "EventDrivenMapB200.hpp"
#include "InterpB200.hpp"
#include "NewtonSolver.hpp"
#include "Stability.hpp"

namespace {
thread_local std::string g_err;

// Analytic test problems (no GPU): F_i(u) = u_i^2 - (i+2) + 0.1 * u_{(i+1) mod n}
class QuadraticProblem : public AbstractNonlinearProblem, public AbstractNonlinearProblemJacobian {
 public:
  int calls = 0, post = 0;
  void ComputeF(const arma::vec& u, arma::vec& f) {
    const arma::uword n = u.n_elem;
    f.set_size(n);
    for (arma::uword i = 0; i < n; ++i) f(i) = u(i) * u(i) - double(i + 2) + 0.1 * u((i + 1) % n);
    ++calls;
  }
  void PostProcess() { ++post; }
  void ComputeDFDU(const arma::vec& u, arma::mat& J) {
    const arma::uword n = u.n_elem;
    J.zeros(n, n);
    for (arma::uword i = 0; i < n; ++i) { J(i, i) += 2.0 * u(i); J(i, (i + 1) % n) += 0.1; }
  }
};

// the same problem offering F and dF/dU in one call (AbstractNonlinearProblemFused): `fused` counts those calls
class QuadraticProblemFused : public QuadraticProblem, public AbstractNonlinearProblemFused {
 public:
  int fused = 0, given = 0;
  bool oneBatch = true;
  void ComputeFAndDFDU(const arma::vec& u, arma::vec& f, arma::mat& J) {
    QuadraticProblem::ComputeF(u, f); --calls;
    QuadraticProblem::ComputeDFDU(u, J);
    ++fused;
  }
  void ComputeDFDUGivenF(const arma::vec& u, const arma::vec& f, arma::mat& J) {
    (void)f;
    QuadraticProblem::ComputeDFDU(u, J);
    ++given;
  }
  bool PrefersOneBatchPerIterate() const { return oneBatch; }
};

// Linear map problem F(u) = A u - u with user matrix A (for the Stability tests)
class LinearProblem : public AbstractNonlinearProblem {
 public:
  arma::mat A;
  void ComputeF(const arma::vec& u, arma::vec& f) { f = A * u - u; }
};
}  // namespace

extern "C" {

const char* b200_host_last_error() { return g_err.c_str(); }

// Newton on the analytic problem.  use_jacobian: 0 = solver's finite differences, 1 = analytic, 2 / 3 = analytic through
// AbstractNonlinearProblemFused, one batch per iterate / Jacobian given the residual (f_calls then = plain ComputeF
// calls + 1000 * fused calls + 1000000 * given-F calls).
// out: solution[n], history[max_it+1] (NaN padded), returns iterations*4 + converged*2 + post_called
int b200_host_newton_quadratic(int n, const double* guess, double tol, int max_it, double eps, double damping,
                               int use_jacobian, double* solution, double* history, int* n_history,
                               int* f_calls, double* jac_out) {
  try {
    QuadraticProblemFused prob_fused;
    QuadraticProblem prob_plain;
    prob_fused.oneBatch = use_jacobian == 2;
    QuadraticProblem& prob = use_jacobian >= 2 ? static_cast<QuadraticProblem&>(prob_fused) : prob_plain;
    arma::vec g(n), sol(n), hist;
    for (int i = 0; i < n; ++i) g(i) = guess[i];
    NewtonSolver::ParameterList pars;
    pars.printOutput = false;
    NewtonSolver* solver = use_jacobian >= 2 ? new NewtonSolver(&prob_fused, &prob_fused, &g, &pars)
                         : use_jacobian ? new NewtonSolver(&prob, &prob, &g, &pars) : new NewtonSolver(&prob, &g, &pars);
    // edits after construction must apply (Driver.cu:37)
    pars.tolerance = tol; pars.maxIterations = max_it; pars.finiteDifferenceEpsilon = eps; pars.damping = damping;
    AbstractNonlinearSolver::ExitFlagType flag;
    arma::mat J(n, n);
    solver->Solve(sol, hist, flag, jac_out ? &J : NULL);
    delete solver;
    for (int i = 0; i < n; ++i) solution[i] = sol(i);
    *n_history = (int)hist.n_elem;
    for (arma::uword i = 0; i < hist.n_elem; ++i) history[i] = hist(i);
    *f_calls = prob.calls + 1000 * prob_fused.fused + 1000000 * prob_fused.given;
    if (jac_out) std::memcpy(jac_out, J.memptr(), sizeof(double) * n * n);
    return ((int)hist.n_elem - 1) * 4 + (flag == AbstractNonlinearSolver::ExitFlagType::converged ? 2 : 0) + (prob.post == 1 ? 1 : 0);
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Stability of the linear map u -> A u given as F(u) = A u - u.  type: 0 flow, 1 map, 2 equationFree.
int b200_host_stability_linear(int n, const double* A_colmajor, int type, double eps, int via_matrix,
                               double* eig_re, double* eig_im) {
  try {
    LinearProblem prob;
    prob.A.set_size(n, n);
    std::memcpy(prob.A.memptr(), A_colmajor, sizeof(double) * n * n);
    Stability::ProblemType t = type == 0 ? Stability::ProblemType::flow : type == 1 ? Stability::ProblemType::map : Stability::ProblemType::equationFree;
    Stability st(t, &prob);
    st.SetFiniteDifferenceEpsilon(eps);
    arma::vec u(n);
    for (int i = 0; i < n; ++i) u(i) = 0.1 * (i + 1);
    if (eig_re) {
      arma::cx_vec w = via_matrix ? arma::eig_gen(prob.A) : st.ComputeEigenvalues(u);
      for (int i = 0; i < n; ++i) { eig_re[i] = w(i).real(); eig_im[i] = w(i).imag(); }
    }
    return via_matrix ? st.ComputeNumUnstableEigenvalues(prob.A) : st.ComputeNumUnstableEigenvalues(u);
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

int b200_host_solve(int n, const double* A_colmajor, const double* b, double* x) {
  try {
    arma::mat A(n, n);
    std::memcpy(A.memptr(), A_colmajor, sizeof(double) * n * n);
    arma::vec bb(n), xx;
    for (int i = 0; i < n; ++i) bb(i) = b[i];
    if (!arma::solve(xx, A, bb)) return 1;
    for (int i = 0; i < n; ++i) x[i] = xx(i);
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// ---- GPU: the drop-in class driven by the host solvers (needs a B200) ----
// mode 0: NewtonSolver 3-arg ctor (its own sequential FD loop over ComputeF)
// mode 1: NewtonSolver 4-arg ctor (EventDrivenMapB200::ComputeDFDU, one batched launch)
int b200_host_edm_newton(double beta, unsigned R, unsigned N, const double* guess, int n, double tol, int max_it,
                         double eps, int mode, double sigma, double* solution, double* history, int* n_history,
                         double* jac_out) {
  try {
    arma::vec p(1);
    p(0) = beta;
    EventDrivenMapB200 map(&p, R, N, (unsigned)n);
    map.SetPrintOutput(false);
    map.SetFiniteDifferenceEpsilon(eps);
    if (sigma > 0) map.SetParameterStdDev((float)sigma);
    arma::vec g(n), sol(n), hist;
    for (int i = 0; i < n; ++i) g(i) = guess[i];
    NewtonSolver::ParameterList pars;
    pars.tolerance = tol; pars.maxIterations = max_it; pars.printOutput = false; pars.finiteDifferenceEpsilon = eps;
    NewtonSolver* solver = mode ? new NewtonSolver(&map, &map, &g, &pars) : new NewtonSolver(&map, &g, &pars);
    if (mode == 3) solver->SetFusedEvaluation(false);   // plug-in Jacobian with the reference's call sequence (F, then dF/dU)
    AbstractNonlinearSolver::ExitFlagType flag;
    arma::mat J(n, n);
    solver->Solve(sol, hist, flag, &J);
    delete solver;
    for (int i = 0; i < n; ++i) solution[i] = sol(i);
    *n_history = (int)hist.n_elem;
    for (arma::uword i = 0; i < hist.n_elem; ++i) history[i] = hist(i);
    if (jac_out) std::memcpy(jac_out, J.memptr(), sizeof(double) * n * n);
    return flag == AbstractNonlinearSolver::ExitFlagType::converged ? 1 : 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Stability (equationFree) of the map at u: number of unstable eigenvalues + the spectrum of I + J
int b200_host_edm_stability(double beta, unsigned R, unsigned N, const double* u_in, int n, double eps, int mode,
                            double* eig_re, double* eig_im) {
  try {
    arma::vec p(1);
    p(0) = beta;
    EventDrivenMapB200 map(&p, R, N, (unsigned)n);
    map.SetPrintOutput(false);
    map.SetFiniteDifferenceEpsilon(eps);
    arma::vec u(n);
    for (int i = 0; i < n; ++i) u(i) = u_in[i];
    Stability st = mode ? Stability(Stability::ProblemType::equationFree, &map, &map)
                        : Stability(Stability::ProblemType::equationFree, &map);
    st.SetFiniteDifferenceEpsilon(eps);
    arma::cx_vec w = st.ComputeEigenvalues(u);
    for (int i = 0; i < n; ++i) { eig_re[i] = w(i).real(); eig_im[i] = w(i).imag(); }
    return st.ComputeNumUnstableEigenvalues(u);
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}


// ---- BASELINE config 4: NewtonSolver with the reference driver's settings (Driver.cu:28-37,71) on the drop-in
// map spread over `ndev` devices of this process (EventDrivenMapB200::SetDevices -> NCCL all-gather inside the
// C-ABI).  mode as above.  ms_out[0] = wall time of Solve(), ms_out[1] = of one extra ComputeDFDU at the solution.
int b200_host_edm_newton_multi(double beta, unsigned R, unsigned N, const double* guess, int n, double tol, int max_it,
                               double eps, int mode, double sigma, int ndev, const int* devs, double* solution,
                               double* history, int* n_history, double* jac_out, double* ms_out) {
  try {
    arma::vec p(1);
    p(0) = beta;
    EventDrivenMapB200 map(&p, R, N, (unsigned)n);
    map.SetPrintOutput(false);
    map.SetFiniteDifferenceEpsilon(eps);
    if (sigma > 0) map.SetParameterStdDev((float)sigma);
    if (ndev > 1) map.SetDevices(devs, (unsigned)ndev);
    arma::vec g(n), sol(n), hist;
    for (int i = 0; i < n; ++i) g(i) = guess[i];
    NewtonSolver::ParameterList pars;
    pars.tolerance = tol; pars.maxIterations = max_it; pars.printOutput = false; pars.damping = 1.0;
    NewtonSolver* solver = mode ? new NewtonSolver(&map, &map, &g, &pars) : new NewtonSolver(&map, &g, &pars);
    if (mode == 3) solver->SetFusedEvaluation(false);
    pars.finiteDifferenceEpsilon = eps;      // set after construction, as Driver.cu:37
    AbstractNonlinearSolver::ExitFlagType flag;
    arma::mat J(n, n);
    { arma::vec warm(n); map.ComputeF(g, warm); }          // context / allocations outside the timed region
    auto t0 = std::chrono::steady_clock::now();
    solver->Solve(sol, hist, flag, &J);
    auto t1 = std::chrono::steady_clock::now();
    arma::mat J2(n, n);
    map.ComputeDFDU(sol, J2);
    auto t2 = std::chrono::steady_clock::now();
    delete solver;
    if (ms_out) {
      ms_out[0] = std::chrono::duration<double, std::milli>(t1 - t0).count();
      ms_out[1] = std::chrono::duration<double, std::milli>(t2 - t1).count();
    }
    for (int i = 0; i < n; ++i) solution[i] = sol(i);
    *n_history = (int)hist.n_elem;
    for (arma::uword i = 0; i < hist.n_elem; ++i) history[i] = hist(i);
    if (jac_out) std::memcpy(jac_out, J.memptr(), sizeof(double) * n * n);
    return flag == AbstractNonlinearSolver::ExitFlagType::converged ? 1 : 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// ---- BASELINE config 5: Stability::ComputeNumUnstableEigenvalues (Stability.cpp:22-36) of the profile map
// (n = 2 n_coarse) through the C++ classes, Jacobian via the plug-in (Stability.cpp:59-62) over `ndev` devices,
// eigenvalues via arma::eig_gen.  ms_out[0] = the whole call (Jacobian + eigenvalues), ms_out[1] = a Jacobian
// alone, ms_out[2] = eig_gen alone on that Jacobian.  jac_out (n x n, nullable) receives the Jacobian.
int b200_host_profile_stability(double beta, unsigned R, unsigned N, unsigned n_coarse, double T, const double* u_in,
                                double eps, int ndev, const int* devs, double* ms_out, double* jac_out,
                                double* eig_re, double* eig_im) {
  try {
    arma::vec p(1);
    p(0) = beta;
    const int n = 2 * (int)n_coarse;
    EventDrivenMapB200 map(&p, R, N, 3);
    map.SetPrintOutput(false);
    map.SetTimeHorizon((float)T);
    map.SetProfileMode(n_coarse);
    map.SetFiniteDifferenceEpsilon(eps);
    if (ndev > 1) map.SetDevices(devs, (unsigned)ndev);
    arma::vec u(n);
    for (int i = 0; i < n; ++i) u(i) = u_in[i];
    Stability st(Stability::ProblemType::equationFree, &map, &map);
    arma::mat J(n, n);
    map.ComputeDFDU(u, J);                                  // warm-up: allocations, NCCL channels
    { arma::mat W = J + arma::mat(n, n, arma::fill::eye); arma::eig_gen(W); }   // ... and the eigen-solver's library, kernels, workspace
    auto t0 = std::chrono::steady_clock::now();
    const int unstable = st.ComputeNumUnstableEigenvalues(u);
    auto t1 = std::chrono::steady_clock::now();
    map.ComputeDFDU(u, J);
    auto t2 = std::chrono::steady_clock::now();
    arma::mat JI = J + arma::mat(n, n, arma::fill::eye);    // Stability.cpp:68-71
    arma::cx_vec w = arma::eig_gen(JI);
    auto t3 = std::chrono::steady_clock::now();
    if (ms_out) {
      ms_out[0] = std::chrono::duration<double, std::milli>(t1 - t0).count();
      ms_out[1] = std::chrono::duration<double, std::milli>(t2 - t1).count();
      ms_out[2] = std::chrono::duration<double, std::milli>(t3 - t2).count();
    }
    if (jac_out) std::memcpy(jac_out, J.memptr(), sizeof(double) * n * n);
    if (eig_re) for (int i = 0; i < n; ++i) { eig_re[i] = w(i).real(); eig_im[i] = w(i).imag(); }
    return unstable;
  } catch (const std::exception& e) { g_err = e.what(); return -1000; }
}

// NewtonSolver on the PROFILE map (n = 2 n_coarse unknowns): u -> a zero of Phi_T(u) - u, Jacobian through the
// plug-in (one batch of n or n + 1 evaluations per iteration, over `ndev` devices).  Returns 1 converged, 0 not,
// -1 error; history[max_it + 1].
int b200_host_profile_newton(double beta, unsigned R, unsigned N, unsigned n_coarse, double T, const double* guess,
                             double tol, int max_it, double eps, int ndev, const int* devs, double* solution,
                             double* history, int* n_history, double* ms_out) {
  try {
    arma::vec p(1);
    p(0) = beta;
    const int n = 2 * (int)n_coarse;
    EventDrivenMapB200 map(&p, R, N, 3);
    map.SetPrintOutput(false);
    map.SetTimeHorizon((float)T);
    map.SetProfileMode(n_coarse);
    map.SetFiniteDifferenceEpsilon(eps);
    if (ndev > 1) map.SetDevices(devs, (unsigned)ndev);
    arma::vec g(n), sol(n), hist;
    for (int i = 0; i < n; ++i) g(i) = guess[i];
    NewtonSolver::ParameterList pars;
    pars.tolerance = tol; pars.maxIterations = max_it; pars.printOutput = false; pars.finiteDifferenceEpsilon = eps;
    NewtonSolver solver(&map, &map, &g, &pars);
    AbstractNonlinearSolver::ExitFlagType flag;
    auto t0 = std::chrono::steady_clock::now();
    solver.Solve(sol, hist, flag);
    auto t1 = std::chrono::steady_clock::now();
    if (ms_out) ms_out[0] = std::chrono::duration<double, std::milli>(t1 - t0).count();
    for (int i = 0; i < n; ++i) solution[i] = sol(i);
    *n_history = (int)hist.n_elem;
    for (arma::uword i = 0; i < hist.n_elem; ++i) history[i] = hist(i);
    return flag == AbstractNonlinearSolver::ExitFlagType::converged ? 1 : 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// arma::eig_gen as the host layer sees it (cuSOLVER behind the shim for n >= 256, own QR below / on request)
int b200_host_eig_gen(int n, const double* A_colmajor, double* eig_re, double* eig_im, double* ms_out) {
  try {
    arma::mat A(n, n);
    std::memcpy(A.memptr(), A_colmajor, sizeof(double) * n * n);
    auto t0 = std::chrono::steady_clock::now();
    arma::cx_vec w = arma::eig_gen(A);
    auto t1 = std::chrono::steady_clock::now();
    if (ms_out) *ms_out = std::chrono::duration<double, std::milli>(t1 - t0).count();
    for (int i = 0; i < n; ++i) { eig_re[i] = w(i).real(); eig_im[i] = w(i).imag(); }
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}


// ---- the Armadillo-facing interpolation adaptor (InterpB200.hpp), driven like a C++ user would ----
// mode 0: b200::interp1 (one-shot), 1: Interp1Plan + SetValues(y2) (y2 may be NULL)
int b200_host_interp1(const double* x, const double* y, int n, const double* xi, int ni, double* yi, double extrap,
                      const char* method, int mode, const double* y2) {
  try {
    arma::vec X(n), Y(n), XI(ni), YI;
    for (int i = 0; i < n; ++i) { X(i) = x[i]; Y(i) = y[i]; }
    for (int i = 0; i < ni; ++i) XI(i) = xi[i];
    if (mode == 0) b200::interp1(X, Y, XI, YI, method, extrap);
    else {
      b200::Interp1Plan plan(X, Y);
      if (y2) { arma::vec Y2(n); for (int i = 0; i < n; ++i) Y2(i) = y2[i]; plan.SetValues(Y2); }
      plan(XI, YI, extrap);
    }
    if ((int)YI.n_elem != ni) { g_err = "YI has the wrong size"; return -1; }
    for (int i = 0; i < ni; ++i) yi[i] = YI(i);
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Interp1Plan(X, Y).Grad with nx knots and ny values (different lengths are rejected by the plan): yi, dydx get ni entries
int b200_host_interp1_grad(const double* x, int nx, const double* y, int ny, const double* xi, int ni, double* yi,
                           double* dydx, double extrap) {
  try {
    arma::vec X(nx), Y(ny), XI(ni), YI, DY;
    for (int i = 0; i < nx; ++i) X(i) = x[i];
    for (int i = 0; i < ny; ++i) Y(i) = y[i];
    for (int i = 0; i < ni; ++i) XI(i) = xi[i];
    b200::Interp1Plan plan(X, Y);
    plan.Grad(XI, YI, DY, extrap);
    if ((int)YI.n_elem != ni || (int)DY.n_elem != ni) { g_err = "YI or DYDX has the wrong size"; return -1; }
    for (int i = 0; i < ni; ++i) { yi[i] = YI(i); dydx[i] = DY(i); }
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Interp1Plan(X, Y).Adjoint with ni entries of XI and ng of G: dy (n values); returns -1 with the exception's text when
// the lengths differ or dY comes back with another size
int b200_host_interp1_adjoint(const double* x, const double* y, int n, const double* xi, int ni, const double* g, int ng,
                              double* dy) {
  try {
    arma::vec X(n), Y(n), XI(ni), G(ng), dY;
    for (int i = 0; i < n; ++i) { X(i) = x[i]; Y(i) = y[i]; }
    for (int i = 0; i < ni; ++i) XI(i) = xi[i];
    for (int i = 0; i < ng; ++i) G(i) = g[i];
    b200::Interp1Plan plan(X, Y);
    plan.Adjoint(XI, G, dY);
    if ((int)dY.n_elem != n) { g_err = "dY has the wrong size"; return -1; }
    for (int i = 0; i < n; ++i) dy[i] = dY(i);
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// arma::fvec overload of b200::interp1
int b200_host_interp1_f32(const float* x, const float* y, int n, const float* xi, int ni, float* yi, float extrap) {
  try {
    arma::fvec X(n), Y(n), XI(ni), YI;
    for (int i = 0; i < n; ++i) { X(i) = x[i]; Y(i) = y[i]; }
    for (int i = 0; i < ni; ++i) XI(i) = xi[i];
    b200::interp1(X, Y, XI, YI, "*linear", extrap);
    for (int i = 0; i < ni; ++i) yi[i] = YI(i);
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// mode 0: b200::interp2 (tensor grid, zi is nyi x nxi column-major), 1: Interp2Plan::Grid,
// 2: Interp2Plan::Scattered (nxi == nyi queries, zi has nxi entries)
int b200_host_interp2(const double* x, int nx, const double* y, int ny, const double* z_colmajor, const double* xi, int nxi,
                      const double* yi, int nyi, double* zi, double extrap, int mode) {
  try {
    arma::vec X(nx), Y(ny), XI(nxi), YI(nyi);
    arma::mat Z(ny, nx);
    for (int i = 0; i < nx; ++i) X(i) = x[i];
    for (int i = 0; i < ny; ++i) Y(i) = y[i];
    for (int i = 0; i < nx * ny; ++i) Z.memptr()[i] = z_colmajor[i];
    for (int i = 0; i < nxi; ++i) XI(i) = xi[i];
    for (int i = 0; i < nyi; ++i) YI(i) = yi[i];
    if (mode == 2) {
      arma::vec ZQ;
      b200::Interp2Plan plan(X, Y, Z);
      plan.Scattered(XI, YI, ZQ, extrap);
      for (int i = 0; i < nxi; ++i) zi[i] = ZQ(i);
      return 0;
    }
    arma::mat ZI;
    if (mode == 0) b200::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap);
    else { b200::Interp2Plan plan(X, Y, Z); plan.Grid(XI, YI, ZI, extrap); }
    if ((int)ZI.n_rows != nyi || (int)ZI.n_cols != nxi) { g_err = "ZI has the wrong shape"; return -1; }
    for (int i = 0; i < nxi * nyi; ++i) zi[i] = ZI.memptr()[i];
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Interp2Plan from Z1 (ny x nx), then SetValues with Z2 (z2_rows x z2_cols, column-major), then Scattered at nq
// points (xq[k], yq[k]) -> zq[k]
int b200_host_interp2_set_values(const double* x, int nx, const double* y, int ny, const double* z1_colmajor,
                                 const double* z2_colmajor, int z2_rows, int z2_cols, const double* xq,
                                 const double* yq, int nq, double* zq, double extrap) {
  try {
    arma::vec X(nx), Y(ny), XQ(nq), YQ(nq), ZQ;
    arma::mat Z1(ny, nx), Z2(z2_rows, z2_cols);
    for (int i = 0; i < nx; ++i) X(i) = x[i];
    for (int i = 0; i < ny; ++i) Y(i) = y[i];
    for (int i = 0; i < nx * ny; ++i) Z1.memptr()[i] = z1_colmajor[i];
    for (int i = 0; i < z2_rows * z2_cols; ++i) Z2.memptr()[i] = z2_colmajor[i];
    for (int i = 0; i < nq; ++i) { XQ(i) = xq[i]; YQ(i) = yq[i]; }
    b200::Interp2Plan plan(X, Y, Z1);
    plan.SetValues(Z2);
    plan.Scattered(XQ, YQ, ZQ, extrap);
    for (int i = 0; i < nq; ++i) zq[i] = ZQ(i);
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Interp2Plan(X, Y, Z).ScatteredGrad at nxq x-queries and nyq y-queries (different lengths are rejected):
// zq, dzdx, dzdy get nxq entries
int b200_host_interp2_scattered_grad(const double* x, int nx, const double* y, int ny, const double* z_colmajor,
                                     const double* xq, int nxq, const double* yq, int nyq, double* zq, double* dzdx,
                                     double* dzdy, double extrap) {
  try {
    arma::vec X(nx), Y(ny), XQ(nxq), YQ(nyq), ZQ, DX, DY;
    arma::mat Z(ny, nx);
    for (int i = 0; i < nx; ++i) X(i) = x[i];
    for (int i = 0; i < ny; ++i) Y(i) = y[i];
    for (int i = 0; i < nx * ny; ++i) Z.memptr()[i] = z_colmajor[i];
    for (int i = 0; i < nxq; ++i) XQ(i) = xq[i];
    for (int i = 0; i < nyq; ++i) YQ(i) = yq[i];
    b200::Interp2Plan plan(X, Y, Z);
    plan.ScatteredGrad(XQ, YQ, ZQ, DX, DY, extrap);
    for (int i = 0; i < nxq; ++i) { zq[i] = ZQ(i); dzdx[i] = DX(i); dzdy[i] = DY(i); }
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// Interp2Plan(X, Y, Z).ScatteredAdjoint with nxq, nyq, ng entries of XQ, YQ, G: dz (column-major ny x nx); returns -1 with
// the exception's text when the lengths differ or dZ comes back with another shape
int b200_host_interp2_scattered_adjoint(const double* x, int nx, const double* y, int ny, const double* z_colmajor,
                                        const double* xq, int nxq, const double* yq, int nyq, const double* g, int ng,
                                        double* dz) {
  try {
    arma::vec X(nx), Y(ny), XQ(nxq), YQ(nyq), G(ng);
    arma::mat Z(ny, nx), dZ;
    for (int i = 0; i < nx; ++i) X(i) = x[i];
    for (int i = 0; i < ny; ++i) Y(i) = y[i];
    for (int i = 0; i < nx * ny; ++i) Z.memptr()[i] = z_colmajor[i];
    for (int i = 0; i < nxq; ++i) XQ(i) = xq[i];
    for (int i = 0; i < nyq; ++i) YQ(i) = yq[i];
    for (int i = 0; i < ng; ++i) G(i) = g[i];
    b200::Interp2Plan plan(X, Y, Z);
    plan.ScatteredAdjoint(XQ, YQ, G, dZ);
    if ((int)dZ.n_rows != ny || (int)dZ.n_cols != nx) { g_err = "dZ has the wrong shape"; return -1; }
    for (int i = 0; i < nx * ny; ++i) dz[i] = dZ.memptr()[i];
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

}  // extern "C"
