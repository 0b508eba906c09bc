/* edm_ref_wrapper.cu — C entry points around the UNMODIFIED reference map, built into
 * oracle/_ref/libedm_ref.so.  TEST INFRASTRUCTURE ONLY (the pin for oracle/ and for the product's
 * FP32 compatibility mode); never linked, imported or called by the product.
 *
 * The reference translation unit is included where it lies (-I$(REF), the reference checkout); nothing
 * of it is copied into this repository.  `private` is lifted so that the device buffers the
 * reference's own Save* dumpers print with "%f" (EventDrivenMap.cu:406-503) can be read back in
 * full precision instead.
 *
 * edm_ref_run() calls the reference's ComputeF (EventDrivenMap.cu:154-240) for F, then replays the
 * same launch sequence stage by stage (the reference's own kernels, same order, same arguments) to
 * capture what ComputeF overwrites on the way (lift output, pre-restriction event times, accept
 * flags before CountRealisationsKernel stores the count into accept[0]); the replayed averages
 * are compared with ComputeF's bit for bit (rc 3 when they differ; both are returned). */
#define private public
#include "EventDrivenMap.cu"
#include "NewtonSolver.hpp"
#include "Stability.hpp"
#undef private
#include <chrono>
#include <cstring>
#include <exception>
#include <vector>

namespace {
template <class T> int fetch(T* dst, const T* dev, size_t n) {
  if (!dst) return 0;
  return cudaMemcpy(dst, dev, n * sizeof(T), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : 1;
}
EventDrivenMap* make_map(double beta, unsigned R, int N, float T, float sigma, unsigned long long seed) {
  arma::vec par(1);
  par[0] = beta;
  EventDrivenMap* m = new EventDrivenMap(&par, R);   /* N = 1024 (EventDrivenMap.cu:70) */
  if (N != 1024) m->SetNoThreads(N);                 /* asserts N < 1024 (EventDrivenMap.cu:285) */
  m->SetTimeHorizon(T);
  m->SetParameterStdDev(sigma);
  m->mSeed = seed;                                   /* the reference seeds from clock() (:104) */
  return m;
}
}  // namespace

extern "C" {

/* One reference evaluation with every intermediate.  z[3] = (c, T2, T3).  Any output may be NULL.
 * Layouts are the reference's: per-front arrays are [m][r] (m*R + r). */
int edm_ref_run(double beta, unsigned R, int N, float T, float sigma, unsigned long long seed,
                const double* z, double* f_out, float* coupling /*[N]*/, unsigned short* init_index /*[3]*/,
                float* lift_v /*[R*N]*/, float* lift_s /*[R*N]*/, unsigned short* last_index /*[3R]*/,
                float* last_time /*[3R]*/, unsigned short* crossed_index /*[3R]*/, float* crossed_time /*[3R]*/,
                unsigned int* accept /*[R]*/, float* position /*[3R]*/, float* mean /*[3]*/,
                float* beta_out /*[R*N]*/, float* position_cf /*[3R] positions left by ComputeF itself*/,
                float* mean_replay /*[3]*/) {
  EventDrivenMap* m = make_map(beta, R, N, T, sigma, seed);
  const size_t RN = (size_t)R * N, R3 = (size_t)R * noSpikes;
  arma::vec Z(noSpikes), f(noSpikes);
  for (int i = 0; i < noSpikes; ++i) Z[i] = z[i];
  m->ComputeF(Z, f);
  if (cudaDeviceSynchronize() != cudaSuccess) return 1;
  if (f_out) for (int i = 0; i < noSpikes; ++i) f_out[i] = f[i];
  float mean_cf[noSpikes];
  int bad = fetch(mean_cf, m->mpDev_U, noSpikes);
  bad |= fetch(position_cf, m->mpDev_lastSpikeTime, R3);

  /* staged replay of EventDrivenMap.cu:162-224 */
  arma::vec U0(noSpikes + 1);
  m->initialSpikeInd(Z);
  m->ZtoU(Z, U0);
  arma::fvec fU = arma::conv_to<arma::fvec>::from(U0);
  bad |= cudaMemcpy(m->mpDev_U, fU.begin(), (noSpikes + 1) * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess;
  m->ResetSeed();
  bad |= curandGenerateNormal(m->mGen, m->mpDev_beta, RN, (*m->mpHost_p)[0], m->mParStdDev) != CURAND_STATUS_SUCCESS;
  LiftKernel<<<R, N>>>(m->mpDev_s, m->mpDev_v, m->mpDev_p, m->mpDev_U, R);
  bad |= cudaDeviceSynchronize() != cudaSuccess;
  if (init_index) memcpy(init_index, m->mpHost_lastSpikeInd, noSpikes * sizeof(unsigned short));
  bad |= fetch(coupling, m->mpDev_w, N);
  bad |= fetch(lift_v, m->mpDev_v, RN);
  bad |= fetch(lift_s, m->mpDev_s, RN);
  bad |= fetch(beta_out, m->mpDev_beta, RN);
  bad |= cudaMemset(m->mpDev_accept, 0, R * sizeof(int)) != cudaSuccess;
  EvolveKernel<<<R, N>>>(m->mpDev_v, m->mpDev_s, m->mpDev_beta, m->mpDev_w, m->mFinalTime, m->mpDev_lastSpikeInd,
                         m->mpDev_lastSpikeTime, m->mpDev_crossedSpikeInd, m->mpDev_crossedSpikeTime,
                         m->mpDev_accept, R);
  bad |= cudaDeviceSynchronize() != cudaSuccess;
  bad |= fetch(last_index, m->mpDev_lastSpikeInd, R3);
  bad |= fetch(last_time, m->mpDev_lastSpikeTime, R3);
  bad |= fetch(crossed_index, m->mpDev_crossedSpikeInd, R3);
  bad |= fetch(crossed_time, m->mpDev_crossedSpikeTime, R3);
  bad |= fetch(accept, m->mpDev_accept, R);
  RestrictKernel<<<noSpikes * R, N>>>(m->mpDev_lastSpikeTime, m->mpDev_lastSpikeInd, m->mpDev_crossedSpikeTime,
                                      m->mpDev_crossedSpikeInd, m->mFinalTime, R);
  bad |= cudaDeviceSynchronize() != cudaSuccess;
  bad |= fetch(position, m->mpDev_lastSpikeTime, R3);
  CountRealisationsKernel<<<(R + N - 1) / N, N>>>(m->mpDev_accept, R);
  realisationReductionKernelBlocks<<<noSpikes, N>>>(m->mpDev_U, m->mpDev_lastSpikeTime, R, m->mpDev_accept);
  bad |= cudaDeviceSynchronize() != cudaSuccess;
  float mean_rp[noSpikes];
  bad |= fetch(mean_rp, m->mpDev_U, noSpikes);
  if (mean) memcpy(mean, mean_cf, sizeof(mean_cf));
  if (mean_replay) memcpy(mean_replay, mean_rp, sizeof(mean_rp));
  /* rc 3 = the replay's averages differ from ComputeF's (the reference's kernels are racy for
   * heterogeneous rings: SURVEY Q2/Q3); outputs are still filled */
  int rc = bad ? 2 : (memcmp(mean_rp, mean_cf, sizeof(mean_cf)) ? 3 : 0);
  delete m;
  return rc;
}

/* The reference's NewtonSolver (NewtonSolver.cpp:40-161, FD Jacobian :164-197) on the reference map
 * with the reference driver's call pattern (Driver.cu:28-37,71).  residual_history has
 * max_iterations+1 entries (never trimmed: NewtonSolver.cpp:134 discards head()).  Returns the
 * exit flag (0 converged, 1 not) or a negative error. */
int edm_ref_newton(double beta, unsigned R, int N, float T, float sigma, unsigned long long seed,
                   const double* z0, double tolerance, int max_iterations, double fd_epsilon, double damping,
                   double* z_out, double* residual_history, double* jacobian_out /*3x3 col-major, last iterate*/) {
  EventDrivenMap* m = make_map(beta, R, N, T, sigma, seed);
  arma::vec guess(noSpikes), sol(noSpikes), hist;
  for (int i = 0; i < noSpikes; ++i) guess[i] = z0[i];
  NewtonSolver::ParameterList pars;
  pars.tolerance = tolerance;
  pars.maxIterations = max_iterations;
  pars.printOutput = false;
  pars.damping = damping;
  NewtonSolver* ns = new NewtonSolver(m, &guess, &pars);
  pars.finiteDifferenceEpsilon = fd_epsilon;             /* set after construction, as Driver.cu:37 */
  AbstractNonlinearSolver::ExitFlagType flag = AbstractNonlinearSolver::ExitFlagType::notConverged;
  arma::mat jac(noSpikes, noSpikes);
  /* the reference lets arma::solve's exception escape (a singular FD Jacobian aborts its driver): caught
   * here so that the history up to that point can still be read; returns -2 */
  bool threw = false;
  try { ns->Solve(sol, hist, flag, &jac); } catch (const std::exception&) { threw = true; }
  for (int i = 0; i < noSpikes; ++i) z_out[i] = sol[i];
  for (int i = 0; i <= max_iterations; ++i) residual_history[i] = (i < (int)hist.n_elem) ? hist[i] : -1.0;
  if (jacobian_out) memcpy(jacobian_out, jac.memptr(), sizeof(double) * noSpikes * noSpikes);
  delete ns;
  delete m;
  if (threw) return -2;
  return flag == AbstractNonlinearSolver::ExitFlagType::converged ? 0 : 1;
}

/* Stability::ComputeNumUnstableEigenvalues (Stability.cpp:22-36) of the reference map at z.
 * mFiniteDifferenceEpsilon has no setter and is never initialised in the reference
 * (Stability.hpp:50); it is set here through the lifted access. */
/* wall time of `reps` calls of the reference's own EventDrivenMap::ComputeF (after `warm` untimed ones), in ms per
 * call; ComputeF ends with a blocking cudaMemcpy (EventDrivenMap.cu:234), so the host clock sees the device work */
double edm_ref_time_compute_f(double beta, unsigned R, int N, float T, float sigma, unsigned long long seed,
                              const double* z, int warm, int reps) {
  EventDrivenMap* m = make_map(beta, R, N, T, sigma, seed);
  arma::vec Z(noSpikes), F(noSpikes);
  for (int i = 0; i < noSpikes; ++i) Z[i] = z[i];
  for (int i = 0; i < warm; ++i) m->ComputeF(Z, F);
  cudaDeviceSynchronize();
  const auto t0 = std::chrono::steady_clock::now();
  for (int i = 0; i < reps; ++i) m->ComputeF(Z, F);
  cudaDeviceSynchronize();
  const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() / (reps > 0 ? reps : 1);
  delete m;
  return ms;
}

int edm_ref_unstable(double beta, unsigned R, int N, float T, float sigma, unsigned long long seed,
                     const double* z, double fd_epsilon) {
  EventDrivenMap* m = make_map(beta, R, N, T, sigma, seed);
  Stability* st = new Stability(Stability::ProblemType::equationFree, m);   /* Driver.cu:46 */
  st->mFiniteDifferenceEpsilon = fd_epsilon;
  arma::vec Z(noSpikes);
  for (int i = 0; i < noSpikes; ++i) Z[i] = z[i];
  int n = -2;
  try { n = st->ComputeNumUnstableEigenvalues(Z); } catch (const std::exception&) {}
  /* ~Stability is declared but never defined in the reference (Stability.hpp:28): leak it, as Driver.cu does */
  delete m;
  return n;
}
}
