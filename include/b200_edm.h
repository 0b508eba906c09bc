/* b200_edm.h — C-ABI of the event-driven coarse time-stepper ("lift -> evolve -> restrict").
 *
 * What it replaces: class EventDrivenMap of the reference, i.e. the host wrapper
 * EventDrivenMap.hpp:11-121 / EventDrivenMap.cu:57-503 and the six kernels
 * EventDrivenMap.cu:378-386, 505-945.  The reference has no C layer (Armadillo and CUDA
 * share one nvcc TU); the functions below are the minimal surface its public methods
 * imply, one entry point per method:
 *
 *   EventDrivenMap(const arma::vec* p, unsigned noReal)  EventDrivenMap.cu:57   -> b200_edm_create
 *   ~EventDrivenMap()                                    EventDrivenMap.cu:131  -> b200_edm_destroy
 *   ComputeF(const arma::vec& Z, arma::vec& f)           EventDrivenMap.cu:154  -> b200_edm_compute_f
 *   SetTimeHorizon(float)                                EventDrivenMap.cu:242  -> b200_edm_set_time_horizon
 *   SetNoRealisations(int)                               EventDrivenMap.cu:249  -> b200_edm_set_no_realisations
 *   SetNoThreads(int)   (= neurons per ring)             EventDrivenMap.cu:282  -> b200_edm_set_no_neurons
 *   SetParameterStdDev(float)                            EventDrivenMap.cu:317  -> b200_edm_set_param_stddev
 *   SetParameters(unsigned parId, float)                 EventDrivenMap.cu:324  -> b200_edm_set_parameter
 *   ResetSeed() / SetNewSeed() / PostProcess()           EventDrivenMap.cu:332-346 -> b200_edm_set_seed / _new_seed
 *   SetDebugFlag(bool) + Save*()                         EventDrivenMap.cu:348,406-503 -> b200_edm_debug_fetch
 *   FD Jacobian column loop of the callers               NewtonSolver.cpp:164-197, Stability.cpp:76-111
 *                                                        -> b200_edm_compute_f_batch / b200_edm_compute_dfdu
 *
 * All vectors crossing the boundary are double (arma::vec) and column-major.
 * Every realisation is one thread-block-resident ring of `no_neurons` integrate-and-fire
 * neurons; (column, realisation) pairs are the independent work items that shard across
 * GPUs (b200_edm_evolve_items_dev / b200_edm_reduce_items_dev).
 */
#ifndef B200_EDM_H
#define B200_EDM_H

#include "b200_common.h"
#include "b200_interp.h"   /* b200_dtype */

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200_edm b200_edm;

/* Model constants: the macros of parameters.hpp:1-15 as a runtime struct. */
typedef struct {
  double vth;            /* parameters.hpp:1  (1.0f) firing threshold                    */
  double a1, a2, b1, b2; /* parameters.hpp:3-6 (11,7,5,3.5) Mexican-hat coupling         */
  double I;              /* parameters.hpp:7  (0.9f) constant drive                       */
  double L;              /* parameters.hpp:8  (3.0f) half-length of the ring              */
  double tol;            /* parameters.hpp:9  (1e-6, a double literal) Newton tolerance   */
  double time_horizon;   /* parameters.hpp:15 (5.0f)                                      */
  uint32_t counter_max;  /* EventDrivenMap.cu:564 uses an UNDEFINED macro; we pick 100    */
  uint32_t quirks;       /* B200_EDM_QUIRK_* bits; 0 = intended semantics                 */
} b200_edm_model;

/* Q1 (SURVEY §8a): reproduce CountRealisationsKernel storing the count into accept[0]
 * (EventDrivenMap.cu:801) so that realisation 0 is dropped from the sum but kept in
 * the divisor (single-block behaviour). */
#define B200_EDM_QUIRK_ACCEPT0_BIAS 1u

/* Fill `m` with the values of parameters.hpp; float literals are widened exactly,
 * e.g. I = (double)0.9f. */
void b200_edm_model_default(b200_edm_model* m);

/* params[0] = beta (Driver.cu:15-16); further entries are stored but unused, as in the
 * reference.  no_fronts is the reference's compile-time noSpikes (parameters.hpp:12).
 * precision: B200_F64 (primary, 1e-10 parity) or B200_F32 (the reference's arithmetic). */
int b200_edm_create(const double* params, size_t nparams, uint32_t no_realisations,
                    uint32_t no_neurons, uint32_t no_fronts, b200_dtype precision,
                    b200_edm** handle);
int b200_edm_destroy(b200_edm* h);

int b200_edm_set_model(b200_edm* h, const b200_edm_model* m);
int b200_edm_get_model(const b200_edm* h, b200_edm_model* m);
int b200_edm_set_time_horizon(b200_edm* h, double T);
int b200_edm_set_no_realisations(b200_edm* h, uint32_t no_realisations);
int b200_edm_set_no_neurons(b200_edm* h, uint32_t no_neurons);
int b200_edm_set_param_stddev(b200_edm* h, double sigma);
int b200_edm_set_parameter(b200_edm* h, uint32_t par_id, double value);
/* The reference seeds cuRAND from clock() and re-applies the SAME seed on every
 * ComputeF (common random numbers, EventDrivenMap.cu:178,332-335).  Here the seed is
 * explicit and the generator is counter-based, so every column / GPU / run sees the
 * identical ensemble. */
int b200_edm_set_seed(b200_edm* h, uint64_t seed);
int b200_edm_get_seed(const b200_edm* h, uint64_t* seed);
/* PostProcess()/SetNewSeed(): advance to a new, deterministic seed. */
int b200_edm_new_seed(b200_edm* h);

/* f = F(z): one map evaluation.  n must equal no_fronts.  z = (c, T_2, ..., T_M). */
int b200_edm_compute_f(b200_edm* h, const double* z, size_t n, double* f_out);

/* ncols evaluations in one launch: z_cols and f_cols_out are n x ncols column-major. */
int b200_edm_compute_f_batch(b200_edm* h, const double* z_cols, size_t n, size_t ncols,
                             double* f_cols_out);

/* Forward-difference Jacobian exactly as NewtonSolver.cpp:164-197 forms it:
 * J(:,i) = (F(u + eps e_i) - F(u)) * pow(eps,-1), all n+1 evaluations in one batch.
 * f0_out (nullable) receives F(u). jac is n x n column-major. */
int b200_edm_compute_dfdu(b200_edm* h, const double* u, size_t n, double eps,
                          double* jac_out, double* f0_out);
/* The same Jacobian when the caller already holds f0 = F(u) — NewtonSolver.cpp:110 evaluates the residual before
 * :93 / :191 ask for the Jacobian, which then repeats it: only the n perturbed columns are evaluated here and
 * J(:,i) = (F(u + eps e_i) - f0) * pow(eps,-1).  With f0 = b200_edm_compute_f(u) the result is bitwise that of
 * b200_edm_compute_dfdu. */
int b200_edm_compute_dfdu_given_f(b200_edm* h, const double* u, size_t n, double eps,
                                  const double* f0, double* jac_out);

/* ---- profile map (BASELINE config 5: "1e3-dim coarse profile"; NEW, not in the reference) ----
 * The reference's coarse variable is 3 numbers (wave speed + front delays, noSpikes in
 * parameters.hpp:12).  With n_coarse > 0 the same handle instead evaluates the equation-free map on
 * coarse PROFILES u = (V_c[n_coarse], S_c[n_coarse]) sampled at X_c[i] = -L + (2L/n_coarse) i:
 *   lift     : linear interpolation (the interp1 rule, periodic ring) of (V_c, S_c) onto the no_neurons
 *              grid, neurons at/above threshold reset as in LiftKernel (EventDrivenMap.cu:540);
 *   evolve   : the reference's event-driven dynamics (EventDrivenMap.cu:544-618) for exactly time_horizon;
 *   restrict : linear interpolation of the fine state back onto the coarse knots, mean over realisations;
 *   F(u)     : Phi_T(u) - u (the equationFree convention of Stability.cpp:68-71).
 * Every entry point (compute_f, compute_f_batch, compute_dfdu, evolve/reduce_items_dev) then takes
 * vectors of length n = 2 n_coarse; B200_EDM_DBG_POSITION holds the restricted profiles [ncols][R][n].
 * n_coarse = 0 switches back to the reference's front map. */
int b200_edm_set_profile_mode(b200_edm* h, uint32_t n_coarse);

/* ---- in-process multi-GPU (for C++ callers without a launcher) ----
 * After this call compute_f / compute_f_batch / compute_dfdu shard over the listed devices of THIS process
 * (device_ids[0] must be the handle's device), so the reference's own callers — the finite-difference loops of
 * NewtonSolver.cpp:91-94,181-195 and Stability.cpp:59-62,95-109 — scale without change:
 *   - many columns (>= 4 per device, e.g. the 1001 evaluations of a 1000-dim Jacobian): every device owns a block
 *     of WHOLE columns — perturbed columns formed on the device, lift, evolve, fixed-order mean, difference
 *     quotient all local — and ONE ncclAllGather (single process, ncclCommInitAll) moves the n-vector of each
 *     column to every device; the base column F(u) is evaluated redundantly instead of being broadcast;
 *   - few columns (the reference's n = 3): the (column, realisation) work items are split, positions + accept
 *     flags are all-gathered and the primary reduces.
 * Results are bitwise those of a single device.  NCCL (libnccl.so.2) is loaded on first use and is
 * required for more than one device.  The reference is single-GPU (EventDrivenMap.cu:182,196). */
int b200_edm_set_devices(b200_edm* h, const int* device_ids, size_t ndevices);

/* Eigenvalues of a real general n x n matrix (column-major), the call behind arma::eig_gen in
 * Stability::ComputeEigenvalues / ComputeNumUnstableEigenvalues (Stability.cpp:40,72): cuSOLVER's 64-bit GEEV
 * on the current device (loaded on first use).  w_re / w_im receive the n eigenvalues. */
int b200_eig_gen_f64(size_t n, const double* a_colmajor, double* w_re, double* w_im);

/* ---- sharded evaluation (one process per GPU; see INTEGRATION.md) ----
 * Work item id = col * no_realisations + r.  evolve_items runs items [item_begin,
 * item_end) of the batch and writes, for local item k, M restricted front positions to
 * pos_dev[k*M .. k*M+M) and the accept flag to accept_dev[k].  After the slices of all
 * ranks are gathered (item order), reduce_items forms the masked mean per column in a
 * fixed order and the residual F — bitwise independent of how items were split.
 * z_cols is a HOST pointer (n x ncols parameters); pos / accept / f_cols are DEVICE
 * pointers; positions cross the boundary as double whatever the handle's precision. */
int b200_edm_evolve_items_dev(b200_edm* h, const double* z_cols, size_t n, size_t ncols,
                              size_t item_begin, size_t item_end, double* pos_dev,
                              int32_t* accept_dev, void* stream);
int b200_edm_reduce_items_dev(b200_edm* h, const double* z_cols, size_t n, size_t ncols,
                              const double* pos_all_dev, const int32_t* accept_all_dev,
                              double* f_cols_dev, void* stream);

/* ---- observability (replaces the Save*() text dumps, EventDrivenMap.cu:406-503) ---- */
typedef enum {
  B200_EDM_DBG_INIT_INDEX    = 0, /* int32  [ncols][M]      initialSpikeInd                 */
  B200_EDM_DBG_LIFT_V        = 1, /* double [ncols][N]      testLift.dat col 1               */
  B200_EDM_DBG_LIFT_S        = 2, /* double [ncols][N]      testLift.dat col 2               */
  B200_EDM_DBG_LAST_INDEX    = 3, /* int32  [ncols][R][M]   testLastSpikeInd.dat             */
  B200_EDM_DBG_LAST_TIME     = 4, /* double [ncols][R][M]   testLastSpikeTime.dat            */
  B200_EDM_DBG_CROSSED_INDEX = 5, /* int32  [ncols][R][M]   testCrossedSpikeInd.dat          */
  B200_EDM_DBG_CROSSED_TIME  = 6, /* double [ncols][R][M]   testCrossedSpikeTime.dat         */
  B200_EDM_DBG_ACCEPT        = 7, /* int32  [ncols][R]      testAcceptFlag.dat               */
  B200_EDM_DBG_POSITION      = 8, /* double [ncols][R][M]   testAverages.dat                 */
  B200_EDM_DBG_EVENT_COUNT   = 9, /* int32  [ncols][R]      events processed per realisation */
  B200_EDM_DBG_MEAN          = 10,/* double [ncols][M]      testAveraged.dat                 */
  B200_EDM_DBG_BETA          = 11,/* double [R][N]          per-neuron beta ensemble         */
  B200_EDM_DBG_COUPLING      = 12 /* double [N]             test.dat (coupling kernel w)     */
} b200_edm_debug_what;

/* Copy an array of the most recent compute_f / compute_f_batch / compute_dfdu call to
 * host memory.  Available only while the debug flag is set (SetDebugFlag). */
int b200_edm_set_debug(b200_edm* h, int on);
int b200_edm_debug_fetch(b200_edm* h, b200_edm_debug_what what, void* out, size_t bytes);

/* Bench introspection: device time (ms, CUDA events on the launch stream) of the evolve
 * kernel of the most recent call, and total number of events it processed. */
int b200_edm_last_evolve_ms(const b200_edm* h, double* ms);
int b200_edm_last_event_total(const b200_edm* h, uint64_t* events);
int b200_edm_enable_timing(b200_edm* h, int on);
/* Work counters of the most recent call (valid while timing or debug is on):
 * out[0] events, out[1] neurons that survived the candidate filter, out[2] Newton
 * iterations, out[3] block-wide exact passes (ring gone quiet). */
int b200_edm_last_counters(const b200_edm* h, uint64_t out[4]);
/* SURVEY Q15 soft flag of the most recent call: 1 if some front started outside the
 * domain (EventDrivenMap.cu:365-372 leaves the index unassigned; here it is 0). */
int b200_edm_last_init_clamped(const b200_edm* h, int* clamped);
/* Launch tuning: neurons handled by one thread (0 = choose from no_neurons; 4, 8 or 16).
 * The reference fixes one neuron per thread (EventDrivenMap.cu:182,196). */
int b200_edm_set_tuning(b200_edm* h, int neurons_per_thread);

#ifdef __cplusplus
}
#endif
#endif /* B200_EDM_H */
