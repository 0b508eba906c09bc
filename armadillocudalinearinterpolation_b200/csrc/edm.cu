// edm.cu — event-driven coarse time-stepper ("lift -> evolve -> restrict") for sm_100a
// (include/b200_edm.h).
//
// Replaces class EventDrivenMap of the reference: host wrapper EventDrivenMap.cu:57-503 and
// kernels EventDrivenMap.cu:378-386, 505-945.  Same map, different program:
//
//  reference (Kepler, FP32)                     here (B200, FP64 primary / FP32 compat)
//  ------------------------------------------   -------------------------------------------
//  6 launches + cuRAND + 3 H2D + memset / eval  3 launches per BATCH of evaluations
//  LiftKernel on R*N threads (R-fold redundant) prepare kernel: once per column
//  one thread per neuron, 1024-thread blocks    NPT neurons per thread, 128..256-thread CTAs,
//                                               several CTAs resident per SM
//  every neuron: pow + Newton chain per event   two-stage candidate test: a conservative
//                                               MUFU (lg2/ex2) filter proves "cannot fire"
//                                               for ~99% of neurons; survivors are compacted
//                                               into one warp that runs the exact FP64
//                                               pow + Newton (identical iterates)
//  shuffle-tree arg-min over 1024 threads,      REDUX arg-min over the handful of candidates,
//  2 barriers, undefined tie rule               smallest (time, index) — SURVEY Q5
//  every thread: 3 exp per event                event-uniform exponentials computed once per
//                                               event by the finalising thread (homogeneous
//                                               ensemble) -> 3 FMA per neuron advance
//  RestrictKernel on 3R*N threads for 3R items  folded into the evolve epilogue
//  racy count + mean                            fixed-order masked mean (bitwise independent
//                                               of how items were sharded over GPUs)
//
// The event sequence (which neuron fires when) is identical to the CPU restatement in
// oracle/edm_oracle_impl.inc: the filter only ever skips neurons for which the reference's
// `decision` predicate (EventDrivenMap.cu:559) is provably false.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <new>
#include <vector>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>
#include "b200_edm.h"
#include "common.cuh"

namespace b200 {
namespace {

// ---------------------------------------------------------------- math helpers ----
template <typename T> struct M;
template <> struct M<double> {
  static __device__ __forceinline__ double exp_(double x) { return exp(x); }
  static __device__ __forceinline__ double pow_(double x, double y) { return pow(x, y); }
  static __device__ __forceinline__ double nan_() { return __longlong_as_double(0x7ff8000000000000ll); }
};
template <> struct M<float> {
  static __device__ __forceinline__ float exp_(float x) { return expf(x); }
  static __device__ __forceinline__ float pow_(float x, float y) { return powf(x, y); }
  static __device__ __forceinline__ float nan_() { return __int_as_float(0x7fc00000); }
};

// ---- short-latency FP64 exp / divide for the event loop ----
// The loop's critical path is a serial Newton chain (divide -> two exps -> f, df) run by a
// handful of lanes while the rest of the CTA waits at a barrier, so what matters is the length of
// the dependent-instruction chain, not instruction count.  exp(x) = 2^(k/64) * exp(r) with a
// 64-entry table of 2^(j/64) in shared memory and a degree-5 polynomial in Estrin form
// (|r| <= ln2/128, truncation 3.5e-17): ~10 dependent operations instead of ~30, about 1 ulp.
// Division uses MUFU.RCP64H + two Newton steps + one residual correction (no IEEE fix-up path).
__device__ __forceinline__ double fast_exp(double x, const double* __restrict__ tab) {
  if (!(fabs(x) < 690.0)) return exp(x);  // overflow / underflow / NaN: library path
  const double t = fma(x, 92.33248261689366, 6755399441055744.0);  // 64/ln2, round-to-nearest magic
  const int k = __double2loint(t);
  const double kd = t - 6755399441055744.0;
  double r = fma(kd, -0x1.62e42fee00000p-7, x);    // ln2/64, high 32 bits (kd * hi is exact)
  r = fma(kd, -0x1.a39ef35793c76p-39, r);           // ln2/64, low part
  const double r2 = r * r;
  const double a = fma(r, 1.0 / 6.0, 0.5);
  const double b = fma(r, 1.0 / 120.0, 1.0 / 24.0);
  const double q = fma(r2, fma(r2, b, a), r);          // exp(r) - 1
  const double tj = tab[k & 63];
  const double m = fma(tj, q, tj);
  const int e = k >> 6;
  return __hiloint2double(__double2hiint(m) + (e << 20), __double2loint(m));
}
__device__ __forceinline__ float fast_exp(float x, const float*) { return expf(x); }
// Two exponentials at once.  fast_exp's range test is a branch, and two calls in a row become two control-flow
// regions that a warp executes one after the other (in-order issue): ~2 x 11 dependent FP64 operations.  One range
// test for both arguments and the two chains written side by side let them overlap (same operations, same bits).
__device__ __forceinline__ void fast_exp_pair(double x1, double x2, const double* __restrict__ tab, double& o1, double& o2) {
  if (!(fabs(x1) < 690.0 && fabs(x2) < 690.0)) { o1 = fast_exp(x1, tab); o2 = fast_exp(x2, tab); return; }
  const double t1 = fma(x1, 92.33248261689366, 6755399441055744.0), t2 = fma(x2, 92.33248261689366, 6755399441055744.0);
  const int k1 = __double2loint(t1), k2 = __double2loint(t2);
  const double kd1 = t1 - 6755399441055744.0, kd2 = t2 - 6755399441055744.0;
  double r1 = fma(kd1, -0x1.62e42fee00000p-7, x1), r2 = fma(kd2, -0x1.62e42fee00000p-7, x2);
  r1 = fma(kd1, -0x1.a39ef35793c76p-39, r1); r2 = fma(kd2, -0x1.a39ef35793c76p-39, r2);
  const double s1 = r1 * r1, s2 = r2 * r2;
  const double a1 = fma(r1, 1.0 / 6.0, 0.5), a2 = fma(r2, 1.0 / 6.0, 0.5);
  const double b1 = fma(r1, 1.0 / 120.0, 1.0 / 24.0), b2 = fma(r2, 1.0 / 120.0, 1.0 / 24.0);
  const double q1 = fma(s1, fma(s1, b1, a1), r1), q2 = fma(s2, fma(s2, b2, a2), r2);
  const double tj1 = tab[k1 & 63], tj2 = tab[k2 & 63];
  const double m1 = fma(tj1, q1, tj1), m2 = fma(tj2, q2, tj2);
  o1 = __hiloint2double(__double2hiint(m1) + ((k1 >> 6) << 20), __double2loint(m1));
  o2 = __hiloint2double(__double2hiint(m2) + ((k2 >> 6) << 20), __double2loint(m2));
}
__device__ __forceinline__ void fast_exp_pair(float x1, float x2, const float*, float& o1, float& o2) { o1 = expf(x1); o2 = expf(x2); }
// G exponentials at once, written stage by stage so that the G chains overlap (heterogeneous ensembles need one
// exponential per neuron and event: eight calls in a row were eight serial regions)
template <int G>
__device__ __forceinline__ void fast_exp_vec(const double (&x)[G], const double* __restrict__ tab, double (&o)[G]) {
  bool in = true;
#pragma unroll
  for (int i = 0; i < G; ++i) in = in && (fabs(x[i]) < 690.0);
  if (!in) {
#pragma unroll
    for (int i = 0; i < G; ++i) o[i] = fast_exp(x[i], tab);
    return;
  }
  double t[G], r[G], q[G], tj[G];
  int k[G];
#pragma unroll
  for (int i = 0; i < G; ++i) { t[i] = fma(x[i], 92.33248261689366, 6755399441055744.0); k[i] = __double2loint(t[i]); }
#pragma unroll
  for (int i = 0; i < G; ++i) { const double kd = t[i] - 6755399441055744.0; r[i] = fma(kd, -0x1.a39ef35793c76p-39, fma(kd, -0x1.62e42fee00000p-7, x[i])); tj[i] = tab[k[i] & 63]; }
#pragma unroll
  for (int i = 0; i < G; ++i) {
    const double r2 = r[i] * r[i];
    q[i] = fma(r2, fma(r2, fma(r[i], 1.0 / 120.0, 1.0 / 24.0), fma(r[i], 1.0 / 6.0, 0.5)), r[i]);
  }
#pragma unroll
  for (int i = 0; i < G; ++i) {
    const double m = fma(tj[i], q[i], tj[i]);
    o[i] = __hiloint2double(__double2hiint(m) + ((k[i] >> 6) << 20), __double2loint(m));
  }
}
template <int G>
__device__ __forceinline__ void fast_exp_vec(const float (&x)[G], const float*, float (&o)[G]) {
#pragma unroll
  for (int i = 0; i < G; ++i) o[i] = expf(x[i]);
}
__device__ __forceinline__ double fast_div(double a, double b) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
  y = fma(y, fma(-b, y, 1.0), y);
  y = fma(y, fma(-b, y, 1.0), y);
  const double q = a * y;
  return fma(fma(-q, b, a), y, q);
}
__device__ __forceinline__ float fast_div(float a, float b) { return a / b; }

// model constants in the arithmetic type of the run (parameters.hpp:1-15)
template <typename T>
struct Consts {
  T vth, a1, a2, b1, b2, I, L, T_end;
  double tol;  // parameters.hpp:9: a double literal; |f| is widened for the compare
  unsigned counter_max;
};

// counter-based standard normal (the CPU restatement mirrors this construction)
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__device__ __forceinline__ double normal_at(unsigned long long seed, unsigned long long index) {
  unsigned long long h1 = splitmix64(seed ^ splitmix64(2 * index));
  unsigned long long h2 = splitmix64(seed ^ splitmix64(2 * index + 1));
  double u1 = ((double)(h1 >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  double u2 = ((double)(h2 >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  return sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925286766559 * u2);
}

// per-neuron beta ensemble; replaces curandGenerateNormal (EventDrivenMap.cu:179)
template <typename T>
__global__ void edm_beta_kernel(T* __restrict__ beta, size_t n, double mean, double sigma,
                                unsigned long long seed) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) beta[i] = (T)(mean + sigma * normal_at(seed, i));
}

// coupling kernel w[d] = kernel at ring distance d (BuildCouplingKernel + circshift,
// EventDrivenMap.cu:111-129, 826-841)
template <typename T>
__global__ void edm_coupling_kernel(Consts<T> k, unsigned N, T* __restrict__ w) {
  unsigned d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= N) return;
  unsigned i = (d + N / 2) % N;  // circshift by N/2
  T x = -k.L + (T)(2 * k.L / N) * i;
  T ax = fabs(x);
  w[d] = (k.a1 * M<T>::exp_(-k.b1 * ax) - k.a2 * M<T>::exp_(-k.b2 * ax)) * 2 * k.L / N;
}

// ---------------------------------------------------------------- prepare (lift) ----
// One CTA per column: initial front indices (initialSpikeInd, EventDrivenMap.cu:361-372),
// ZtoU (:388-396) and the analytic travelling-wave profile (LiftKernel, :505-542).  The
// lift is identical for every realisation (it uses the mean beta, SURVEY Q7), so it is
// evaluated once per column instead of once per (realisation, neuron).
template <typename T>
struct FrontCoef {  // x-independent factors of front m (U[m] = tau)
  T y;                 // c * tau
  T p1, p2;            // K+_i * exp(y (1+c b_i)/c) * exp(-b_i y)   (d > 0 branch, first two terms)
  T q1, q2;            // K+_i * exp(-b_i y)                        (d <= 0 branch)
  T g1, g2, e_tau;     // G_i * exp(beta tau),  exp(tau (1-beta))
  T h1, h2, k1, k2;    // H_i * exp(b_i y),  exp(y (1 - c b_i)/c)
};

template <typename T>
__global__ void __launch_bounds__(256)
edm_prepare_kernel(Consts<T> k, unsigned N, unsigned Mf, T beta, const double* __restrict__ z_cols,
                   int32_t* __restrict__ init_index, int32_t* __restrict__ clamped,
                   T* __restrict__ lift_v, T* __restrict__ lift_s) {
  extern __shared__ unsigned char smem_prep[];
  FrontCoef<T>* fc = reinterpret_cast<FrontCoef<T>*>(smem_prep);
  const unsigned col = blockIdx.x;
  const double* z = z_cols + (size_t)col * Mf;
  const T one = (T)1, two = (T)2;
  const T c = (T)z[0];
  const T a1 = k.a1, a2 = k.a2, b1 = k.b1, b2 = k.b2, L = k.L;
  const T cb1 = c * b1, cb2 = c * b2;

  if (threadIdx.x == 0) {
    // descending scan for the last grid point left of each front
    int32_t prev = (int32_t)(N / 2);
    init_index[(size_t)col * Mf] = prev;
    int any_clamped = 0;
    for (unsigned m = 1; m < Mf; ++m) {
      const double target = -z[0] * z[m];
      int32_t found = 0;
      int hit = 0;
      for (int32_t i = prev; i > 0; --i) {
        if ((double)(-L + (T)(2 * (unsigned)i * L / N)) < target) { found = i; hit = 1; break; }
      }
      if (!hit) any_clamped = 1;  // SURVEY Q15: front outside the domain -> index 0 + soft flag
      init_index[(size_t)col * Mf + m] = found;
      prev = found;
    }
    if (any_clamped) atomicOr(clamped, 1);
  }
  // x-independent coefficients, one thread per front
  for (unsigned m = threadIdx.x; m < Mf; m += blockDim.x) {
    const T tau = (m == 0) ? (T)0 : (T)z[m];  // U = (c, 0, T_2, ..., T_M)
    const T y = c * tau;
    FrontCoef<T> f;
    f.y = y;
    const T Kp1 = (a1 * beta * c) / ((beta + cb1) * (one + cb1));
    const T Kp2 = (a2 * beta * c) / ((beta + cb2) * (one + cb2));
    f.q1 = Kp1 * M<T>::exp_(-b1 * y);
    f.q2 = Kp2 * M<T>::exp_(-b2 * y);
    f.p1 = Kp1 * M<T>::exp_(y * ((one + cb1) / c)) * M<T>::exp_(-b1 * y);
    f.p2 = Kp2 * M<T>::exp_(y * ((one + cb2) / c)) * M<T>::exp_(-b2 * y);
    f.g1 = (a1 * beta * c / (one - beta)) * M<T>::exp_(beta * tau) * (one / (beta + cb1) + one / (cb1 - beta));
    f.g2 = (a2 * beta * c / (one - beta)) * M<T>::exp_(beta * tau) * (one / (beta + cb2) + one / (cb2 - beta));
    f.e_tau = M<T>::exp_(tau * (one - beta));
    f.h1 = (a1 * beta * c / ((cb1 - beta) * (one - cb1))) * M<T>::exp_(b1 * y);
    f.h2 = (a2 * beta * c / ((cb2 - beta) * (one - cb2))) * M<T>::exp_(b2 * y);
    f.k1 = M<T>::exp_(y * ((one - cb1) / c));
    f.k2 = M<T>::exp_(y * ((one - cb2) / c));
    fc[m] = f;
  }
  __syncthreads();

  // synaptic-profile constants of the "behind the front" branch
  const T s_a1 = beta * a1 * (c / (beta + cb1)), s_a2 = beta * a2 * (c / (beta + cb2));
  const T s_c1 = (two * a1 / b1) * (beta / (one - ((beta * beta) / (c * c * b1 * b1))));
  const T s_c2 = (two * a2 / b2) * (beta / (one - ((beta * beta) / (c * c * b2 * b2))));
  const T s_d1 = beta * a1 * (c / (cb1 - beta)), s_d2 = beta * a2 * (c / (cb2 - beta));

  for (unsigned j = threadIdx.x; j < N; j += blockDim.x) {
    // two rounded operations (no FMA): a grid point that coincides with a front must land on
    // the same side of it as in the CPU restatement
    const T x = sub_rn(L, mul_rn((T)(2 * L / N), (T)j));
    // factors that depend on x only
    const T ex_beta = M<T>::exp_((x / c) * (one - beta));
    const T ex_m1 = M<T>::exp_(x * ((one - cb1) / c)), ex_m2 = M<T>::exp_(x * ((one - cb2) / c));
    const T ex_p1 = M<T>::exp_(x * ((one + cb1) / c)), ex_p2 = M<T>::exp_(x * ((one + cb2) / c));
    const T ex_lead = M<T>::exp_(-x / c);
    T acc_v = (T)0, acc_s = (T)0;
    for (unsigned m = 0; m < Mf; ++m) {
      const FrontCoef<T> f = fc[m];
      const T d = x - f.y;
      // both branches are evaluated and multiplied by 0/1 masks exactly as the reference
      // does, so overflow-to-NaN behaviour (SURVEY Q8, FP32) is preserved
      const T gt = (T)(d > (T)0), le = (T)(d <= (T)0);
      const T ahead = f.p1 - f.p2 + f.g1 * (ex_beta - f.e_tau) - f.h1 * (ex_m1 - f.k1)
                      - f.g2 * (ex_beta - f.e_tau) + f.h2 * (ex_m2 - f.k2);
      const T behind = f.q1 * ex_p1 - f.q2 * ex_p2;
      const T dv = (gt * ahead + le * behind) * ex_lead;
      acc_v += dv - gt * M<T>::exp_(-d / c) + le * (T)0;
      const T e = f.y - x;  // = -d
      const T gt2 = (T)(e > (T)0), le2 = (T)(e <= (T)0);
      acc_s += gt2 * (s_a1 * M<T>::exp_(b1 * (x - f.y)) - s_a2 * M<T>::exp_(b2 * (x - f.y)))
             + le2 * (s_c1 * M<T>::exp_(-(beta / c) * (x - f.y)) - s_d1 * M<T>::exp_(b1 * (f.y - x))
                      - s_c2 * M<T>::exp_(-(beta / c) * (x - f.y)) + s_d2 * M<T>::exp_(b2 * (f.y - x)));
    }
    T v = k.I + acc_v;
    v *= (T)(v < one);  // neurons lifted above threshold start from reset
    lift_v[(size_t)col * N + j] = v;
    lift_s[(size_t)col * N + j] = acc_s;
  }
}

// ---------------------------------------------------------------- profile map helpers ----
// Periodic linear interpolation on the ring grid X[i] = -L + (2L/n) i (X[n] = L carries y[0]) with the
// interp1 rule (w = |X[a]-x| / (|X[a]-x| + |X[b]-x|), (1-w) y[a] + w y[b]); every operation individually
// rounded so that the lifted / restricted profiles equal the CPU restatement bit for bit.
template <typename T>
__device__ __forceinline__ T periodic_interp(const T* __restrict__ y, unsigned n, T L, T x) {
  const T h = div_rn(mul_rn((T)2, L), (T)n);
  long long a = (long long)div_rn(add_rn(x, L), h);
  a = max(0ll, min(a, (long long)n - 1));
  while (a > 0 && add_rn(-L, mul_rn(h, (T)a)) > x) --a;
  while (a + 1 <= (long long)n - 1 && add_rn(-L, mul_rn(h, (T)(a + 1))) <= x) ++a;
  const T xa = add_rn(-L, mul_rn(h, (T)a));
  const T xb = (a + 1 == (long long)n) ? L : add_rn(-L, mul_rn(h, (T)(a + 1)));
  const T ya = y[a], yb = y[(a + 1) % n];
  const T ea = fabs(sub_rn(xa, x)), eb = fabs(sub_rn(xb, x));
  const T w = (ea > (T)0) ? div_rn(ea, add_rn(ea, eb)) : (T)0;
  return add_rn(mul_rn(sub_rn((T)1, w), ya), mul_rn(w, yb));
}

// Lift of the profile map: coarse (V_c, S_c) -> neurons, one CTA per column; neurons lifted at or above
// threshold start from reset, as in LiftKernel (EventDrivenMap.cu:540).
template <typename T>
__global__ void __launch_bounds__(256)
edm_profile_lift_kernel(Consts<T> k, unsigned N, unsigned nc, const double* __restrict__ u_cols,
                        T* __restrict__ uc_scratch, T* __restrict__ lift_v, T* __restrict__ lift_s) {
  const unsigned col = blockIdx.x;
  const double* u = u_cols + (size_t)col * 2 * nc;
  T* uc = uc_scratch + (size_t)col * 2 * nc;   // the column in the arithmetic type of the run
  for (unsigned i = threadIdx.x; i < 2 * nc; i += blockDim.x) uc[i] = (T)u[i];
  __syncthreads();
  for (unsigned j = threadIdx.x; j < N; j += blockDim.x) {
    const T x = add_rn(-k.L, mul_rn((T)(2 * k.L / N), (T)j));
    T v = periodic_interp<T>(uc, nc, k.L, x);
    v *= (T)(v < (T)1);
    lift_v[(size_t)col * N + j] = v;
    lift_s[(size_t)col * N + j] = periodic_interp<T>(uc + nc, nc, k.L, x);
  }
}

// Mean over accepted realisations in a fixed order, F = mean - u.  One thread per (column, entry).
template <typename T>
__global__ void __launch_bounds__(256)
edm_profile_reduce_kernel(unsigned R, unsigned n, size_t ncols, const double* __restrict__ u_cols,
                          const T* __restrict__ restricted, const int32_t* __restrict__ accept,
                          double* __restrict__ f_cols) {
  const size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= ncols * n) return;
  const size_t col = g / n;
  const unsigned m = (unsigned)(g % n);
  const T* base = restricted + col * R * n + m;
  const int32_t* acc = accept + col * R;
  T sum = (T)0;
  unsigned count = 0;
  for (unsigned r = 0; r < R; ++r)
    if (acc[r] == 1) { sum += base[(size_t)r * n]; ++count; }
  f_cols[g] = (double)(sum / count) - u_cols[g];
}

// ---------------------------------------------------------------- evolve ----
// `decision` predicate of eventTime (EventDrivenMap.cu:559), evaluated exactly as written.
template <typename T>
__device__ __forceinline__ bool exact_decision(const Consts<T>& k, T v, T s, T beta) {
  const T one = (T)1;
  const T r = s / (k.vth - k.I);
  const T p = M<T>::pow_(r, one / beta);
  return v > k.vth * p + k.I * (one - p) - (k.vth - k.I) / (beta - one) * (r - p);
}

// Newton from t = 0 on the closed-form membrane solution (fun/dfun/eventTime,
// EventDrivenMap.cu:544-573): same iterates, same stopping test as the reference.
template <typename T>
__device__ __forceinline__ T newton_event_time(const Consts<T>& k, T v, T s, T beta, const T* etab,
                                               unsigned& its, T* e1_final = nullptr, T* e2_final = nullptr,
                                               bool* e_valid = nullptr) {
  const T one = (T)1;
  const T i1mb = fast_div(one, one - beta), ibm1 = -i1mb;
  T t = (T)0;
  T f = v - k.vth;         // fun(0)  : exp(0) = 1 makes every other term exactly 0
  T df = (k.I - v) + s;    // dfun(0)
  unsigned counter = 0;
  // the Newton step f/df is formed BEFORE the stopping test of its iteration is resolved, so that the compare and
  // the loop branch hide behind the divide's dependency chain (a warp issues in order); the step of the converged
  // iterate is computed and dropped.  Same iterates, same stopping rule.
  T step = fast_div(f, df);
  T e1 = one, e2 = one;    // exp(-t), exp((1-beta) t) at the current iterate
  while (((double)fabs(f) > k.tol) && (counter < k.counter_max)) {
    t -= step;
    fast_exp_pair(-t, (one - beta) * t, etab, e1, e2);
    const T se1 = s * e1;
    f = v * e1 + k.I * (one - e1) + se1 * i1mb * (e2 - one) - k.vth;
    df = k.I * e1 - v * e1 + se1 * e2 + (se1 * (e2 - one)) * ibm1;
    step = fast_div(f, df);
    counter++;
  }
  its += counter;
  T out = fabs(t);
  if (out != out) out = (T)100;  // Q5: a NaN event time never wins the arg-min
  // the exponentials of the final iterate are what the event message needs if this neuron wins (event time = t for
  // t >= 0): handed back so that the publishing thread need not recompute them (uncapped build only)
  if (e1_final) { *e1_final = e1; *e2_final = e2; *e_valid = (t >= (T)0) && counter > 0; }
  return out;
}

template <typename T>
__device__ __forceinline__ T exact_event_time(const Consts<T>& k, T v, T s, T beta, const T* etab, unsigned& its) {
  if (!exact_decision<T>(k, v, s, beta)) return (T)100;
  return newton_event_time<T>(k, v, s, beta, etab, its);
}

// order-preserving integer key of a non-negative, non-NaN time
__device__ __forceinline__ unsigned long long time_key(double t) { return (unsigned long long)__double_as_longlong(t); }
__device__ __forceinline__ unsigned long long time_key(float t) { return (unsigned long long)__float_as_uint(t); }

// warp-wide lexicographic min of (key, idx); every lane gets the result
__device__ __forceinline__ void warp_argmin(unsigned long long& key, unsigned& idx) {
  const unsigned full = 0xffffffffu;
  unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
  unsigned mhi = __reduce_min_sync(full, hi);
  unsigned lo_c = (hi == mhi) ? lo : 0xffffffffu;
  unsigned mlo = __reduce_min_sync(full, lo_c);
  unsigned id_c = (hi == mhi && lo == mlo) ? idx : 0xffffffffu;
  idx = __reduce_min_sync(full, id_c);
  key = ((unsigned long long)mhi << 32) | mlo;
}

template <typename T>
struct EventMsg {       // written by thread 0 after the arg-min, read by everybody after the barrier
  T dt, e1, cA, cB, e12;  // event-uniform advance coefficients (cB, e12: homogeneous ensemble)
  unsigned idx;
  int fallback;         // 1: nobody can fire within 100 time units -> block-wide exact pass
  int last;             // profile map: final event-free advance to the horizon
};

template <typename T>
struct EvolveArgs {
  Consts<T> k;
  unsigned N, R, Mf;
  T beta_mean;
  const T* beta;        // [R][N] or nullptr (homogeneous)
  const T* w;           // [N]
  const T* lift_v;      // [ncols][N]
  const T* lift_s;
  const int32_t* init_index;  // [ncols][M]
  unsigned long long item_begin;
  // outputs, indexed by local item (blockIdx.x)
  T* position;          // [items][M]
  int32_t* accept;      // [items]
  int32_t* event_count; // [items]
  int32_t* last_index;  // [items][M]   (nullable group: debug)
  int32_t* crossed_index;
  T* last_time;
  T* crossed_time;
  unsigned long long* counters;  // [4]: events, candidates (filter survivors), newton its, fallbacks (nullable)
  unsigned profile_nc;   // 0: front map (the reference); > 0: profile map on profile_nc coarse knots
};

// The candidate list holds at most kCandCap neurons (typically ~10 survive the filter); if more
// do, the event is resolved by the exact block-wide pass instead.
constexpr unsigned kCandCap = 256;
__host__ __device__ inline unsigned cand_cap(unsigned N) { return N < kCandCap ? N : kCandCap; }

template <typename T>
__host__ __device__ inline size_t evolve_smem_bytes(unsigned N, unsigned Mf, bool het, bool profile = false) {
  size_t b = profile ? 2 * sizeof(T) * N : 0;   // fine state staged for the restriction
  const unsigned cap = cand_cap(N);
  b += sizeof(T) * N;                       // bw / w
  b += sizeof(T) * cap * (het ? 3 : 2);     // cand_v, cand_s, (cand_b)
  b += sizeof(int) * cap;                   // cand_i
  b += (sizeof(T) * 2 + sizeof(int) * 2 + 4) * Mf;  // front bookkeeping
  b += sizeof(T) * 64;                      // exp table
  b += 256;                                 // scalars + alignment slack
  b += 32 * 16;                             // per-warp partial results
  return b;
}

template <typename T, int NPT, bool HET, int MAXT, int MINB, bool FULL>
__global__ void __launch_bounds__(MAXT, MINB)
edm_evolve_kernel(const EvolveArgs<T> A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned N = A.N, Mf = A.Mf;
  const unsigned tid = threadIdx.x, nthr = blockDim.x;
  const unsigned lane = tid & 31, warp = tid >> 5, nwarps = (nthr + 31) >> 5;
  // ---- shared memory carve-up ----
  unsigned char* sp = smem_raw;
  T* bw = reinterpret_cast<T*>(sp); sp += sizeof(T) * N;            // w[d] (x beta when homogeneous)
  const unsigned cap = cand_cap(N);
  T* cand_v = reinterpret_cast<T*>(sp); sp += sizeof(T) * cap;
  T* cand_s = reinterpret_cast<T*>(sp); sp += sizeof(T) * cap;
  T* cand_b = nullptr;
  if (HET) { cand_b = reinterpret_cast<T*>(sp); sp += sizeof(T) * cap; }
  T* last_t = reinterpret_cast<T*>(sp); sp += sizeof(T) * Mf;
  T* cross_t = reinterpret_cast<T*>(sp); sp += sizeof(T) * Mf;
  T* etab = reinterpret_cast<T*>(sp); sp += sizeof(T) * 64;         // 2^(j/64) for fast_exp
  sp = smem_raw + (((size_t)(sp - smem_raw) + 15) & ~(size_t)15);
  unsigned long long* wkey = reinterpret_cast<unsigned long long*>(sp); sp += 8 * 32;
  EventMsg<T>* ev = reinterpret_cast<EventMsg<T>*>(sp); sp += ((sizeof(EventMsg<T>) + 15) / 16) * 16;
  unsigned long long* fb_key = reinterpret_cast<unsigned long long*>(sp); sp += 8;
  int* cand_i = reinterpret_cast<int*>(sp); sp += sizeof(int) * cap;
  int* last_i = reinterpret_cast<int*>(sp); sp += sizeof(int) * Mf;
  int* cross_i = reinterpret_cast<int*>(sp); sp += sizeof(int) * Mf;
  unsigned* widx = reinterpret_cast<unsigned*>(sp); sp += 4 * 32;
  int* ncand = reinterpret_cast<int*>(sp); sp += 8;                 // [2], double buffered
  unsigned* fb_idx = reinterpret_cast<unsigned*>(sp); sp += 4;
  int* stop = reinterpret_cast<int*>(sp); sp += 4;
  unsigned char* crossed = sp; sp += Mf;                            // [Mf]
  sp = smem_raw + (((size_t)(sp - smem_raw) + 15) & ~(size_t)15);
  T* sv = reinterpret_cast<T*>(sp);                                 // profile map only: [N] + [N]
  T* ss = sv + N;

  const unsigned long long item = A.item_begin + blockIdx.x;
  const unsigned col = (unsigned)(item / A.R), r = (unsigned)(item % A.R);
  const Consts<T> k = A.k;
  const T one = (T)1;

  // ---- per-neuron state in registers; neuron j = tid + q * nthr ----
  T v[NPT], s[NPT], bt[HET ? NPT : 1], ibm1[HET ? NPT : 1];
  bool filt[HET ? NPT : 1];
#pragma unroll
  for (int q = 0; q < NPT; ++q) {
    const unsigned j = tid + q * nthr;
    if (j < N) {
      v[q] = A.lift_v[(size_t)col * N + j];
      s[q] = A.lift_s[(size_t)col * N + j];
      if (HET) {
        bt[q] = A.beta[(size_t)r * N + j];
        ibm1[q] = one / (bt[q] - one);
        filt[q] = bt[q] >= (T)1.5 && (k.vth - k.I) > (T)0;
      }
    } else {
      v[q] = (T)0; s[q] = (T)0;
      if (HET) { bt[q] = (T)2; ibm1[q] = one; filt[q] = true; }
    }
  }
  // homogeneous-ensemble constants
  const T hb = A.beta_mean;
  const T h_ibm1 = one / (hb - one);
  const T h_i1mb = one / (one - hb);
  // the conservative filter assumes vth - I > 0 and beta > 1 (g decreasing in p); outside that regime every
  // neuron is handed to the exact predicate instead (advisor finding, round 1)
  const bool h_filt = hb >= (T)1.5 && (k.vth - k.I) > (T)0;
  const float h_invb32 = (float)(one / hb);
  const T inv_vmI = one / (k.vth - k.I);
  const T vmI = k.vth - k.I;

  for (unsigned d = tid; d < N; d += nthr) bw[d] = HET ? A.w[d] : hb * A.w[d];
  for (unsigned i = tid; i < 64; i += nthr) etab[i] = (T)exp2((double)i * (1.0 / 64.0));
  if (tid == 0) {
    ncand[0] = 0; ncand[1] = 0; *stop = 0;
    for (unsigned m = 0; m < Mf; ++m) {
      last_i[m] = A.init_index[(size_t)col * Mf + m];  // EventDrivenMap.cu:595-599
      last_t[m] = (T)0;                                // Q4
      cross_i[m] = 0; cross_t[m] = (T)0; crossed[m] = 0;
    }
  }
  // finalising-thread state
  T t_now = (T)0;
  unsigned n_crossed = 0;
  int n_events = 0;
  unsigned stat_cand = 0, stat_newton = 0, stat_fb = 0;
  __syncthreads();

  // Conservative candidate test.  The reference's predicate is
  //   v > vth p + I (1-p) - (vth-I)/(beta-1) (r - p),  r = s/(vth-I), p = r^(1/beta),
  // i.e. g := (v - vth) - (vth-I) * ((beta p - r)/(beta-1) - 1) > 0.  Stage 2 evaluates p with
  // the MUFU lg2/ex2 units (relative error < 2e-6); the neuron is dropped only when g is below
  // -1e-4 (1 + p), orders of magnitude more than that error can move it.
  // Two passes so that the common case is straight-line code: stage 1 for all NPT neurons of the thread without a
  // branch (a bit per survivor), then — only in the few warps that sit on a front — stage 2 and the append.
  auto scan_straight = [&](int parity) {
    unsigned mask = 0;
    // stage by stage over the thread's NPT neurons, not neuron by neuron: a warp issues in order, so the NPT
    // independent dependency chains only overlap if they are interleaved in the instruction stream (the
    // neuron-by-neuron form cost ~800 cycles per event in the single-ring profile, profiles/r2_edm_single_ring.md)
    // (GS neurons at a time: all NPT with 128 registers, half of them in the register-capped build)
    constexpr int GS = (MINB <= 4) ? NPT : (NPT >= 4 ? NPT / 2 : NPT);
#pragma unroll
    for (int g0 = 0; g0 < NPT; g0 += GS) {
      T rr[GS], d1[GS], ga[GS], gb[GS];
#pragma unroll
      for (int i = 0; i < GS; ++i) { const int q = g0 + i; rr[i] = s[q] * inv_vmI; d1[i] = v[q] - k.vth; }
#pragma unroll
      for (int i = 0; i < GS; ++i) {
        const int q = g0 + i;
        // stage 1: p >= 1 when r >= 1 and p >= r when r < 1 bound g from above with two FP64 operations
        ga[i] = d1[i] + (s[q] - vmI) * (HET ? ibm1[q] : h_ibm1);     // r >= 1
        gb[i] = (d1[i] - s[q]) + vmI;                               // r <  1
      }
#pragma unroll
      for (int i = 0; i < GS; ++i) {
        const int q = g0 + i;
        const unsigned j = tid + q * nthr;
        if (!FULL && j >= N) continue;
        const bool fo = HET ? filt[q] : h_filt;
        const T g_ub = (rr[i] >= one) ? ga[i] : gb[i];
        // margin above the rounding of g_ub's own terms in the run's arithmetic (FP32: ~1e-7 relative)
        const T m1 = sizeof(T) == 4 ? (T)1e-5 * (one + fabs(d1[i]) + fabs(s[q])) : (T)1e-9;
        // r < 0 or NaN: pow() is NaN, the predicate is false; r == 0 and unfiltered neurons go to the exact path
        const bool st1 = fo ? ((rr[i] > (T)0) ? !(g_ub < -m1) : (rr[i] == (T)0)) : true;
        mask |= (st1 ? 1u : 0u) << q;
      }
    }
    // stage 2 and the append for the survivors, one set bit at a time (rarely more than one per thread); the
    // neuron's state is picked with selects, so no per-neuron branch is paid by the warps that sit on a front
    while (mask) {
      const int q = __ffs(mask) - 1;
      mask &= mask - 1;
      T vq = v[0], sq = s[0], b = HET ? bt[0] : hb, iq = HET ? ibm1[0] : h_ibm1;
      bool fo = HET ? filt[0] : h_filt;
#pragma unroll
      for (int i = 1; i < NPT; ++i)
        if (q == i) { vq = v[i]; sq = s[i]; if (HET) { b = bt[i]; iq = ibm1[i]; fo = filt[i]; } }
      const unsigned j = tid + (unsigned)q * nthr;
      const T rr = sq * inv_vmI;
      bool maybe = true, certain = false;
      if (fo && rr > (T)1e-30 && rr < (T)1e30) {
        const float p32 = exp2f(__log2f((float)rr) * (HET ? (float)(one / b) : h_invb32));
        const T p = (T)p32;
        const T g = (vq - k.vth) - vmI * ((b * p - rr) * iq - one);
        const T margin = (T)1e-4 * (one + p);
        maybe = !(g < -margin);
        certain = g > margin;   // the predicate is provably true: no pow() needed either
      }
      if (maybe) {
        const int slot = atomicAdd(&ncand[parity], 1);
        if (slot < (int)cap) {
          cand_v[slot] = vq; cand_s[slot] = sq;
          cand_i[slot] = (int)j | (certain ? (int)0x80000000 : 0);
          if (HET) cand_b[slot] = b;
        }
      }
    }
  };

  // The branchy form of the same test, neuron by neuron: fewer live registers — used by the builds capped at 64-72
  // registers (7-8 rings per SM), where the straight-line form spills inside the loop and loses (measured, round 2:
  // 4.63 vs 3.62 ms per default evaluation; folding the nested tests into one predicate: 3.99 ms; handing the winner's
  // final exponentials to the publishing thread instead of recomputing them: 3.70 ms — both spill more; with 128
  // registers the straight-line form wins, 2.54 vs 2.78 ms per ring).
  auto scan_branchy = [&](int parity) {
#pragma unroll
    for (int q = 0; q < NPT; ++q) {
      const unsigned j = tid + q * nthr;
      if (!FULL && j >= N) continue;
      const T b = HET ? bt[q] : hb;
      const bool fo = HET ? filt[q] : h_filt;
      const T rr = s[q] * inv_vmI;
      bool maybe, certain = false;
      if (!fo) maybe = true;
      else if (rr > (T)0) {
        // stage 1: p >= 1 when r >= 1 and p >= r when r < 1 bound g from above with two FP64
        // operations; whole warps far from the fronts leave here without touching the MUFU path
        const T d1 = v[q] - k.vth;
        const T g_ub = (rr >= one) ? d1 + (s[q] - vmI) * (HET ? ibm1[q] : h_ibm1) : (d1 - s[q]) + vmI;
        // margin above the rounding of g_ub's own terms in the run's arithmetic (FP32: ~1e-7 relative)
        const T m1 = sizeof(T) == 4 ? (T)1e-5 * (one + fabs(d1) + fabs(s[q])) : (T)1e-9;
        if (g_ub < -m1) maybe = false;
        else if (rr > (T)1e-30 && rr < (T)1e30) {
          const float p32 = exp2f(__log2f((float)rr) * (HET ? (float)(one / b) : h_invb32));
          const T p = (T)p32;
          const T g = (v[q] - k.vth) - vmI * ((b * p - rr) * (HET ? ibm1[q] : h_ibm1) - one);
          const T margin = (T)1e-4 * (one + p);
          maybe = !(g < -margin);
          certain = g > margin;   // the predicate is provably true: no pow() needed either
        } else maybe = true;
      } else maybe = (rr == (T)0);  // r < 0 or NaN: pow() is NaN, the predicate is false
      if (maybe) {
        const int slot = atomicAdd(&ncand[parity], 1);
        if (slot < (int)cap) {
          cand_v[slot] = v[q]; cand_s[slot] = s[q];
          cand_i[slot] = (int)j | (certain ? (int)0x80000000 : 0);
          if (HET) cand_b[slot] = b;
        }
      }
    }
  };

  constexpr bool kStraight = (MINB <= 4);
  auto scan = [&](int parity) { if (kStraight) scan_straight(parity); else scan_branchy(parity); };

  // The event message: (dt, idx) and the event-uniform advance coefficients.
  const bool prof = A.profile_nc != 0;
  int prof_ok = 1;
  auto publish = [&](T dt, unsigned idx, bool have_e = false, T e1w = (T)0, T e2w = (T)0) {
    EventMsg<T> m;
    m.last = 0;
    if (prof) {
      // profile map: evolve for exactly T; the event that would overshoot becomes a plain advance
      if (!(t_now + dt <= k.T_end)) { m.last = 1; dt = k.T_end - t_now; have_e = false; }
      else {
        t_now += dt;
        if (++n_events >= 64 * (int)N) { prof_ok = 0; *stop = 1; }
      }
    }
    m.dt = dt; m.idx = idx; m.fallback = 0;
    // (the winner's last Newton iterate evaluated the same exponentials of the same arguments: same bits)
    T e1 = e1w, e2 = e2w;
    if (!have_e) {
      if (!HET) fast_exp_pair(-dt, (one - hb) * dt, etab, e1, e2);
      else e1 = fast_exp(-dt, etab);
    }
    m.e1 = e1;
    m.cA = k.I * (one - e1);
    m.cB = m.e12 = (T)0;
    if (!HET) {
      m.cB = e1 * h_i1mb * (e2 - one);
      m.e12 = e1 * e2;
    }
    *ev = m;
  };

  // Bookkeeping of one event (EventDrivenMap.cu:620-643): which front it belongs to, last-before-T
  // / first-after-T records, loop condition (:601).  It runs one event LATE, on a thread of a warp
  // that would otherwise idle at the barrier while warp 0 runs the next Newton chain; the event
  // that was speculatively resolved meanwhile is simply dropped when the loop condition fails
  // (the state after the last event is never read).
  const unsigned bk_tid = (nwarps > 1) ? 32u : 0u;
  bool pending = false;
  T pend_dt = (T)0;
  unsigned pend_idx = 0;
  auto bookkeep = [&]() {
    t_now += pend_dt;
    n_events++;
    const int idx = (int)pend_idx;
    unsigned mi = 0;
    for (unsigned i = 1; i < Mf; ++i) {  // literal `minIndex += (closer)` — SURVEY Q14
      const int di = abs(idx - last_i[i]);
      const int dm = abs(idx - last_i[mi]);
      mi += (unsigned)(di < dm);
    }
    if (!crossed[mi]) {
      if (t_now > k.T_end) { cross_t[mi] = t_now; cross_i[mi] = idx; crossed[mi] = 1; n_crossed++; }
      else { last_t[mi] = t_now; last_i[mi] = idx; }
    }
    if (!((n_crossed < Mf) && (t_now < 2 * k.T_end))) *stop = 1;  // :601
  };

  int parity = 0;
  scan(parity);
  for (;;) {
    __syncthreads();  // B1: candidate list of this event is complete
    const int n_found = ncand[parity];
    const bool overflow = n_found > (int)cap;   // block-uniform: resolve this event exactly
    const int n = overflow ? 0 : n_found;
    if (tid == 0) ncand[parity ^ 1] = 0;
    if (tid == bk_tid && pending) bookkeep();
    // ---- exact event times of the candidates, compacted into the first warps ----
    const unsigned long long kInf = ~0ull;
    unsigned long long key = kInf;
    unsigned bidx = 0xffffffffu;
    T my_e1 = (T)0, my_e2 = (T)0;
    bool my_ev = false;
    for (int c = (int)tid; c < n; c += (int)nthr) {
      unsigned its = 0;
      const int ci = cand_i[c];
      const T cb = HET ? cand_b[c] : hb;
      const T cv = cand_v[c], cs = cand_s[c];
      T tc = (T)100, ce1 = (T)0, ce2 = (T)0;
      bool cev = false;
      if (ci < 0 || exact_decision<T>(k, cv, cs, cb)) {
        if (kStraight) tc = newton_event_time<T>(k, cv, cs, cb, etab, its, &ce1, &ce2, &cev);
        else tc = newton_event_time<T>(k, cv, cs, cb, etab, its);
      }
      if (A.counters) stat_newton += its;
      const unsigned long long kc = time_key(tc);
      const unsigned ic = (unsigned)(ci & 0x7fffffff);
      if (kc < key || (kc == key && ic < bidx)) { key = kc; bidx = ic; if (kStraight) { my_e1 = ce1; my_e2 = ce2; my_ev = cev; } }
    }
    const bool multi = n > 32;  // block-uniform
    const unsigned long long my_key = key;
    const unsigned my_idx = bidx;
    if (warp == 0 || (multi && warp * 32 < (unsigned)n)) warp_argmin(key, bidx);
    // uncapped build, single-warp case: the lane that owns the winner hands its final exponentials to thread 0
    bool win_e = false;
    T win_e1 = (T)0, win_e2 = (T)0;
    if (kStraight && warp == 0 && !multi) {
      const unsigned owner = __ballot_sync(0xffffffffu, my_key == key && my_idx == bidx && my_ev);
      if (owner) {
        const int src = __ffs(owner) - 1;
        win_e1 = __shfl_sync(0xffffffffu, my_e1, src);
        win_e2 = __shfl_sync(0xffffffffu, my_e2, src);
        win_e = true;
      }
    }
    if (multi) {
      if (lane == 0) { wkey[warp] = (warp * 32 < (unsigned)n) ? key : kInf; widx[warp] = bidx; }
      __syncthreads();
      if (warp == 0) {
        key = (lane < nwarps) ? wkey[lane] : kInf;
        bidx = (lane < nwarps) ? widx[lane] : 0xffffffffu;
        warp_argmin(key, bidx);
      }
    }
    if (tid == 0) {
      if (A.counters) stat_cand += (unsigned)n;
      // all non-candidates sit at exactly 100: if no candidate beats that, the winner is
      // the smallest-index neuron at 100 and must be found by the exact block-wide pass
      if (n == 0 || key >= time_key((T)100)) {
        EventMsg<T> m;
        m.dt = m.e1 = m.cA = m.cB = m.e12 = (T)0; m.idx = 0; m.fallback = 1; m.last = 0;
        *ev = m;
        *fb_key = kInf; *fb_idx = 0xffffffffu;
        stat_fb++;
      } else {
        T dt;
        if (sizeof(T) == 8) dt = (T)__longlong_as_double((long long)key);
        else dt = (T)__uint_as_float((unsigned)key);
        publish(dt, bidx, win_e, win_e1, win_e2);
      }
    }
    __syncthreads();  // B2: event message and the (late) loop condition are visible
    if (*stop) break;
    if (ev->fallback) {
      // exact pass over every neuron (rare: the ring has gone quiet)
      unsigned long long mk = kInf;
      unsigned long long keys[NPT];
#pragma unroll
      for (int q = 0; q < NPT; ++q) {
        const unsigned j = tid + q * nthr;
        keys[q] = kInf;
        if (j < N) {
          unsigned its = 0;
          keys[q] = time_key(exact_event_time<T>(k, v[q], s[q], HET ? bt[q] : hb, etab, its));
          if (keys[q] < mk) mk = keys[q];
        }
      }
      atomicMin(fb_key, mk);
      __syncthreads();
      const unsigned long long gk = *fb_key;
#pragma unroll
      for (int q = 0; q < NPT; ++q) {
        const unsigned j = tid + q * nthr;
        if (j < N && keys[q] == gk) atomicMin(fb_idx, j);
      }
      __syncthreads();
      if (tid == 0) {
        T dt;
        if (sizeof(T) == 8) dt = (T)__longlong_as_double((long long)gk);
        else dt = (T)__uint_as_float((unsigned)gk);
        publish(dt, *fb_idx);
      }
      __syncthreads();
    }
    const EventMsg<T> m = *ev;
    if (tid == bk_tid && !prof) { pending = true; pend_dt = m.dt; pend_idx = m.idx; }
    if (m.last) {  // profile map: no spike, no kick; the state at exactly T is the result
#pragma unroll
      for (int q = 0; q < NPT; ++q) {
        const T e2 = HET ? fast_exp((one - bt[q]) * m.dt, etab) : (T)0;
        const T cB = HET ? m.e1 * (-ibm1[q]) * (e2 - one) : m.cB;
        v[q] = v[q] * m.e1 + (m.cA + s[q] * cB);
        s[q] = s[q] * (HET ? m.e1 * e2 : m.e12);
      }
      break;
    }
    // ---- advance every neuron to the event, reset the firing one, deliver the kick
    //      (EventDrivenMap.cu:612-618), then test who can fire next ----
    parity ^= 1;
    const int rel0 = (int)tid - (int)m.idx;
    if (HET) {
      // one exponential per neuron (its own beta): four neurons at a time, their chains side by side
      constexpr int GE = NPT >= 4 ? 4 : NPT;
#pragma unroll
      for (int g0 = 0; g0 < NPT; g0 += GE) {
        T xe[GE], e2[GE];
#pragma unroll
        for (int i = 0; i < GE; ++i) xe[i] = (one - bt[g0 + i]) * m.dt;
        fast_exp_vec<GE>(xe, etab, e2);
#pragma unroll
        for (int i = 0; i < GE; ++i) {
          const int q = g0 + i;
          const unsigned j = tid + q * nthr;
          if (!FULL && j >= N) continue;
          const unsigned dist = (unsigned)abs(rel0 + q * (int)nthr);
          const T b = bt[q];
          const T cB = m.e1 * (-ibm1[q]) * (e2[i] - one);
          T vn = v[q] * m.e1 + (m.cA + s[q] * cB);
          v[q] = (!(FULL && kStraight) && dist == 0) ? (T)0 : vn;
          s[q] = s[q] * (m.e1 * e2[i]) + b * bw[dist];
        }
      }
    } else {
#pragma unroll
      for (int q = 0; q < NPT; ++q) {
        const unsigned j = tid + q * nthr;
        if (!FULL && j >= N) continue;
        const unsigned dist = (unsigned)abs(rel0 + q * (int)nthr);
        T vn = v[q] * m.e1 + (m.cA + s[q] * m.cB);
        v[q] = (!(FULL && kStraight) && dist == 0) ? (T)0 : vn;
        s[q] = s[q] * m.e12 + bw[dist];
      }
    }
    if (FULL && kStraight) {   // the one neuron that fired: reset outside the straight-line loop (its owner is one thread)
      const unsigned qf = m.idx / nthr;
      if (tid == m.idx - qf * nthr) {
#pragma unroll
        for (int q = 0; q < NPT; ++q) if ((unsigned)q == qf) v[q] = (T)0;
      }
    }
    scan(parity);
  }

  // ---- epilogue: restriction by two-point linear interpolation in time
  //      (RestrictKernel, EventDrivenMap.cu:769-785) and the accept flag (:669-672) ----
  if (prof) {
    // restriction of the profile map: the fine state at time T, sampled back at the coarse knots
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NPT; ++q) {
      const unsigned j = tid + q * nthr;
      if (j < N) { sv[j] = v[q]; ss[j] = s[q]; }
    }
    __syncthreads();
    const unsigned nc = A.profile_nc;
    T* out = A.position + (size_t)blockIdx.x * 2 * nc;
    for (unsigned i = tid; i < nc; i += nthr) {
      const T x = add_rn(-k.L, mul_rn((T)(2 * k.L / nc), (T)i));
      out[i] = periodic_interp<T>(sv, N, k.L, x);
      out[nc + i] = periodic_interp<T>(ss, N, k.L, x);
    }
    if (tid == 0) {
      A.accept[blockIdx.x] = prof_ok;
      A.event_count[blockIdx.x] = n_events;
      if (A.counters) {
        atomicAdd(&A.counters[0], (unsigned long long)n_events);
        atomicAdd(&A.counters[1], (unsigned long long)stat_cand);
        atomicAdd(&A.counters[3], (unsigned long long)stat_fb);
      }
    }
  } else if (tid == bk_tid) {
    const size_t o = (size_t)blockIdx.x;
    for (unsigned m = 0; m < Mf; ++m) {
      const T t0 = last_t[m], t1 = cross_t[m];
      const T x0 = -k.L + (T)2 * k.L / N * last_i[m];
      const T x1 = -k.L + (T)2 * k.L / N * cross_i[m];
      A.position[o * Mf + m] = x0 + (k.T_end - t0) * (x1 - x0) / (t1 - t0);
      if (A.last_index) {
        A.last_index[o * Mf + m] = last_i[m];
        A.crossed_index[o * Mf + m] = cross_i[m];
        A.last_time[o * Mf + m] = t0;
        A.crossed_time[o * Mf + m] = t1;
      }
    }
    A.accept[o] = (n_crossed == Mf) ? 1 : 0;
    A.event_count[o] = n_events;
    if (A.counters) atomicAdd(&A.counters[0], (unsigned long long)n_events);
  }
  if (tid == 0 && A.counters && !prof) {
    atomicAdd(&A.counters[1], (unsigned long long)stat_cand);
    atomicAdd(&A.counters[3], (unsigned long long)stat_fb);
  }
  if (A.counters) {
    // Newton iterations were counted by whichever thread ran them
    unsigned tot = stat_newton;
    for (int off = 16; off > 0; off >>= 1) tot += __shfl_down_sync(0xffffffffu, tot, off);
    if (lane == 0 && tot) atomicAdd(&A.counters[2], (unsigned long long)tot);
  }
}

// ---------------------------------------------------------------- reduce ----
// Masked mean over realisations in a FIXED order (CountRealisationsKernel +
// realisationReductionKernelBlocks, EventDrivenMap.cu:787-824) and the residual
// F = -c U[1..M] - X_T + c T (EventDrivenMap.cu:239).  One CTA per column.
template <typename T>
__global__ void __launch_bounds__(256)
edm_reduce_kernel(unsigned R, unsigned Mf, double T_end, unsigned quirks,
                  const double* __restrict__ z_cols, const T* __restrict__ position,
                  const int32_t* __restrict__ accept, double* __restrict__ f_cols,
                  double* __restrict__ mean_cols) {
  __shared__ T part[256];
  __shared__ unsigned cnt_part[256];
  __shared__ unsigned s_count;
  const unsigned col = blockIdx.x, tid = threadIdx.x;
  const T* pos = position + (size_t)col * R * Mf;
  const int32_t* acc = accept + (size_t)col * R;
  unsigned c = 0;
  for (unsigned rr = tid; rr < R; rr += 256) c += (unsigned)(acc[rr] == 1);
  cnt_part[tid] = c;
  __syncthreads();
  for (unsigned o = 128; o > 0; o >>= 1) {
    if (tid < o) cnt_part[tid] += cnt_part[tid + o];
    __syncthreads();
  }
  if (tid == 0) s_count = cnt_part[0];
  __syncthreads();
  const unsigned count = s_count;
  const double* z = z_cols + (size_t)col * Mf;
  for (unsigned m = 0; m < Mf; ++m) {
    T sum = (T)0;
    for (unsigned rr = tid; rr < R; rr += 256) {
      bool take = acc[rr] == 1;
      if ((quirks & B200_EDM_QUIRK_ACCEPT0_BIAS) && rr == 0) take = (count == 1);
      if (take) sum += pos[(size_t)rr * Mf + m];
    }
    part[tid] = sum;
    __syncthreads();
    for (unsigned o = 128; o > 0; o >>= 1) {
      if (tid < o) part[tid] += part[tid + o];
      __syncthreads();
    }
    if (tid == 0) {
      const T mean = part[0] / count;
      const double Um = (m == 0) ? 0.0 : z[m];
      f_cols[(size_t)col * Mf + m] = (-z[0]) * Um - (double)mean + z[0] * T_end;
      if (mean_cols) mean_cols[(size_t)col * Mf + m] = (double)mean;
    }
    __syncthreads();
  }
}

template <typename T, typename U>
__global__ void convert_kernel(const T* __restrict__ in, U* __restrict__ out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (U)in[i];
}

// ---------------------------------------------------------------- finite differences ----
// The callers' column loop (NewtonSolver.cpp:181-195, Stability.cpp:95-109) formed on the device:
// local column k < ncols_pert is u + eps e_{col_begin+k} (one rounded add, as `du(i) += epsilon`),
// the last local column is u itself (the base evaluation every device repeats).
__global__ void edm_fd_columns_kernel(const double* __restrict__ u, unsigned n, double eps, unsigned col_begin,
                                      unsigned ncols_pert, double* __restrict__ z, unsigned with_base) {
  const size_t total = (size_t)(ncols_pert + with_base) * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const unsigned k = (unsigned)(i / n), r = (unsigned)(i % n);
    double v = u[r];
    if (k < ncols_pert && r == col_begin + k) v = __dadd_rn(v, eps);
    z[i] = v;
  }
}
// jacobian.col(i) = (df - f) * pow(epsilon,-1)  (NewtonSolver.cpp:194, Stability.cpp:108); f = local column ncols_pert,
// or f0_given when the caller already holds F(u) (NewtonSolver.cpp:110 computes it before the Jacobian)
__global__ void edm_fd_jacobian_kernel(const double* __restrict__ f, unsigned n, unsigned ncols_pert, double inv_eps,
                                       double* __restrict__ jac, const double* __restrict__ f0_given) {
  const size_t total = (size_t)ncols_pert * n;
  const double* f0 = f0_given ? f0_given : f + (size_t)ncols_pert * n;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    jac[i] = __dmul_rn(__dsub_rn(f[i], f0[i % n]), inv_eps);
}

}  // namespace
}  // namespace b200

using namespace b200;

// ---------------------------------------------------------------- handle ----
struct b200_edm {
  std::vector<double> params;
  b200_edm_model model;
  uint32_t R, N, Mf;
  b200_dtype prec;
  double sigma = 0.0;
  uint64_t seed = 42;
  int debug = 0, timing = 0, npt = 0;
  uint32_t profile_nc = 0;   // 0: front map; > 0: profile map on this many coarse knots
  // in-process multi-GPU: helper handles on other devices of this process (b200_edm_set_devices)
  std::vector<b200_edm*> helpers;
  std::vector<int> devs;             // devs[0] = this handle's device, then the helpers'
  std::vector<ncclComm_t> comms;     // one communicator per device (ncclCommInitAll); empty: peer copies
  void* d_gather = nullptr;          // all-gather buffer (every device holds the full result)
  size_t gather_cap = 0;
  int32_t* d_gather_acc = nullptr;
  size_t gather_acc_cap = 0;
  double* d_u = nullptr;             // base vector of a finite-difference Jacobian
  size_t u_cap = 0;
  double* d_jac = nullptr;           // item-sharded Jacobian: difference quotients formed on the primary
  size_t jac_cap = 0;
  bool last_sliced = false;          // the last evaluation left only a slice of the per-item arrays here
  bool last_pos_external = false;
  cudaEvent_t ev_helper = nullptr;
  void* d_uc = nullptr;      // profile map: columns converted to the run's arithmetic type
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_up = nullptr, ev_done = nullptr;
  bool up_pending = false;
  cudaStream_t last_stream = nullptr;
  bool done_pending = false;
  // ensemble-level device state
  void* w = nullptr;
  void* beta = nullptr;
  bool w_dirty = true, beta_dirty = true;
  // batch-level device state (capacity in columns / items)
  size_t cap_cols = 0, cap_items = 0;
  double* d_z = nullptr;
  double* d_f = nullptr;
  double* d_mean = nullptr;
  int32_t* d_init = nullptr;
  int32_t* d_clamped = nullptr;
  void* d_lv = nullptr;
  void* d_ls = nullptr;
  void* d_pos = nullptr;
  int32_t* d_accept = nullptr;
  int32_t* d_evcount = nullptr;
  int32_t* d_last_i = nullptr;
  int32_t* d_cross_i = nullptr;
  void* d_last_t = nullptr;
  void* d_cross_t = nullptr;
  unsigned long long* d_counters = nullptr;
  double* h_pin = nullptr;  // pinned staging for z in / f out
  size_t h_pin_cap = 0;
  // last call
  size_t last_cols = 0;
  double last_ms = 0.0;
  unsigned long long last_counters[4] = {0, 0, 0, 0};
  int last_clamped = 0;
  char err[256] = "";
};

namespace {

size_t esize(const b200_edm* h) { return h->prec == B200_F64 ? 8 : 4; }
// length of the coarse vector: fronts (reference map) or 2 x coarse knots (profile map)
size_t ndim(const b200_edm* h) { return h->profile_nc ? 2 * (size_t)h->profile_nc : (size_t)h->Mf; }

template <typename T>
Consts<T> make_consts(const b200_edm* h) {
  Consts<T> k;
  k.vth = (T)h->model.vth; k.a1 = (T)h->model.a1; k.a2 = (T)h->model.a2;
  k.b1 = (T)h->model.b1; k.b2 = (T)h->model.b2; k.I = (T)h->model.I; k.L = (T)h->model.L;
  k.T_end = (T)h->model.time_horizon; k.tol = h->model.tol; k.counter_max = h->model.counter_max;
  return k;
}

void free_ensemble(b200_edm* h) {
  cudaFree(h->w); cudaFree(h->beta);
  h->w = h->beta = nullptr;
  h->w_dirty = h->beta_dirty = true;
}
void free_batch(b200_edm* h) {
  cudaFree(h->d_uc); h->d_uc = nullptr;
  cudaFree(h->d_z); cudaFree(h->d_f); cudaFree(h->d_mean); cudaFree(h->d_init); cudaFree(h->d_lv);
  cudaFree(h->d_ls); cudaFree(h->d_pos); cudaFree(h->d_accept); cudaFree(h->d_evcount);
  cudaFree(h->d_last_i); cudaFree(h->d_cross_i); cudaFree(h->d_last_t); cudaFree(h->d_cross_t);
  h->d_z = h->d_f = h->d_mean = nullptr; h->d_init = nullptr; h->d_lv = h->d_ls = h->d_pos = nullptr;
  h->d_accept = h->d_evcount = h->d_last_i = h->d_cross_i = nullptr; h->d_last_t = h->d_cross_t = nullptr;
  h->cap_cols = h->cap_items = 0;
}

int ensure_pinned(b200_edm* h, size_t doubles) {
  if (doubles <= h->h_pin_cap) return B200_OK;
  if (h->h_pin) cudaFreeHost(h->h_pin);
  h->h_pin = nullptr; h->h_pin_cap = 0;
  B200_CUDA(cudaHostAlloc((void**)&h->h_pin, doubles * sizeof(double), cudaHostAllocDefault));
  h->h_pin_cap = doubles;
  return B200_OK;
}

int ensure_batch(b200_edm* h, size_t ncols, size_t nitems) {
  const size_t es = esize(h), N = h->N, Mf = ndim(h);
  const bool prof = h->profile_nc != 0;
  if (ncols > h->cap_cols) {
    cudaFree(h->d_z); cudaFree(h->d_f); cudaFree(h->d_mean); cudaFree(h->d_init); cudaFree(h->d_lv); cudaFree(h->d_ls);
    cudaFree(h->d_uc); h->d_uc = nullptr;
    h->d_z = h->d_f = h->d_mean = nullptr; h->d_init = nullptr; h->d_lv = h->d_ls = nullptr; h->cap_cols = 0;
    if (prof) B200_CUDA(cudaMalloc(&h->d_uc, ncols * Mf * es));
    B200_CUDA(cudaMalloc(&h->d_z, ncols * Mf * sizeof(double)));
    B200_CUDA(cudaMalloc(&h->d_f, ncols * Mf * sizeof(double)));
    B200_CUDA(cudaMalloc(&h->d_mean, ncols * Mf * sizeof(double)));
    B200_CUDA(cudaMalloc(&h->d_init, ncols * Mf * sizeof(int32_t)));
    B200_CUDA(cudaMalloc(&h->d_lv, ncols * N * es));
    B200_CUDA(cudaMalloc(&h->d_ls, ncols * N * es));
    h->cap_cols = ncols;
  }
  if (nitems > h->cap_items) {
    cudaFree(h->d_pos); cudaFree(h->d_accept); cudaFree(h->d_evcount); cudaFree(h->d_last_i);
    cudaFree(h->d_cross_i); cudaFree(h->d_last_t); cudaFree(h->d_cross_t);
    h->d_pos = nullptr; h->d_accept = h->d_evcount = h->d_last_i = h->d_cross_i = nullptr;
    h->d_last_t = h->d_cross_t = nullptr; h->cap_items = 0;
    B200_CUDA(cudaMalloc(&h->d_pos, nitems * Mf * es));
    B200_CUDA(cudaMalloc(&h->d_accept, nitems * sizeof(int32_t)));
    B200_CUDA(cudaMalloc(&h->d_evcount, nitems * sizeof(int32_t)));
    if (!prof) {  // front records exist only for the reference map
      B200_CUDA(cudaMalloc(&h->d_last_i, nitems * Mf * sizeof(int32_t)));
      B200_CUDA(cudaMalloc(&h->d_cross_i, nitems * Mf * sizeof(int32_t)));
      B200_CUDA(cudaMalloc(&h->d_last_t, nitems * Mf * es));
      B200_CUDA(cudaMalloc(&h->d_cross_t, nitems * Mf * es));
    }
    h->cap_items = nitems;
  }
  if (!h->d_clamped) B200_CUDA(cudaMalloc(&h->d_clamped, sizeof(int32_t)));
  if (!h->d_counters) B200_CUDA(cudaMalloc(&h->d_counters, 4 * sizeof(unsigned long long)));
  return B200_OK;
}

// (re)build the coupling kernel and the beta ensemble when their inputs changed
template <typename T>
int ensure_ensemble(b200_edm* h, cudaStream_t st) {
  if (h->w_dirty) {
    cudaFree(h->w); h->w = nullptr;
    B200_CUDA(cudaMalloc(&h->w, (size_t)h->N * sizeof(T)));
    edm_coupling_kernel<T><<<(h->N + 255) / 256, 256, 0, B200_CNT(st)>>>(make_consts<T>(h), h->N, (T*)h->w);
    B200_CUDA(cudaGetLastError());
    h->w_dirty = false;
  }
  if (h->sigma != 0.0) {
    if (h->beta_dirty) {
      cudaFree(h->beta); h->beta = nullptr;
      const size_t n = (size_t)h->R * h->N;
      B200_CUDA(cudaMalloc(&h->beta, n * sizeof(T)));
      edm_beta_kernel<T><<<(unsigned)((n + 255) / 256), 256, 0, B200_CNT(st)>>>((T*)h->beta, n, h->params[0], h->sigma, h->seed);
      B200_CUDA(cudaGetLastError());
      h->beta_dirty = false;
    }
  }
  return B200_OK;
}

int pick_npt(const b200_edm* h) {
  if (h->npt > 0) return h->npt;
  const unsigned N = h->N;
  if (N <= 512) return 4;
  if (N <= 2048) return 8;
  return 16;
}

// 128-thread CTAs, 7 resident per SM (72 registers): the default ensemble (1000 rings = 6.8 per SM) is one wave,
// and the kernel does not spill (at 8 per SM = 64 registers it spilled 444 / 1196 bytes, homogeneous / heterogeneous)
constexpr int kRingsPerSm = 7;

template <typename T, int NPT, bool HET>
int launch_evolve_npt(b200_edm* h, const EvolveArgs<T>& A, size_t nitems, cudaStream_t st) {
  unsigned threads = (h->N + NPT - 1) / NPT;
  threads = (threads + 31) / 32 * 32;
  if (threads > 1024) return fail(B200_ERR_UNSUPPORTED, "no_neurons=%u needs more than 1024 threads at %d neurons/thread", h->N, NPT);
  const size_t smem = evolve_smem_bytes<T>(h->N, A.Mf, HET, h->profile_nc != 0);
  if (smem > 227 * 1024) return fail(B200_ERR_UNSUPPORTED, "no_neurons=%u / no_fronts=%u need %zu B of shared memory (max 232448)", h->N, h->Mf, smem);
  auto go = [&](auto kern) -> int {
    B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)nitems, threads, smem, B200_CNT(st)>>>(A);
    return B200_OK;
  };
  // 128-thread CTAs capped at 64 registers: 8 rings resident per SM, i.e. 8 serial Newton
  // chains overlapping (measured: 5.9 -> 4.5 ms per default evaluation vs 4 rings at 118 regs)
  const bool full = (h->N == threads * (unsigned)NPT);  // no ragged tail: bounds checks compiled out
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
  if (threads <= 128) {
    // Few rings (one wave even at 4 per SM): the uncapped build (116 registers, no spills) has the shorter
    // serial chain — 2.34 instead of 2.81 ms for a default ring (profiles/edm_evolve_r1.md).
    bool done = false;
    if constexpr (NPT == 8) {   // (only the default 8 neurons/thread gets the second build: compile time)
      if (full && nitems <= (size_t)sms * 4) { B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 128, 4, true>)); done = true; }
      // front map with several waves of rings (a Jacobian batch: 4000 rings): 8 per SM at 64 registers moves more
      // rings per second than 7 at 72 (13.4 vs 14.3 ms); one wave (the default ensemble) and the profile map are
      // faster at 7 (3.62 vs 3.68 ms; 734 vs 787 ms) — measured, round 2
      else if (full && !h->profile_nc && nitems > (size_t)sms * kRingsPerSm) { B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 128, 8, true>)); done = true; }
    }
    if (done) {}
    else if (full) B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 128, kRingsPerSm, true>));
    else B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 128, kRingsPerSm, false>));
  } else if (threads <= 256) {
    B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 256, 2, false>));
  } else {
    B200_TRY(go(edm_evolve_kernel<T, NPT, HET, 1024, 1, false>));
  }
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

template <typename T, bool HET>
int launch_evolve(b200_edm* h, const EvolveArgs<T>& A, size_t nitems, cudaStream_t st) {
  switch (pick_npt(h)) {
    case 4: return launch_evolve_npt<T, 4, HET>(h, A, nitems, st);
    case 8: return launch_evolve_npt<T, 8, HET>(h, A, nitems, st);
    case 16: return launch_evolve_npt<T, 16, HET>(h, A, nitems, st);
    default: return fail(B200_ERR_INVALID_ARG, "neurons per thread must be 4, 8 or 16");
  }
}

// prepare (lift) for ncols columns whose z already sits in h->d_z
template <typename T>
int run_prepare(b200_edm* h, size_t ncols, cudaStream_t st) {
  B200_CUDA(cudaMemsetAsync(h->d_clamped, 0, sizeof(int32_t), st));
  if (h->profile_nc) {
    edm_profile_lift_kernel<T><<<(unsigned)ncols, 256, 0, B200_CNT(st)>>>(make_consts<T>(h), h->N, h->profile_nc, h->d_z,
                                                                (T*)h->d_uc, (T*)h->d_lv, (T*)h->d_ls);
    B200_CUDA(cudaGetLastError());
    return B200_OK;
  }
  const size_t smem = sizeof(FrontCoef<T>) * h->Mf;
  if (smem > 200 * 1024) return fail(B200_ERR_UNSUPPORTED, "no_fronts=%u too large for the lift kernel", h->Mf);
  auto kern = edm_prepare_kernel<T>;
  B200_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)ncols, 256, smem, B200_CNT(st)>>>(make_consts<T>(h), h->N, h->Mf, (T)h->params[0], h->d_z,
                                           h->d_init, h->d_clamped, (T*)h->d_lv, (T*)h->d_ls);
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

// evolve items [item_begin, item_end) into pos/accept (local item order)
template <typename T>
int run_evolve(b200_edm* h, size_t item_begin, size_t item_end, T* pos, int32_t* accept, cudaStream_t st) {
  EvolveArgs<T> A;
  A.k = make_consts<T>(h);
  A.N = h->N; A.R = h->R; A.Mf = h->profile_nc ? 0 : h->Mf;
  A.profile_nc = h->profile_nc;
  A.beta_mean = (T)h->params[0];
  A.beta = (h->sigma != 0.0) ? (const T*)h->beta : nullptr;
  A.w = (const T*)h->w;
  A.lift_v = (const T*)h->d_lv; A.lift_s = (const T*)h->d_ls;
  A.init_index = h->d_init;
  A.item_begin = item_begin;
  A.position = pos; A.accept = accept; A.event_count = h->d_evcount;
  A.last_index = h->profile_nc ? nullptr : h->d_last_i; A.crossed_index = h->d_cross_i;
  A.last_time = (T*)h->d_last_t; A.crossed_time = (T*)h->d_cross_t;
  A.counters = (h->debug || h->timing) ? h->d_counters : nullptr;
  const size_t nitems = item_end - item_begin;
  if (nitems == 0) return B200_OK;
  if (nitems > 0x7fffffffull) return fail(B200_ERR_UNSUPPORTED, "too many work items in one launch");
  if (A.counters) B200_CUDA(cudaMemsetAsync(h->d_counters, 0, 4 * sizeof(unsigned long long), st));
  if (h->timing) B200_CUDA(cudaEventRecord(h->ev0, st));
  int rc = (h->sigma != 0.0) ? launch_evolve<T, true>(h, A, nitems, st) : launch_evolve<T, false>(h, A, nitems, st);
  if (rc != B200_OK) return rc;
  if (h->timing) B200_CUDA(cudaEventRecord(h->ev1, st));
  return B200_OK;
}

template <typename T>
int run_reduce(b200_edm* h, size_t ncols, const T* pos, const int32_t* accept, double* f_cols, cudaStream_t st) {
  if (h->profile_nc) {
    const size_t n = ndim(h), total = ncols * n;
    edm_profile_reduce_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, B200_CNT(st)>>>(h->R, (unsigned)n, ncols, h->d_z, pos, accept, f_cols);
    B200_CUDA(cudaGetLastError());
    return B200_OK;
  }
  edm_reduce_kernel<T><<<(unsigned)ncols, 256, 0, B200_CNT(st)>>>(h->R, h->Mf, (double)(T)h->model.time_horizon,
                                                        h->model.quirks, h->d_z, pos, accept, f_cols, h->d_mean);
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

// The handle's buffers are shared by every call: work issued on a different stream than the
// previous call first waits for that call's tail.
int order_after_previous(b200_edm* h, cudaStream_t st) {
  if (h->done_pending && st != h->last_stream) B200_CUDA(cudaStreamWaitEvent(st, h->ev_done, 0));
  return B200_OK;
}
int mark_done(b200_edm* h, cudaStream_t st) {
  B200_CUDA(cudaEventRecord(h->ev_done, st));
  h->last_stream = st;
  h->done_pending = true;
  return B200_OK;
}

int check_handle(const b200_edm* h, const char* fn) {
  if (!h) return fail(B200_ERR_INVALID_ARG, "%s: NULL handle", fn);
  return B200_OK;
}

int upload_z(b200_edm* h, const double* z_cols, size_t n, size_t ncols, cudaStream_t st) {
  if (n != ndim(h))
    return fail(B200_ERR_INVALID_ARG, "vector length %zu != %s %zu", n, h->profile_nc ? "2 x coarse knots" : "no_fronts", ndim(h));
  if (!h->profile_nc)
    for (size_t c = 0; c < ncols; ++c)
      if (!(z_cols[c * n] == z_cols[c * n]) || z_cols[c * n] == 0.0)
        return fail(B200_ERR_INVALID_ARG, "column %zu: wave speed z[0] must be finite and non-zero", c);
  // the pinned staging block is reused: wait for the previous upload to have left it
  if (h->up_pending) { B200_CUDA(cudaEventSynchronize(h->ev_up)); h->up_pending = false; }
  B200_TRY(ensure_pinned(h, 2 * n * ncols));
  memcpy(h->h_pin, z_cols, n * ncols * sizeof(double));
  B200_CUDA(cudaMemcpyAsync(h->d_z, h->h_pin, n * ncols * sizeof(double), cudaMemcpyHostToDevice, st));
  B200_CUDA(cudaEventRecord(h->ev_up, st));
  h->up_pending = true;
  return B200_OK;
}

// copy everything that defines the map from the primary handle to a helper on another device
void sync_helper(const b200_edm* h, b200_edm* g) {
  if (g->params != h->params || g->sigma != h->sigma || g->seed != h->seed || g->R != h->R || g->N != h->N) g->beta_dirty = true;
  if (g->N != h->N || memcmp(&g->model, &h->model, sizeof(h->model)) != 0) g->w_dirty = true;
  if (g->R != h->R || g->N != h->N || g->Mf != h->Mf || g->profile_nc != h->profile_nc) { cudaSetDevice(g->device); free_batch(g); }
  g->params = h->params; g->model = h->model; g->R = h->R; g->N = h->N; g->Mf = h->Mf; g->prec = h->prec;
  g->sigma = h->sigma; g->seed = h->seed; g->npt = h->npt; g->profile_nc = h->profile_nc;
  g->debug = 0; g->timing = 0;
}

// ---- NCCL, loaded on first use (the library has no link-time dependency on it) ----
struct NcclApi {
  void* so = nullptr;
  decltype(&ncclCommInitAll) comm_init_all = nullptr;
  decltype(&ncclCommDestroy) comm_destroy = nullptr;
  decltype(&ncclAllGather) all_gather = nullptr;
  decltype(&ncclGroupStart) group_start = nullptr;
  decltype(&ncclGroupEnd) group_end = nullptr;
  decltype(&ncclGetErrorString) error_string = nullptr;
  bool tried = false, ok = false;
};
NcclApi g_nccl;
bool load_nccl() {
  NcclApi& a = g_nccl;
  if (a.tried) return a.ok;
  a.tried = true;
  for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
    a.so = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
    if (a.so) break;
  }
  if (!a.so) return false;
#define B200_SYM(field, sym) a.field = (decltype(a.field))dlsym(a.so, #sym); if (!a.field) return false
  B200_SYM(comm_init_all, ncclCommInitAll);
  B200_SYM(comm_destroy, ncclCommDestroy);
  B200_SYM(all_gather, ncclAllGather);
  B200_SYM(group_start, ncclGroupStart);
  B200_SYM(group_end, ncclGroupEnd);
  B200_SYM(error_string, ncclGetErrorString);
#undef B200_SYM
  return a.ok = true;
}
#define B200_NCCL(call)                                                                            \
  do {                                                                                             \
    ncclResult_t r__ = (call);                                                                     \
    if (r__ != ncclSuccess) return fail(B200_ERR_CUDA, "NCCL error %d (%s) in %s", (int)r__, g_nccl.error_string(r__), #call); \
  } while (0)

b200_edm* dev_handle(b200_edm* h, size_t d) { return d == 0 ? h : h->helpers[d - 1]; }

int ensure_gather(b200_edm* g, size_t bytes, size_t acc_items) {
  if (bytes > g->gather_cap) {
    cudaFree(g->d_gather); g->d_gather = nullptr; g->gather_cap = 0;
    B200_CUDA(cudaMalloc(&g->d_gather, bytes));
    g->gather_cap = bytes;
  }
  if (acc_items > g->gather_acc_cap) {
    cudaFree(g->d_gather_acc); g->d_gather_acc = nullptr; g->gather_acc_cap = 0;
    B200_CUDA(cudaMalloc(&g->d_gather_acc, acc_items * sizeof(int32_t)));
    g->gather_acc_cap = acc_items;
  }
  return B200_OK;
}
int ensure_u(b200_edm* g, size_t n) {
  if (n > g->u_cap) {
    cudaFree(g->d_u); g->d_u = nullptr; g->u_cap = 0;
    B200_CUDA(cudaMalloc(&g->d_u, n * sizeof(double)));
    g->u_cap = n;
  }
  return B200_OK;
}

// every device holds `slot_bytes` of results at slot d of its gather buffer: exchange them so that every
// device (in particular the primary) holds all slots.  One in-place ncclAllGather per device inside one
// group (single process driving several devices; b200_edm_set_devices created the communicators).
int exchange_slots(b200_edm* h, cudaStream_t st, size_t slot_bytes, size_t acc_slot_items) {
  const size_t ndev = h->helpers.size() + 1;
  NvtxRange nvtx("edm:nccl_all_gather");
  B200_NCCL(g_nccl.group_start());
  ncclResult_t bad = ncclSuccess;   // a failed call must not leave the thread inside an open group
  for (size_t d = 0; d < ndev && bad == ncclSuccess; ++d) {
    b200_edm* g = dev_handle(h, d);
    cudaStream_t gs = d == 0 ? st : g->stream;
    if (slot_bytes)
      bad = g_nccl.all_gather((const char*)g->d_gather + d * slot_bytes, g->d_gather, slot_bytes, ncclChar, h->comms[d], gs);
    if (acc_slot_items && bad == ncclSuccess)
      bad = g_nccl.all_gather(g->d_gather_acc + d * acc_slot_items, g->d_gather_acc, acc_slot_items, ncclInt32, h->comms[d], gs);
  }
  const ncclResult_t end = g_nccl.group_end();
  if (bad != ncclSuccess) return fail(B200_ERR_CUDA, "NCCL error %d (%s) in ncclAllGather", (int)bad, g_nccl.error_string(bad));
  if (end != ncclSuccess) return fail(B200_ERR_CUDA, "NCCL error %d (%s) in ncclGroupEnd", (int)end, g_nccl.error_string(end));
  return B200_OK;
}

// One batch of evaluations over all devices of the handle (1 = just this one).
//   fd == false: z_or_u = n x ncols host columns; result = F of every column.
//   fd == true : z_or_u = u (n entries); the ncols = n perturbed columns u + eps e_i are formed on the
//                device; result = the Jacobian columns (F(u + eps e_i) - F(u)) / eps and F(u).
// Sharding (SURVEY 8e): with many columns every device owns a contiguous block of WHOLE columns
// (lift, evolve, fixed-order reduction and, for fd, the difference quotient all local; the base column is
// evaluated redundantly on every device) and only the n-vectors per column are all-gathered.  With few
// columns (the reference's n = 3) the (column, realisation) work items are split instead, positions and
// accept flags are all-gathered and the primary reduces.  Either way the result is bitwise that of one device.
template <typename T>
int compute_multi(b200_edm* h, const double* z_or_u, size_t n, size_t ncols, bool fd, double eps, double* out_cols,
                  double* f0_out, const double* f0_in = nullptr) {
  DeviceScope callers_device(-1);   // the loop below switches devices; the caller gets its own back on every exit
  B200_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  const size_t ndev = h->helpers.size() + 1, R = h->R, nd = ndim(h), es = esize(h);
  if (n != nd)
    return fail(B200_ERR_INVALID_ARG, "vector length %zu != %s %zu", n, h->profile_nc ? "2 x coarse knots" : "no_fronts", nd);
  B200_TRY(order_after_previous(h, st));
  if (h->up_pending) { B200_CUDA(cudaEventSynchronize(h->ev_up)); h->up_pending = false; }
  B200_TRY(ensure_pinned(h, 2 * n * (ncols + 1)));     // z / u in, results out (never re-allocated below)
  const bool by_columns = ndev == 1 || ncols >= 4 * ndev;
  const size_t cpd = by_columns ? (ncols + ndev - 1) / ndev : ncols;          // result columns per device slot
  const size_t base = (fd && !f0_in) ? 1 : 0;   // the base evaluation F(u) rides along unless the caller already holds it
  const size_t nitems_all = (ncols + base) * R;
  const size_t per = (nitems_all + ndev - 1) / ndev;                            // item mode: items per device
  h->last_sliced = ndev > 1;
  h->last_pos_external = false;

  for (size_t dd = 0; dd < ndev; ++dd) {
    const size_t d = ndev - 1 - dd;            // helpers first: they run while the primary is being fed
    b200_edm* g = dev_handle(h, d);
    cudaStream_t gs = d == 0 ? st : g->stream;
    if (d) sync_helper(h, g);
    B200_CUDA(cudaSetDevice(g->device));
    // local column set
    size_t c_lo = 0, c_hi = ncols;
    if (by_columns) { c_lo = d * cpd < ncols ? d * cpd : ncols; c_hi = (d + 1) * cpd < ncols ? (d + 1) * cpd : ncols; }
    const size_t cols_res = c_hi - c_lo;                       // result columns computed here
    const size_t cols_loc = cols_res + base;                   // + the base column
    size_t i_lo = 0, i_hi = cols_loc * R;
    if (!by_columns) { i_lo = d * per < nitems_all ? d * per : nitems_all; i_hi = (d + 1) * per < nitems_all ? (d + 1) * per : nitems_all; }
    B200_TRY(ensure_batch(g, cols_loc > cpd + 1 ? cols_loc : cpd + 1, (i_hi - i_lo) ? (i_hi - i_lo) : 1));
    B200_TRY(ensure_ensemble<T>(g, gs));
    if (by_columns) B200_TRY(ensure_gather(g, ndev * cpd * nd * sizeof(double), 0));
    else B200_TRY(ensure_gather(g, ndev * per * nd * es, ndev * per));
    if (cols_res == 0 && by_columns) continue;                 // more devices than columns: idle, still joins the gather
    {
    NvtxRange nvtx("edm:lift");
    if (fd) {
      B200_TRY(ensure_u(g, 2 * n));                            // u, then the caller's F(u) if given
      if (g->up_pending) { B200_CUDA(cudaEventSynchronize(g->ev_up)); g->up_pending = false; }
      B200_TRY(ensure_pinned(g, 2 * n));
      memcpy(g->h_pin, z_or_u, n * sizeof(double));
      if (f0_in) memcpy(g->h_pin + n, f0_in, n * sizeof(double));
      B200_CUDA(cudaMemcpyAsync(g->d_u, g->h_pin, (f0_in ? 2 : 1) * n * sizeof(double), cudaMemcpyHostToDevice, gs));
      B200_CUDA(cudaEventRecord(g->ev_up, gs));
      g->up_pending = true;
      const size_t total = cols_loc * n;
      edm_fd_columns_kernel<<<(unsigned)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184), 256, 0, B200_CNT(gs)>>>(
          g->d_u, (unsigned)n, eps, (unsigned)c_lo, (unsigned)cols_res, g->d_z, (unsigned)base);
      B200_CUDA(cudaGetLastError());
    } else {
      B200_TRY(upload_z(g, z_or_u + c_lo * n, n, cols_loc, gs));
    }
    B200_TRY(run_prepare<T>(g, cols_loc, gs));
    }
    {
      NvtxRange nvtx("edm:evolve");
      if (by_columns) {
        B200_TRY(run_evolve<T>(g, 0, cols_loc * R, (T*)g->d_pos, g->d_accept, gs));
      } else {
        B200_TRY(run_evolve<T>(g, i_lo, i_hi, (T*)((char*)g->d_gather + d * per * nd * es), g->d_gather_acc + d * per, gs));
      }
    }
    if (by_columns) {
      NvtxRange nvtx("edm:reduce");
      double* slot = (double*)g->d_gather + d * cpd * nd;
      if (fd) {
        B200_TRY(run_reduce<T>(g, cols_loc, (const T*)g->d_pos, g->d_accept, g->d_f, gs));
        const size_t total = cols_res * n;
        edm_fd_jacobian_kernel<<<(unsigned)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184), 256, 0, B200_CNT(gs)>>>(
            g->d_f, (unsigned)n, (unsigned)cols_res, pow(eps, -1), slot, f0_in ? g->d_u + n : nullptr);
        B200_CUDA(cudaGetLastError());
      } else {
        B200_TRY(run_reduce<T>(g, cols_loc, (const T*)g->d_pos, g->d_accept, slot, gs));
      }
    }
  }
  B200_CUDA(cudaSetDevice(h->device));
  if (ndev > 1) {
    if (by_columns) B200_TRY(exchange_slots(h, st, cpd * nd * sizeof(double), 0));
    else B200_TRY(exchange_slots(h, st, per * nd * es, per));
    B200_CUDA(cudaSetDevice(h->device));
  }
  const double* d_result = (const double*)h->d_gather;
  const double* d_f0 = nullptr;
  if (by_columns) {
    if (base) d_f0 = h->d_f + (((cpd < ncols ? cpd : ncols)) * n);   // the primary's base column (local column cols_res)
  } else {
    // item mode: all positions are here in item order; the usual fixed-order reduction over every column
    NvtxRange nvtx("edm:reduce");
    B200_TRY(run_reduce<T>(h, ncols + base, (const T*)h->d_gather, h->d_gather_acc, h->d_f, st));
    if (fd) {
      const size_t total = ncols * n;
      if (total > h->jac_cap) {
        cudaFree(h->d_jac); h->d_jac = nullptr; h->jac_cap = 0;
        B200_CUDA(cudaMalloc(&h->d_jac, total * sizeof(double)));
        h->jac_cap = total;
      }
      edm_fd_jacobian_kernel<<<(unsigned)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184), 256, 0, B200_CNT(st)>>>(
          h->d_f, (unsigned)n, (unsigned)ncols, pow(eps, -1), h->d_jac, f0_in ? h->d_u + n : nullptr);
      B200_CUDA(cudaGetLastError());
      d_result = h->d_jac;
      if (base) d_f0 = h->d_f + ncols * n;
    } else {
      d_result = h->d_f;
    }
  }
  double* h_res = h->h_pin + n * (ncols + 1);
  B200_CUDA(cudaMemcpyAsync(h_res, d_result, n * ncols * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (d_f0) B200_CUDA(cudaMemcpyAsync(h->h_pin, d_f0, n * sizeof(double), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaMemcpyAsync(&h->last_clamped, h->d_clamped, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (h->debug || h->timing)
    B200_CUDA(cudaMemcpyAsync(h->last_counters, h->d_counters, sizeof(h->last_counters), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  for (size_t d = 1; d < ndev; ++d) {   // helpers have nothing left in flight that the caller's next call could race with
    B200_CUDA(cudaSetDevice(h->helpers[d - 1]->device));
    B200_CUDA(cudaStreamSynchronize(h->helpers[d - 1]->stream));
  }
  B200_CUDA(cudaSetDevice(h->device));
  h->done_pending = false;
  memcpy(out_cols, h_res, n * ncols * sizeof(double));
  if (f0_out && d_f0) memcpy(f0_out, h->h_pin, n * sizeof(double));
  else if (f0_out && f0_in) memcpy(f0_out, f0_in, n * sizeof(double));
  h->last_cols = by_columns ? (cpd < ncols ? cpd : ncols) + base : ncols + base;
  if (h->timing) {
    float ms = 0.f;
    B200_CUDA(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->last_ms = ms;
  }
  return B200_OK;
}

template <typename T>
int compute_batch(b200_edm* h, const double* z_cols, size_t n, size_t ncols, double* f_out) {
  return compute_multi<T>(h, z_cols, n, ncols, false, 0.0, f_out, nullptr);
}

}  // namespace

extern "C" {

void b200_edm_model_default(b200_edm_model* m) {
  if (!m) return;
  // parameters.hpp:1-15; float literals widened exactly
  m->vth = (double)1.0f; m->a1 = (double)11.0f; m->a2 = (double)7.0f; m->b1 = (double)5.0f;
  m->b2 = (double)3.5f; m->I = (double)0.9f; m->L = (double)3.0f; m->tol = 1e-6;
  m->time_horizon = (double)5.0f; m->counter_max = 100; m->quirks = 0;
}

int b200_edm_create(const double* params, size_t nparams, uint32_t no_realisations,
                    uint32_t no_neurons, uint32_t no_fronts, b200_dtype precision, b200_edm** handle) {
  if (!params || nparams < 1 || !handle) return fail(B200_ERR_INVALID_ARG, "edm_create: NULL / empty argument");
  if (precision != B200_F64 && precision != B200_F32) return fail(B200_ERR_INVALID_ARG, "edm_create: bad precision");
  if (no_realisations < 1 || no_neurons < 2 || no_fronts < 1) return fail(B200_ERR_INVALID_ARG, "edm_create: no_realisations >= 1, no_neurons >= 2, no_fronts >= 1 required");
  if (no_neurons > 16384) return fail(B200_ERR_UNSUPPORTED, "edm_create: no_neurons > 16384 (one CTA holds a whole ring)");
  *handle = nullptr;
  B200_TRY(require_device());
  b200_edm* h = new (std::nothrow) b200_edm();
  if (!h) return fail(B200_ERR_INVALID_ARG, "out of host memory");
  h->params.assign(params, params + nparams);
  b200_edm_model_default(&h->model);
  h->R = no_realisations; h->N = no_neurons; h->Mf = no_fronts; h->prec = precision;
  cudaGetDevice(&h->device);
  cudaError_t e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
  if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_up, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming);
  if (e != cudaSuccess) { delete h; return cuda_fail(e, "edm_create", __FILE__, __LINE__); }
  *handle = h;
  return B200_OK;
}

int b200_edm_destroy(b200_edm* h) {
  if (!h) return B200_OK;
  DeviceScope callers_device(-1);
  for (b200_edm* g : h->helpers) b200_edm_destroy(g);
  h->helpers.clear();
  if (!h->comms.empty() && g_nccl.ok) for (ncclComm_t c : h->comms) g_nccl.comm_destroy(c);
  h->comms.clear();
  cudaSetDevice(h->device);
  free_ensemble(h);
  free_batch(h);
  cudaFree(h->d_gather); cudaFree(h->d_gather_acc); cudaFree(h->d_u); cudaFree(h->d_jac);
  cudaFree(h->d_clamped); cudaFree(h->d_counters);
  if (h->h_pin) cudaFreeHost(h->h_pin);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev_up) cudaEventDestroy(h->ev_up);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return B200_OK;
}

int b200_edm_set_model(b200_edm* h, const b200_edm_model* m) {
  B200_TRY(check_handle(h, "edm_set_model"));
  if (!m) return fail(B200_ERR_INVALID_ARG, "edm_set_model: NULL model");
  if (!(m->time_horizon > 0) || !(m->L > 0)) return fail(B200_ERR_INVALID_ARG, "edm_set_model: time_horizon and L must be > 0");
  h->model = *m;
  h->w_dirty = true;
  return B200_OK;
}
int b200_edm_get_model(const b200_edm* h, b200_edm_model* m) {
  B200_TRY(check_handle(h, "edm_get_model"));
  if (!m) return fail(B200_ERR_INVALID_ARG, "edm_get_model: NULL model");
  *m = h->model;
  return B200_OK;
}
int b200_edm_set_time_horizon(b200_edm* h, double T) {
  B200_TRY(check_handle(h, "edm_set_time_horizon"));
  if (!(T > 0)) return fail(B200_ERR_INVALID_ARG, "time horizon must be > 0 (EventDrivenMap.cu:244)");
  h->model.time_horizon = T;
  return B200_OK;
}
int b200_edm_set_no_realisations(b200_edm* h, uint32_t R) {
  B200_TRY(check_handle(h, "edm_set_no_realisations"));
  if (R < 1) return fail(B200_ERR_INVALID_ARG, "no_realisations must be > 0 (EventDrivenMap.cu:251)");
  if (R != h->R) { DeviceScope on_handle_device(h->device); h->R = R; h->beta_dirty = true; free_batch(h); }
  return B200_OK;
}
int b200_edm_set_no_neurons(b200_edm* h, uint32_t N) {
  B200_TRY(check_handle(h, "edm_set_no_neurons"));
  if (N < 2) return fail(B200_ERR_INVALID_ARG, "no_neurons must be >= 2 (EventDrivenMap.cu:284)");
  if (N > 16384) return fail(B200_ERR_UNSUPPORTED, "no_neurons > 16384 (one CTA holds a whole ring)");
  if (N != h->N) { DeviceScope on_handle_device(h->device); h->N = N; h->w_dirty = h->beta_dirty = true; free_batch(h); }
  return B200_OK;
}
int b200_edm_set_param_stddev(b200_edm* h, double sigma) {
  B200_TRY(check_handle(h, "edm_set_param_stddev"));
  if (!(sigma >= 0)) return fail(B200_ERR_INVALID_ARG, "sigma must be >= 0 (EventDrivenMap.cu:319)");
  if (sigma != h->sigma) {
    h->sigma = sigma; h->beta_dirty = true;
    if (sigma == 0.0) { DeviceScope on_handle_device(h->device); cudaFree(h->beta); h->beta = nullptr; }   // no stale ensemble behind DBG_BETA
  }
  return B200_OK;
}
int b200_edm_set_parameter(b200_edm* h, uint32_t par_id, double value) {
  B200_TRY(check_handle(h, "edm_set_parameter"));
  if (par_id >= h->params.size()) return fail(B200_ERR_INVALID_ARG, "parameter id %u out of range (EventDrivenMap.cu:326)", par_id);
  h->params[par_id] = value;
  if (par_id == 0) h->beta_dirty = true;
  return B200_OK;
}
int b200_edm_set_seed(b200_edm* h, uint64_t seed) {
  B200_TRY(check_handle(h, "edm_set_seed"));
  if (seed != h->seed) { h->seed = seed; h->beta_dirty = true; }
  return B200_OK;
}
int b200_edm_get_seed(const b200_edm* h, uint64_t* seed) {
  B200_TRY(check_handle(h, "edm_get_seed"));
  if (!seed) return fail(B200_ERR_INVALID_ARG, "edm_get_seed: NULL");
  *seed = h->seed;
  return B200_OK;
}
int b200_edm_new_seed(b200_edm* h) {
  B200_TRY(check_handle(h, "edm_new_seed"));
  // deterministic successor (the reference draws clock(), EventDrivenMap.cu:339)
  uint64_t x = h->seed + 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  h->seed = x ^ (x >> 31);
  h->beta_dirty = true;
  return B200_OK;
}
int b200_edm_set_devices(b200_edm* h, const int* device_ids, size_t ndevices) {
  B200_TRY(check_handle(h, "edm_set_devices"));
  if (!device_ids || ndevices < 1) return fail(B200_ERR_INVALID_ARG, "edm_set_devices: empty device list");
  DeviceScope callers_device(-1);
  if (device_ids[0] != h->device) return fail(B200_ERR_INVALID_ARG, "edm_set_devices: the first device must be the handle's own (%d)", h->device);
  int count = 0;
  B200_CUDA(cudaGetDeviceCount(&count));
  for (size_t i = 0; i < ndevices; ++i) {
    if (device_ids[i] < 0 || device_ids[i] >= count) return fail(B200_ERR_INVALID_ARG, "edm_set_devices: device %d does not exist", device_ids[i]);
    for (size_t j = 0; j < i; ++j) if (device_ids[j] == device_ids[i]) return fail(B200_ERR_INVALID_ARG, "edm_set_devices: device %d listed twice", device_ids[i]);
  }
  for (b200_edm* g : h->helpers) b200_edm_destroy(g);
  h->helpers.clear();
  if (!h->comms.empty() && g_nccl.ok) for (ncclComm_t c : h->comms) g_nccl.comm_destroy(c);
  h->comms.clear();
  h->devs.assign(device_ids, device_ids + ndevices);
  int rc = B200_OK;
  for (size_t i = 1; i < ndevices && rc == B200_OK; ++i) {
    rc = cudaSetDevice(device_ids[i]) == cudaSuccess ? B200_OK : fail(B200_ERR_CUDA, "cudaSetDevice(%d) failed", device_ids[i]);
    b200_edm* g = nullptr;
    if (rc == B200_OK) rc = b200_edm_create(h->params.data(), h->params.size(), h->R, h->N, h->Mf, h->prec, &g);
    if (rc == B200_OK) {
      h->helpers.push_back(g);
      // direct NVLink copies where the topology allows; staged through the host otherwise
      cudaDeviceEnablePeerAccess(h->device, 0);
      cudaSetDevice(h->device);
      cudaDeviceEnablePeerAccess(device_ids[i], 0);
      cudaGetLastError();
    }
  }
  cudaSetDevice(h->device);
  // the exchange is one NCCL all-gather per evaluation batch (north-star; SURVEY 8e)
  if (rc == B200_OK && ndevices > 1) {
    if (!load_nccl()) rc = fail(B200_ERR_UNSUPPORTED, "edm_set_devices: libnccl.so.2 could not be loaded (%s)", dlerror());
    if (rc == B200_OK) {
      h->comms.resize(ndevices);
      ncclResult_t r = g_nccl.comm_init_all(h->comms.data(), (int)ndevices, h->devs.data());
      if (r != ncclSuccess) {
        h->comms.clear();
        rc = fail(B200_ERR_CUDA, "edm_set_devices: ncclCommInitAll over %zu devices failed: %s", ndevices, g_nccl.error_string(r));
      }
    }
    cudaSetDevice(h->device);
  }
  if (rc != B200_OK) { for (b200_edm* g : h->helpers) b200_edm_destroy(g); h->helpers.clear(); h->devs.resize(1); }
  return rc;
}

int b200_edm_set_profile_mode(b200_edm* h, uint32_t n_coarse) {
  B200_TRY(check_handle(h, "edm_set_profile_mode"));
  if (n_coarse == 1) return fail(B200_ERR_INVALID_ARG, "profile map needs at least 2 coarse knots (0 switches it off)");
  if (n_coarse != h->profile_nc) { DeviceScope on_handle_device(h->device); free_batch(h); h->profile_nc = n_coarse; h->last_cols = 0; }
  return B200_OK;
}

int b200_edm_set_tuning(b200_edm* h, int neurons_per_thread) {
  B200_TRY(check_handle(h, "edm_set_tuning"));
  if (neurons_per_thread != 0 && neurons_per_thread != 4 && neurons_per_thread != 8 && neurons_per_thread != 16)
    return fail(B200_ERR_INVALID_ARG, "neurons per thread must be 0 (auto), 4, 8 or 16");
  h->npt = neurons_per_thread;
  return B200_OK;
}

int b200_edm_compute_f_batch(b200_edm* h, const double* z_cols, size_t n, size_t ncols, double* f_cols_out) {
  B200_TRY(check_handle(h, "edm_compute_f_batch"));
  if (!z_cols || !f_cols_out || ncols < 1) return fail(B200_ERR_INVALID_ARG, "edm_compute_f_batch: NULL / empty argument");
  return h->prec == B200_F64 ? compute_batch<double>(h, z_cols, n, ncols, f_cols_out)
                             : compute_batch<float>(h, z_cols, n, ncols, f_cols_out);
}

int b200_edm_compute_f(b200_edm* h, const double* z, size_t n, double* f_out) {
  return b200_edm_compute_f_batch(h, z, n, 1, f_out);
}

int b200_edm_compute_dfdu(b200_edm* h, const double* u, size_t n, double eps, double* jac_out, double* f0_out) {
  B200_TRY(check_handle(h, "edm_compute_dfdu"));
  if (!u || !jac_out) return fail(B200_ERR_INVALID_ARG, "edm_compute_dfdu: NULL argument");
  if (n != ndim(h)) return fail(B200_ERR_INVALID_ARG, "vector length %zu != problem dimension %zu", n, ndim(h));
  if (!(eps != 0.0)) return fail(B200_ERR_INVALID_ARG, "finite-difference epsilon must be non-zero");
  if (!h->profile_nc && (!(u[0] == u[0]) || u[0] == 0.0 || u[0] + eps == 0.0))
    return fail(B200_ERR_INVALID_ARG, "wave speed u[0] (and u[0] + eps) must be finite and non-zero");
  // columns u + eps e_i (NewtonSolver.cpp:184-188) and the base column u are formed on the device(s);
  // the difference quotients (NewtonSolver.cpp:194) too, next to the columns they belong to
  return h->prec == B200_F64 ? compute_multi<double>(h, u, n, n, true, eps, jac_out, f0_out)
                             : compute_multi<float>(h, u, n, n, true, eps, jac_out, f0_out);
}

int b200_edm_compute_dfdu_given_f(b200_edm* h, const double* u, size_t n, double eps, const double* f0, double* jac_out) {
  B200_TRY(check_handle(h, "edm_compute_dfdu_given_f"));
  if (!u || !f0 || !jac_out) return fail(B200_ERR_INVALID_ARG, "edm_compute_dfdu_given_f: NULL argument");
  if (n != ndim(h)) return fail(B200_ERR_INVALID_ARG, "vector length %zu != problem dimension %zu", n, ndim(h));
  if (!(eps != 0.0)) return fail(B200_ERR_INVALID_ARG, "finite-difference epsilon must be non-zero");
  if (!h->profile_nc && (!(u[0] == u[0]) || u[0] == 0.0 || u[0] + eps == 0.0))
    return fail(B200_ERR_INVALID_ARG, "wave speed u[0] (and u[0] + eps) must be finite and non-zero");
  // only the n perturbed columns are evaluated; the difference quotients use the caller's F(u)
  return h->prec == B200_F64 ? compute_multi<double>(h, u, n, n, true, eps, jac_out, nullptr, f0)
                             : compute_multi<float>(h, u, n, n, true, eps, jac_out, nullptr, f0);
}

int b200_edm_evolve_items_dev(b200_edm* h, const double* z_cols, size_t n, size_t ncols,
                              size_t item_begin, size_t item_end, double* pos_dev,
                              int32_t* accept_dev, void* stream) {
  B200_TRY(check_handle(h, "edm_evolve_items_dev"));
  if (!z_cols || ncols < 1 || item_end < item_begin || item_end > ncols * h->R)
    return fail(B200_ERR_INVALID_ARG, "edm_evolve_items_dev: bad item range / NULL argument");
  const size_t nitems = item_end - item_begin;
  if (nitems && (!pos_dev || !accept_dev)) return fail(B200_ERR_INVALID_ARG, "edm_evolve_items_dev: NULL output");
  DeviceScope on_handle_device(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  B200_TRY(order_after_previous(h, st));
  B200_TRY(ensure_batch(h, ncols, nitems ? nitems : 1));
  if (h->prec == B200_F64) {
    B200_TRY(ensure_ensemble<double>(h, st));
    B200_TRY(upload_z(h, z_cols, n, ncols, st));
    B200_TRY(run_prepare<double>(h, ncols, st));
    B200_TRY(run_evolve<double>(h, item_begin, item_end, pos_dev, accept_dev, st));
  } else {
    B200_TRY(ensure_ensemble<float>(h, st));
    B200_TRY(upload_z(h, z_cols, n, ncols, st));
    B200_TRY(run_prepare<float>(h, ncols, st));
    B200_TRY(run_evolve<float>(h, item_begin, item_end, (float*)h->d_pos, accept_dev, st));
    if (nitems)
      convert_kernel<float, double><<<(unsigned)((nitems * ndim(h) + 255) / 256), 256, 0, B200_CNT(st)>>>((const float*)h->d_pos, pos_dev, nitems * ndim(h));
    B200_CUDA(cudaGetLastError());
  }
  h->last_cols = ncols;
  h->last_sliced = !(item_begin == 0 && item_end == ncols * h->R);
  h->last_pos_external = (h->prec == B200_F64);   // positions went to the caller's buffer, not d_pos
  return mark_done(h, st);
}

int b200_edm_reduce_items_dev(b200_edm* h, const double* z_cols, size_t n, size_t ncols,
                              const double* pos_all_dev, const int32_t* accept_all_dev,
                              double* f_cols_dev, void* stream) {
  B200_TRY(check_handle(h, "edm_reduce_items_dev"));
  if (!z_cols || !pos_all_dev || !accept_all_dev || !f_cols_dev || ncols < 1)
    return fail(B200_ERR_INVALID_ARG, "edm_reduce_items_dev: NULL / empty argument");
  DeviceScope on_handle_device(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  B200_TRY(order_after_previous(h, st));
  B200_TRY(ensure_batch(h, ncols, 1));
  B200_TRY(upload_z(h, z_cols, n, ncols, st));
  if (h->prec == B200_F64) {
    B200_TRY(run_reduce<double>(h, ncols, pos_all_dev, accept_all_dev, f_cols_dev, st));
  } else {
    // positions were widened to double for the exchange; narrow them back so the mean is
    // accumulated in float exactly as the single-GPU path does
    const size_t nitems = ncols * h->R;
    B200_TRY(ensure_batch(h, ncols, nitems));
    convert_kernel<double, float><<<(unsigned)((nitems * ndim(h) + 255) / 256), 256, 0, B200_CNT(st)>>>(pos_all_dev, (float*)h->d_pos, nitems * ndim(h));
    B200_TRY(run_reduce<float>(h, ncols, (const float*)h->d_pos, accept_all_dev, f_cols_dev, st));
  }
  return mark_done(h, st);
}

int b200_edm_set_debug(b200_edm* h, int on) {
  B200_TRY(check_handle(h, "edm_set_debug"));
  h->debug = on ? 1 : 0;
  return B200_OK;
}

int b200_edm_enable_timing(b200_edm* h, int on) {
  B200_TRY(check_handle(h, "edm_enable_timing"));
  h->timing = on ? 1 : 0;
  return B200_OK;
}

int b200_edm_last_evolve_ms(const b200_edm* h, double* ms) {
  B200_TRY(check_handle(h, "edm_last_evolve_ms"));
  if (!ms) return fail(B200_ERR_INVALID_ARG, "NULL");
  *ms = h->last_ms;
  return B200_OK;
}

int b200_edm_last_event_total(const b200_edm* h, uint64_t* events) {
  B200_TRY(check_handle(h, "edm_last_event_total"));
  if (!events) return fail(B200_ERR_INVALID_ARG, "NULL");
  *events = h->last_counters[0];
  return B200_OK;
}

int b200_edm_last_counters(const b200_edm* h, uint64_t out[4]) {
  B200_TRY(check_handle(h, "edm_last_counters"));
  if (!out) return fail(B200_ERR_INVALID_ARG, "NULL");
  for (int i = 0; i < 4; ++i) out[i] = h->last_counters[i];
  return B200_OK;
}

int b200_edm_last_init_clamped(const b200_edm* h, int* clamped) {
  B200_TRY(check_handle(h, "edm_last_init_clamped"));
  if (!clamped) return fail(B200_ERR_INVALID_ARG, "NULL");
  *clamped = h->last_clamped;
  return B200_OK;
}

int b200_edm_debug_fetch(b200_edm* h, b200_edm_debug_what what, void* out, size_t bytes) {
  B200_TRY(check_handle(h, "edm_debug_fetch"));
  if (!out) return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: NULL output");
  if (!h->debug) return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: debug flag is off (SetDebugFlag)");
  if (h->last_cols == 0) return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: no evaluation has run yet");
  DeviceScope on_handle_device(h->device);
  const size_t C = h->last_cols, R = h->R, N = h->N, Mf = ndim(h), es = esize(h);
  if (h->profile_nc && what != B200_EDM_DBG_LIFT_V && what != B200_EDM_DBG_LIFT_S && what != B200_EDM_DBG_ACCEPT &&
      what != B200_EDM_DBG_POSITION && what != B200_EDM_DBG_EVENT_COUNT && what != B200_EDM_DBG_BETA &&
      what != B200_EDM_DBG_COUPLING)
    return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: array %d does not exist for the profile map", (int)what);
  if (h->last_sliced && (what == B200_EDM_DBG_LAST_INDEX || what == B200_EDM_DBG_LAST_TIME || what == B200_EDM_DBG_CROSSED_INDEX ||
                         what == B200_EDM_DBG_CROSSED_TIME || what == B200_EDM_DBG_ACCEPT || what == B200_EDM_DBG_POSITION ||
                         what == B200_EDM_DBG_EVENT_COUNT))
    return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: the last evaluation was sharded (item slice / several devices); "
                                      "per-item arrays are not all on this handle");
  if (h->last_pos_external && what == B200_EDM_DBG_POSITION)
    return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: the last evaluation wrote its positions to the caller's device buffer");
  const void* src = nullptr;
  size_t count = 0;
  bool real = false, is_int = false;
  switch (what) {
    case B200_EDM_DBG_INIT_INDEX: src = h->d_init; count = C * Mf; is_int = true; break;
    case B200_EDM_DBG_LIFT_V: src = h->d_lv; count = C * N; real = true; break;
    case B200_EDM_DBG_LIFT_S: src = h->d_ls; count = C * N; real = true; break;
    case B200_EDM_DBG_LAST_INDEX: src = h->d_last_i; count = C * R * Mf; is_int = true; break;
    case B200_EDM_DBG_LAST_TIME: src = h->d_last_t; count = C * R * Mf; real = true; break;
    case B200_EDM_DBG_CROSSED_INDEX: src = h->d_cross_i; count = C * R * Mf; is_int = true; break;
    case B200_EDM_DBG_CROSSED_TIME: src = h->d_cross_t; count = C * R * Mf; real = true; break;
    case B200_EDM_DBG_ACCEPT: src = h->d_accept; count = C * R; is_int = true; break;
    case B200_EDM_DBG_POSITION: src = h->d_pos; count = C * R * Mf; real = true; break;
    case B200_EDM_DBG_EVENT_COUNT: src = h->d_evcount; count = C * R; is_int = true; break;
    case B200_EDM_DBG_MEAN: src = h->d_mean; count = C * Mf; break;  // always double
    case B200_EDM_DBG_BETA: src = h->beta; count = R * N; real = true; break;
    case B200_EDM_DBG_COUPLING: src = h->w; count = N; real = true; break;
    default: return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: unknown array id %d", (int)what);
  }
  const size_t out_es = is_int ? 4 : 8;
  if (bytes < count * out_es) return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: buffer of %zu B, %zu B needed", bytes, count * out_es);
  B200_CUDA(cudaStreamSynchronize(h->stream));
  if (what == B200_EDM_DBG_BETA && !src) {  // homogeneous ensemble: beta is the mean everywhere
    double* o = (double*)out;
    const double b = h->prec == B200_F64 ? h->params[0] : (double)(float)h->params[0];
    for (size_t i = 0; i < count; ++i) o[i] = b;
    return B200_OK;
  }
  if (!src) return fail(B200_ERR_INVALID_ARG, "edm_debug_fetch: array not available");
  if (real && es == 4) {
    std::vector<float> tmp(count);
    B200_CUDA(cudaMemcpy(tmp.data(), src, count * 4, cudaMemcpyDeviceToHost));
    double* o = (double*)out;
    for (size_t i = 0; i < count; ++i) o[i] = (double)tmp[i];
  } else {
    B200_CUDA(cudaMemcpy(out, src, count * out_es, cudaMemcpyDeviceToHost));
  }
  return B200_OK;
}

}  // extern "C"
