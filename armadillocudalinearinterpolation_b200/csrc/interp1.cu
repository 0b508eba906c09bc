// interp.cu — batched 1-D / 2-D linear interpolation for sm_100a (include/b200_interp.h).
//
// What it stands in for: arma::interp1(X,Y,XI,YI,"*linear",extrap) and
// arma::interp2(X,Y,Z,XI,YI,ZI,"linear",extrap) (Armadillo fn_interp1.hpp / fn_interp2.hpp,
// an un-vendored dependency of the reference: Makefile:5, Driver.o.dep:554), and the two
// interpolation fragments the reference itself contains: the uniform-grid bracket scan of
// EventDrivenMap.cu:361-372 and the two-point blend of EventDrivenMap.cu:779-783.
//
// Design (HBM-bound byte streams, no tensor cores):
//  * queries and outputs are touched once: 256-bit LDG/STG (sm_100a LDG.E.256) with
//    L1::no_allocate + L2::evict_first so they never displace the grid in the 126 MB L2;
//  * the grid is re-laid-out at plan time into one 32-byte "segment" record per knot
//    (x[a], x[a+1], y[a], y[a+1]) so a query costs exactly ONE 32-byte sector gather,
//    fetched with L2::evict_last;
//  * bracket lookup is index arithmetic: bin = (int)((q - x0) * inv_w).  The same rounded
//    expression is applied to knots and queries, so it is monotone and the bracket derived
//    from it is EXACT after a compare against the stored knots (never a float guess):
//      mode 0 (uniform knots: bin(x[j]) == j): a = bin, one backward fix-up compare;
//      mode 1 (any strictly ascending knots): first[bin] table -> bounded forward scan,
//             binary search only inside pathological buckets;
//  * the blend is (1-w)*Y[a] + w*Y[b] with w = |X[a]-q| / (|X[a]-q| + |X[b]-q|), every
//    operation individually rounded (__dmul_rn, ...), bit-identical to the CPU oracle.
// Host buffers go through host_run() (host_staging.cuh), the runner interp2.cu's scattered calls share.
#include "interp_common.cuh"
#include "host_staging.cuh"

namespace b200 {
namespace {

// ------------------------------------------------------------------ interp1 ----
template <typename T> struct Loader1;
template <> struct Loader1<double> { using type = LoadSeg1D; };
template <> struct Loader1<float> { using type = LoadSeg1F; };

// What a call writes besides the value of each query: nothing, the bracket index (int32, -1 out of range) or the
// slope dydx (tests/interp1_grad_oracle.c restates the rules of include/b200_interp.h): (Y[b'] - Y[a']) / (X[b'] - X[a'])
// on the segment (a', b') = (a, a+1), or (n-2, n-1) on the last knot; NaN for a NaN query, +0 for any other
// out-of-range one.  Out1Of<T, OUT>: the element type of that second output stream.
enum Out1 { kValue, kIndex, kSlope };
template <typename T, Out1 OUT> using Out1Of = std::conditional_t<OUT == kSlope, T, int32_t>;

template <typename T>
__device__ __forceinline__ T seg_slope(T xa, T xb, T ya, T yb) { return div_rn(sub_rn(yb, ya), sub_rn(xb, xa)); }

// a query on the last knot: the slope of record n-2 (out of line: rare, and it must not cost the streaming loop
// registers)
template <typename T>
__device__ __noinline__ T slope_last_record(const T* __restrict__ seg, int n) {
  const T* r = seg + 4 * (size_t)(n - 2);
  return seg_slope(r[0], r[1], r[2], r[3]);
}

// the value of one query and, by OUT, its index or its slope (from the record the query already loads) in `out`
template <typename T, Out1 OUT>
__device__ __forceinline__ T interp1_one(const AxisDev<T>& ax, const typename Loader1<T>::type& ld, T q, T extrap,
                                         Out1Of<T, OUT>& out) {
  if (!(q >= ax.x0 && q <= ax.xmax)) {  // out of range -> extrap_val; NaN query -> NaN
    const bool nan = q != q;
    if (OUT == kIndex) out = -1;
    if (OUT == kSlope) out = nan ? qnan<T>() : (T)0;
    return nan ? qnan<T>() : extrap;
  }
  Seg1<T> sg;
  if (sizeof(T) == 8 && ax.mode == 0) {
    // (quasi-)uniform knots, double: the common case — the arithmetic bin is the bracket, the weight operands are in
    // the normal range — as straight-line code with the branch-free divide; anything else takes the generic walk
    const int k = bin_of(ax, q);
    sg = ld(k);
    const double xa = (double)sg.xa, xb = (double)sg.xb, qq = (double)q;
    const double a_err = __dsub_rn(qq, xa), b_err = __dsub_rn(xb, qq), sum = __dadd_rn(a_err, b_err);
    if ((xa <= qq) && (qq < xb) && (a_err >= 0x1p-500) && (sum <= 0x1p500)) {
      if (OUT == kIndex) out = k;
      if (OUT == kSlope) out = seg_slope(sg.xa, sg.xb, sg.ya, sg.yb);
      return blend((T)div_rn_fast(a_err, sum), sg.ya, sg.yb);
    }
  }
  const int a = find_bracket(ax, ld, q, sg);
  if (OUT == kIndex) out = a;
  if (OUT == kSlope) out = a + 1 < ax.n ? seg_slope(sg.xa, sg.xb, sg.ya, sg.yb) : slope_last_record<T>(ld.seg, ax.n);
  return blend(weight_of(sg.xa, sg.xb, q), sg.ya, sg.yb);
}

template <typename T>
__device__ __forceinline__ typename Loader1<T>::type make_loader1(const T* seg);
template <> __device__ __forceinline__ LoadSeg1D make_loader1<double>(const double* seg) { return {seg}; }
template <> __device__ __forceinline__ LoadSeg1F make_loader1<float>(const float* seg) { return {seg, l2_policy_evict_last()}; }

// V results of one vector iteration: yi, and the second stream of OUT (the index: 32 bytes f32 / 16 bytes f64)
template <typename T, Out1 OUT, int V>
__device__ __forceinline__ void st_results(T* yi, Out1Of<T, OUT>* out, const T (&y)[V], const Out1Of<T, OUT> (&o)[V]) {
  st_stream_256(yi, y);
  if constexpr (OUT == kSlope) st_stream_256(out, o);
  if constexpr (OUT == kIndex) {
    if constexpr (V == 8) st_stream_256(out, o);
    else st_stream_128(out, o);
  }
}

// Vector kernel: each thread owns 32 bytes of queries per iteration (4 doubles / 8 floats),
// i.e. V independent gather chains in flight.  Requires 32-byte aligned xi / yi and `out` aligned to its vector
// (plan1_launch).
// (Affine axes could gather the 16-byte value pair instead of the 32-byte record; measured within +-2 %
// of this kernel at 1e7 and 1e8 queries — the gather RATE bounds it, not the bytes — and not kept.)
template <typename T, Out1 OUT>
__global__ void __launch_bounds__(kThreads)
interp1_vec_kernel(AxisDev<T> ax, const T* __restrict__ seg, const T* __restrict__ xi, T* __restrict__ yi,
                   Out1Of<T, OUT>* __restrict__ out, size_t nvec, T extrap) {
  constexpr int V = Vec256<T>::n;
  if (OUT != kSlope) {
    // programmatic dependent launch (plan1_launch): this grid may have been scheduled while the previous kernel of
    // the stream was still draining; nothing is read or written before that kernel has completed and flushed
    // (a no-op for an ordinary launch), and the next launch of the stream may be scheduled from now on
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
  }
  const auto ld = make_loader1<T>(seg);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    T q[V], y[V];
    Out1Of<T, OUT> o[V];
    ld_stream_256(xi + i * V, q);
#pragma unroll
    for (int j = 0; j < V; ++j) y[j] = interp1_one<T, OUT>(ax, ld, q[j], extrap, o[j]);
    st_results<T, OUT>(yi + i * V, out + i * V, y, o);
  }
}

// Scalar kernel: tails and unaligned buffers.
template <typename T, Out1 OUT>
__global__ void __launch_bounds__(kThreads)
interp1_scalar_kernel(AxisDev<T> ax, const T* __restrict__ seg, const T* __restrict__ xi, T* __restrict__ yi,
                      Out1Of<T, OUT>* __restrict__ out, size_t begin, size_t end, T extrap) {
  const auto ld = make_loader1<T>(seg);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += stride) {
    Out1Of<T, OUT> o;
    yi[i] = interp1_one<T, OUT>(ax, ld, xi[i], extrap, o);
    if (OUT != kValue) out[i] = o;
  }
}

// ---- small grids: the whole grid staged in shared memory ----
// The "coarse profile -> fine ensemble" case (a few thousand knots, millions of queries): persistent
// CTAs copy the knots, the values and (for non-uniform knots) the bucket table into shared memory
// once with TMA bulk copies and then stream queries; the bracket lookup and the two value reads never
// leave the SM, so HBM carries exactly 16 bytes (f64) per query.  Affine knots (linspace) are recomputed
// instead of staged: half the shared memory, half the bank-conflicted look-ups (0.79 vs 0.74 of peak).
constexpr int kSmem1Threads = 512;

// the last segment's slope on a staged (or affine) axis, out of line as slope_last_record
template <typename T>
__device__ __noinline__ T slope_last_knot_s(const AxisSmem<T> A, const T* sy) {
  const int a = A.n - 2;
  const T xa = A.affine ? affine_knot(A.affine, A.x0, A.step, A.xmax, A.n, a) : A.x[a];
  return seg_slope(xa, A.xmax, sy[a], sy[a + 1]);
}

// The slope comes from sy[] and the staged or recomputed knots (affine knots are bit-identical to the stored ones).
// find_bracket_s<T, 2>: the slope instance's own copy of the out-of-line knot search (interp_common.cuh), so the
// value instances' register allocation does not depend on it.
template <typename T, Out1 OUT>
__global__ void __launch_bounds__(kSmem1Threads)
interp1_smem_kernel(AxisDev<T> ax, const T* __restrict__ yg, const T* __restrict__ xi, T* __restrict__ yi,
                    Out1Of<T, OUT>* __restrict__ out, size_t nvec, T extrap) {
  extern __shared__ __align__(128) unsigned char smem1[];
  constexpr int V = Vec256<T>::n;
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem1);
  auto pad16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
  const size_t yb_bytes = pad16(sizeof(T) * ax.n);
  const size_t xb_bytes = ax.affine ? 0 : yb_bytes;   // affine knots are recomputed: only the values are staged
  const size_t fb_bytes = (!ax.affine && ax.mode) ? pad16(sizeof(int32_t) * ((size_t)ax.nb + 1)) : 0;
  T* sx = reinterpret_cast<T*>(smem1 + 16);
  T* sy = reinterpret_cast<T*>(smem1 + 16 + xb_bytes);
  int32_t* sf = reinterpret_cast<int32_t*>(smem1 + 16 + xb_bytes + yb_bytes);
  if (threadIdx.x == 0) mbar_init(bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, (unsigned)(xb_bytes + yb_bytes + fb_bytes));
    const unsigned chunk = 16384;
    auto copy = [&](void* dst, const void* src, size_t bytes) {
      for (size_t o = 0; o < bytes; o += chunk)
        tma_bulk_g2s((unsigned char*)dst + o, (const unsigned char*)src + o, (unsigned)(bytes - o < chunk ? bytes - o : chunk), bar);
    };
    if (xb_bytes) copy(sx, ax.x, xb_bytes);
    copy(sy, yg, yb_bytes);
    if (fb_bytes) copy(sf, ax.first, fb_bytes);
  }
  mbar_wait(bar, 0);
  const AxisSmem<T> A = {sx, sf, ax.x0, ax.xmax, ax.inv_w, ax.n, ax.nb, ax.mode, ax.affine, ax.step};
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    T q[V], y[V];
    Out1Of<T, OUT> o[V];
    ld_stream_256(xi + i * V, q);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const T qq = q[j];
      if (!(qq >= A.x0 && qq <= A.xmax)) {
        const bool nan = qq != qq;
        if (OUT == kIndex) o[j] = -1;
        y[j] = nan ? qnan<T>() : extrap;
        if (OUT == kSlope) o[j] = nan ? qnan<T>() : (T)0;
      } else {
        T xa, xb;
        const int a = find_bracket_s<T, OUT == kSlope ? 2 : 0>(A, qq, xa, xb);
        if (OUT == kIndex) o[j] = a;
        if constexpr (OUT == kSlope) {   // (values before the weight here, after it below: each instance's measured schedule)
          const T ya = sy[a], yb = sy[min(a + 1, A.n - 1)];
          y[j] = blend(weight_of(xa, xb, qq), ya, yb);
          o[j] = a + 1 < A.n ? seg_slope(xa, xb, ya, yb) : slope_last_knot_s<T>(A, sy);
        } else {
          y[j] = blend(weight_of(xa, xb, qq), sy[a], sy[min(a + 1, A.n - 1)]);
        }
      }
    }
    st_results<T, OUT>(yi + i * V, out + i * V, y, o);
  }
}

// Value tables of a plan from Y at `y` (device memory): the plan's copy of Y that the shared-memory path stages
// (yg; nullptr when Y was uploaded there directly) and one segment record (x[a], x[b], y[a], y[b]) per knot.
template <typename T>
__global__ void interp1_values_kernel(const T* __restrict__ x, const T* __restrict__ y, int n, T* __restrict__ yg,
                                      T* __restrict__ seg) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n) return;
  const int b = min(a + 1, n - 1);
  const T ya = y[a];
  if (yg) yg[a] = ya;
  const T v[4] = {x[a], x[b], ya, y[b]};
  st_vec4(seg + 4 * (size_t)a, v);
}

// ---- adjoint G = W^T g, deterministic (no atomics) ----
// (1) segment key a per query, sentinel n when it does not contribute; (2) stable radix sort of (key, query index);
// (3) adjoint_offsets_kernel: off[c] = first sorted position of segment c; (4) every term written straight into
// node-major order; (5) the blocked sum R level by level over all nodes at once.
//
// Node j's list at level 0 starts at S_j = off[j-1] + off[j] (off[-1] = 0): segment j-1's role-1 terms, then segment
// j's role-0 terms, and at node n-1 both terms of each last-knot query, interleaved by query; it ends at S_{j+1}
// (S_n = 2 off[n], every term).  Level L+1 holds the block sums of the nodes with more than B items at level L:
// node j's start there is floor(S_j / B) + j, which leaves room for its ceil(len_j / B) sums, so every level's layout
// is a closed form of off[] and no scan is needed between levels.
constexpr int kAdj1B = B200_INTERP1_ADJOINT_BLOCK;

// (1): the exact search on the plan's global knots, whatever the lookup mode
template <typename T>
__global__ void __launch_bounds__(kThreads)
interp1_adjoint_keys_kernel(AxisDev<T> ax, const T* __restrict__ xi, uint32_t ni, uint32_t* __restrict__ keys,
                            uint32_t* __restrict__ idx) {
  const AxisSmem<T> A = {ax.x, ax.first, ax.x0, ax.xmax, ax.inv_w, ax.n, ax.nb, ax.mode, ax.affine, ax.step};
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < ni; i += gridDim.x * blockDim.x) {
    const T q = xi[i];
    uint32_t key = (uint32_t)A.n;
    if (q >= A.x0 && q <= A.xmax) {
      T xa, xb;
      key = (uint32_t)find_bracket_s<T, 2>(A, q, xa, xb);
    }
    keys[i] = key;
    idx[i] = i;
  }
}

// (4): (1-w) g[k] at node a (role 0) and w g[k] at node b (role 1), each rounded once; w is the value call's weight
template <typename T>
__global__ void __launch_bounds__(kThreads)
interp1_adjoint_terms_kernel(const T* __restrict__ x, int n, const T* __restrict__ xi, const T* __restrict__ g,
                             const uint32_t* __restrict__ keys, const uint32_t* __restrict__ idx,
                             const uint32_t* __restrict__ off, uint32_t ni, T* __restrict__ terms) {
  for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < ni; s += gridDim.x * blockDim.x) {
    const uint32_t a = keys[s];
    if (a >= (uint32_t)n) break;   // sorted: the sentinels are last
    const uint32_t k = idx[s];
    const T gk = g[k];
    const T w = weight_of(x[a], x[min((int)a + 1, n - 1)], xi[k]);
    const T t0 = mul_rn(sub_rn((T)1, w), gk), t1 = mul_rn(w, gk);
    if ((int)a + 1 < n) {
      terms[(uint64_t)off[a] + s] = t0;        // node a: after segment a-1's role-1 terms
      terms[(uint64_t)off[a + 1] + s] = t1;    // node a+1: first its role-1 terms
    } else {
      const uint64_t p = 2 * (uint64_t)off[n - 1] + 2 * (uint64_t)(s - off[n - 1]);
      terms[p] = t0;
      terms[p + 1] = t1;
    }
  }
}

// start and length of node j's items at `level` (j == n: start = the level's end), and the length one level up
__device__ __forceinline__ void adj1_node(const uint32_t* __restrict__ off, int n, int j, int level, uint64_t& start,
                                          uint64_t& len, uint64_t& prev_len) {
  if (j >= n) {
    start = 2 * (uint64_t)off[n];
    len = 0;
  } else {
    const uint64_t o0 = j ? off[j - 1] : 0, o1 = off[j], o2 = off[j + 1];
    start = o0 + o1;
    len = (o1 - o0) + (o2 - o1) + (j == n - 1 ? o2 - o1 : 0);
  }
  prev_len = len;
  for (int l = 0; l < level; ++l) {
    start = start / kAdj1B + (uint64_t)j;
    prev_len = len;
    len = (len + kAdj1B - 1) / kAdj1B;
  }
}

template <typename T>
__device__ __forceinline__ T adj1_sum(const T* __restrict__ in, uint64_t b, uint64_t e) {
  T acc = (T)0;
#pragma unroll 8   // (the loads of eight items in flight before their in-order adds)
  for (uint64_t p = b; p < e; ++p) acc = add_rn(acc, __ldg(in + p));
  return acc;
}

// (5), one level: one thread per slot u of level+1.  The slot's node j (binary search on the closed-form starts) either
// is live at this level (more than B items): block u - start_j of its items, summed from +0, goes to out[u]; or has
// reached at most B items here: its first slot writes G[j], the sum of those items from +0.
template <typename T>
__global__ void __launch_bounds__(kThreads)
interp1_adjoint_level_kernel(const uint32_t* __restrict__ off, int n, int level, const T* __restrict__ in,
                             T* __restrict__ out, uint64_t nslots, T* __restrict__ G) {
  uint64_t end, len, prev;
  adj1_node(off, n, n, level + 1, end, len, prev);
  if (end < nslots) nslots = end;
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < nslots; u += (uint64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = n - 1;   // last node whose start one level up is <= u
    while (lo < hi) {
      const int m = (lo + hi + 1) >> 1;
      uint64_t s1;
      adj1_node(off, n, m, level + 1, s1, len, prev);
      if (s1 <= u) lo = m; else hi = m - 1;
    }
    const int j = lo;
    uint64_t s0, s1;
    adj1_node(off, n, j, level, s0, len, prev);
    s1 = s0 / kAdj1B + (uint64_t)j;
    const uint64_t m = u - s1;
    if (len > (uint64_t)kAdj1B) {
      if (m * kAdj1B < len) {
        const uint64_t b = s0 + m * kAdj1B, e = b + kAdj1B < s0 + len ? b + kAdj1B : s0 + len;
        out[u] = adj1_sum(in, b, e);
      }
    } else if (m == 0 && (level == 0 || prev > (uint64_t)kAdj1B)) {
      G[j] = adj1_sum(in, s0, s0 + len);
    }
  }
}

}  // namespace
}  // namespace b200

using namespace b200;

// ------------------------------------------------------------------ interp1 plan ----
struct b200_interp1_plan {
  b200_dtype dtype;
  int device;
  size_t ng;
  Axis<double> ax64;
  Axis<float> ax32;
  void* yg = nullptr;   // device copy of the values
  void* seg = nullptr;  // [ng][4] segment records
  size_t smem_bytes = 0;  // > 0: the grid fits the shared-memory path
  cudaStream_t stream[2] = {nullptr, nullptr};
  HostSlots slots;    // device buffers of the host-buffer calls (host_staging.cuh)
  StagePool pool;     // pinned ring for pageable host buffers
};

namespace {

template <typename T> Axis<T>& axis_of(b200_interp1_plan* p);
template <> Axis<double>& axis_of<double>(b200_interp1_plan* p) { return p->ax64; }
template <> Axis<float>& axis_of<float>(b200_interp1_plan* p) { return p->ax32; }

// The plan's value tables from Y at `y` (device memory) on `st`; write_y: also copy Y into p->yg (the host-buffer
// paths upload it there and pass y == p->yg).  No allocation, no host synchronisation.
template <typename T>
int plan1_build_values(b200_interp1_plan* p, const T* y, bool write_y, cudaStream_t st) {
  Axis<T>& A = axis_of<T>(p);
  interp1_values_kernel<T><<<grid_for(p->ng), kThreads, 0, B200_CNT(st)>>>(A.x, y, (int)p->ng,
                                                                          write_y ? (T*)p->yg : nullptr, (T*)p->seg);
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

template <typename T>
int plan1_create(b200_interp1_plan* p, const T* xg, const T* yg, size_t ng) {
  B200_CUDA(cudaStreamCreateWithFlags(&p->stream[0], cudaStreamNonBlocking));
  B200_CUDA(cudaStreamCreateWithFlags(&p->stream[1], cudaStreamNonBlocking));
  B200_TRY(axis_create<T>(axis_of<T>(p), xg, ng, p->stream[0], "interp1 grid", true));
  B200_CUDA(cudaMalloc(&p->yg, ng * sizeof(T) + 16));  // +16: bulk copies move whole 16-byte units
  B200_CUDA(cudaMemsetAsync(p->yg, 0, ng * sizeof(T) + 16, p->stream[0]));
  B200_CUDA(cudaMalloc(&p->seg, ng * 4 * sizeof(T)));
  B200_CUDA(cudaMemcpyAsync(p->yg, yg, ng * sizeof(T), cudaMemcpyHostToDevice, p->stream[0]));
  B200_TRY(plan1_build_values<T>(p, (const T*)p->yg, false, p->stream[0]));
  B200_CUDA(cudaStreamSynchronize(p->stream[0]));
  {
    auto pad16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const AxisDev<T>& ax = axis_of<T>(p).dev;
    const size_t need = 16 + (ax.affine ? 1 : 2) * pad16(sizeof(T) * ng) +
                        ((!ax.affine && ax.mode) ? pad16(sizeof(int32_t) * ((size_t)ax.nb + 1)) : 0);
    p->smem_bytes = need <= 100 * 1024 ? need : 0;   // two CTAs per SM
  }
  return B200_OK;
}

// Grid of the global-table vector kernels over nvec vectors: 16 resident CTAs per SM, 64 for very large calls,
// grid-stride beyond that.
// measured: 1e7 queries 37.0 us with 16 CTAs per SM vs 38.9 us with 64; 1e8 queries 0.304 ms with 64 vs 0.316 ms with 16
inline int interp1_vec_grid(size_t nvec) {
  const size_t blocks = (nvec + kThreads - 1) / kThreads;
  const size_t mult = blocks > (size_t)148 * 256 ? 64 : 16;
  return (int)(blocks < (size_t)148 * mult ? blocks : (size_t)148 * mult);
}

// Launch on device buffers: yi and at most one of idx / dydx.  Vector kernels when every stream is aligned to its
// vector (32 bytes; the f64 index stream 16): the shared-memory kernel for large calls on a plan whose grid fits it,
// the record kernel otherwise; the scalar kernel takes the tail.
template <typename T>
int plan1_launch(b200_interp1_plan* p, const T* xi, size_t ni, T* yi, int32_t* idx, T* dydx, T extrap,
                 cudaStream_t st) {
  if (ni == 0) return B200_OK;
  constexpr int V = Vec256<T>::n;
  const AxisDev<T>& ax = axis_of<T>(p).dev;
  const T* seg = (const T*)p->seg;
  auto run = [&](auto mode, auto* out) -> int {
    constexpr Out1 OUT = decltype(mode)::value;
    const bool aligned = (((uintptr_t)xi | (uintptr_t)yi) % 32 == 0) && ((uintptr_t)out % (sizeof(*out) * V) == 0);
    const size_t nvec = aligned ? ni / V : 0;
    if (nvec && p->smem_bytes && nvec >= 4096) {
      unsigned grid = 0;
      B200_TRY(persistent_grid(interp1_smem_kernel<T, OUT>, kSmem1Threads, p->smem_bytes, p->device,
                               (nvec + kSmem1Threads - 1) / kSmem1Threads, grid));
      interp1_smem_kernel<T, OUT><<<grid, kSmem1Threads, p->smem_bytes, B200_CNT(st)>>>(ax, (const T*)p->yg, xi, yi, out,
                                                                                      nvec, extrap);
    } else if (nvec) {
      // back-to-back calls on one stream (a caller that batches, the chunks of the host-buffer pipeline): with the
      // programmatic-stream-serialization attribute the next grid is scheduled while this one drains and starts the
      // moment it has completed — no launch bubble between 30-60 us kernels.  Only the instances that wait for the
      // previous grid (griddepcontrol.wait) before they touch memory may be launched so: not the slope instance.
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)interp1_vec_grid(nvec)); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = 0;
      cfg.stream = B200_CNT(st);
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attr; cfg.numAttrs = OUT == kSlope ? 0 : 1;
      B200_CUDA(cudaLaunchKernelEx(&cfg, interp1_vec_kernel<T, OUT>, ax, seg, xi, yi, out, nvec, extrap));
    }
    const size_t done = nvec * V;
    if (done < ni)
      interp1_scalar_kernel<T, OUT><<<capped_grid(ni - done), kThreads, 0, B200_CNT(st)>>>(ax, seg, xi, yi, out, done, ni,
                                                                                           extrap);
    return B200_OK;
  };
  if (dydx) B200_TRY(run(std::integral_constant<Out1, kSlope>(), dydx));
  else if (idx) B200_TRY(run(std::integral_constant<Out1, kIndex>(), idx));
  else B200_TRY(run(std::integral_constant<Out1, kValue>(), idx));
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

// Host buffers: host_run (host_staging.cuh) with plan1_launch
template <typename T>
int plan1_host(b200_interp1_plan* p, const T* xi, size_t ni, T* yi, int32_t* idx, T* dydx, T extrap) {
  std::vector<StageArray> arrays = {{xi, nullptr, sizeof(T)}, {nullptr, yi, sizeof(T)}};
  if (idx) arrays.push_back({nullptr, idx, sizeof(int32_t)});
  if (dydx) arrays.push_back({nullptr, dydx, sizeof(T)});
  return host_run(p->slots, p->stream, p->pool, p->device, dydx ? "interp1:grad_host" : "interp1:exec_host", arrays, ni,
                  [&](const std::vector<void*>& d, size_t n, cudaStream_t st) {
                    return plan1_launch<T>(p, (const T*)d[0], n, (T*)d[1], idx ? (int32_t*)d[2] : nullptr,
                                           dydx ? (T*)d[2] : nullptr, extrap, st);
                  });
}

// Adjoint workspace: the shared parts (AdjointWs), the 2 ni terms and the block sums of the levels above the terms.  A
// node holds at most 2 ni items, so `passes` levels (each dividing that bound by B) bring every node to at most B items.
constexpr int kAdj1MaxPasses = 5;
struct Adjoint1Ws {
  AdjointWs s;
  size_t terms, level[kAdj1MaxPasses];
  uint64_t nslots[kAdj1MaxPasses];   // slots of level L+1 (an upper bound of their end), L = 0 .. passes-1
  int passes;
};

inline int adjoint1_ws(const b200_interp1_plan* p, size_t ni, Adjoint1Ws& w) {
  const uint64_t n = p->ng;   // also the sentinel key
  B200_TRY(adjoint_ws(n, ni, w.s));
  const size_t esz = p->dtype == B200_F64 ? 8 : 4;
  w.terms = w.s.add(2 * ni * esz);
  uint64_t items = 2 * (uint64_t)ni, maxlen = items;
  w.passes = 0;
  for (;;) {
    items = items / kAdj1B + n;   // the end of level L+1 is at most floor(end of level L / B) + n
    w.nslots[w.passes++] = items;
    if (maxlen <= (uint64_t)kAdj1B) break;
    maxlen = (maxlen + kAdj1B - 1) / kAdj1B;
    w.level[w.passes] = w.s.add(items * esz);
  }
  return B200_OK;
}

template <typename T>
int plan1_adjoint_launch(b200_interp1_plan* p, const T* xi, const T* g, size_t ni, T* G, void* workspace,
                         const Adjoint1Ws& w, cudaStream_t st) {
  unsigned char* ws = (unsigned char*)workspace;
  const AxisDev<T>& ax = axis_of<T>(p).dev;
  const int n = (int)p->ng;
  const uint32_t m = (uint32_t)ni;
  const uint32_t* off = (const uint32_t*)(ws + w.s.off);
  T* terms = (T*)(ws + w.terms);
  if (m)
    interp1_adjoint_keys_kernel<T><<<capped_grid(m), kThreads, 0, B200_CNT(st)>>>(ax, xi, m, (uint32_t*)(ws + w.s.keys[0]),
                                                                                 (uint32_t*)(ws + w.s.idx[0]));
  const uint32_t *keys = nullptr, *idx = nullptr;
  B200_TRY(adjoint_sort(ws, w.s, m, (uint64_t)n, st, keys, idx));
  if (m)
    interp1_adjoint_terms_kernel<T><<<capped_grid(m), kThreads, 0, B200_CNT(st)>>>(ax.x, n, xi, g, keys, idx, off, m,
                                                                                  terms);
  const T* in = terms;
  for (int L = 0; L < w.passes; ++L) {
    T* out = L + 1 < w.passes ? (T*)(ws + w.level[L + 1]) : nullptr;
    interp1_adjoint_level_kernel<T><<<capped_grid(w.nslots[L]), kThreads, 0, B200_CNT(st)>>>(off, n, L, in, out,
                                                                                             w.nslots[L], G);
    in = out;
  }
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

void plan1_free(b200_interp1_plan* p) {
  p->ax64.release();
  p->ax32.release();
  cudaFree(p->yg);
  cudaFree(p->seg);
  p->slots.release();
  for (cudaStream_t s : p->stream)
    if (s) cudaStreamDestroy(s);
  delete p;
}

}  // namespace

extern "C" {

int b200_interp1_plan_create(b200_dtype dtype, const void* xg, const void* yg, size_t ng,
                             b200_interp1_plan** plan) {
  if (!xg || !yg || !plan) return fail(B200_ERR_INVALID_ARG, "interp1_plan_create: NULL argument");
  if (dtype != B200_F64 && dtype != B200_F32) return fail(B200_ERR_INVALID_ARG, "interp1_plan_create: bad dtype");
  *plan = nullptr;
  B200_TRY(require_device());
  b200_interp1_plan* p = new (std::nothrow) b200_interp1_plan();
  if (!p) return fail(B200_ERR_INVALID_ARG, "out of host memory");
  p->dtype = dtype;
  p->ng = ng;
  cudaGetDevice(&p->device);
  int rc = dtype == B200_F64 ? plan1_create<double>(p, (const double*)xg, (const double*)yg, ng)
                             : plan1_create<float>(p, (const float*)xg, (const float*)yg, ng);
  if (rc != B200_OK) { plan1_free(p); return rc; }
  *plan = p;
  return B200_OK;
}

int b200_interp1_plan_set_values(b200_interp1_plan* p, const void* yg) {
  if (!p || !yg) return fail(B200_ERR_INVALID_ARG, "interp1_plan_set_values: NULL argument");
  DeviceScope on_plan_device(p->device);
  size_t esz = p->dtype == B200_F64 ? 8 : 4;
  B200_CUDA(cudaMemcpyAsync(p->yg, yg, p->ng * esz, cudaMemcpyHostToDevice, p->stream[0]));
  B200_TRY(p->dtype == B200_F64 ? plan1_build_values<double>(p, (const double*)p->yg, false, p->stream[0])
                                : plan1_build_values<float>(p, (const float*)p->yg, false, p->stream[0]));
  B200_CUDA(cudaStreamSynchronize(p->stream[0]));
  return B200_OK;
}

int b200_interp1_plan_set_values_dev(b200_interp1_plan* p, const void* yg_dev, void* stream) {
  if (!p || !yg_dev) return fail(B200_ERR_INVALID_ARG, "interp1_plan_set_values_dev: NULL argument");
  DeviceScope on_plan_device(p->device);
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == B200_F64 ? plan1_build_values<double>(p, (const double*)yg_dev, true, st)
                              : plan1_build_values<float>(p, (const float*)yg_dev, true, st);
}

int b200_interp1_plan_destroy(b200_interp1_plan* p) {
  if (p) { DeviceScope on_plan_device(p->device); plan1_free(p); }
  return B200_OK;
}

int b200_interp1_plan_lookup_mode(const b200_interp1_plan* p) {
  if (!p) return fail(B200_ERR_INVALID_ARG, "NULL plan");
  if (p->smem_bytes) return 2;
  return p->dtype == B200_F64 ? p->ax64.dev.mode : p->ax32.dev.mode;
}

int b200_interp1_exec(b200_interp1_plan* p, const void* xi, size_t ni, void* yi, int32_t* idx_out,
                      double extrap_val) {
  if (!p || (ni && (!xi || !yi))) return fail(B200_ERR_INVALID_ARG, "interp1_exec: NULL argument");
  DeviceScope on_plan_device(p->device);
  return p->dtype == B200_F64
             ? plan1_host<double>(p, (const double*)xi, ni, (double*)yi, idx_out, nullptr, extrap_val)
             : plan1_host<float>(p, (const float*)xi, ni, (float*)yi, idx_out, nullptr, (float)extrap_val);
}

int b200_interp1_exec_dev(b200_interp1_plan* p, const void* xi_dev, size_t ni, void* yi_dev,
                          int32_t* idx_dev, double extrap_val, void* stream) {
  if (!p || (ni && (!xi_dev || !yi_dev))) return fail(B200_ERR_INVALID_ARG, "interp1_exec_dev: NULL argument");
  DeviceScope on_plan_device(p->device);
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == B200_F64
             ? plan1_launch<double>(p, (const double*)xi_dev, ni, (double*)yi_dev, idx_dev, nullptr, extrap_val, st)
             : plan1_launch<float>(p, (const float*)xi_dev, ni, (float*)yi_dev, idx_dev, nullptr, (float)extrap_val, st);
}

int b200_interp1_grad(b200_interp1_plan* p, const void* xi, size_t ni, void* yi, void* dydx, double extrap_val) {
  if (!p || (ni && (!xi || !yi || !dydx))) return fail(B200_ERR_INVALID_ARG, "interp1_grad: NULL argument");
  DeviceScope on_plan_device(p->device);
  return p->dtype == B200_F64
             ? plan1_host<double>(p, (const double*)xi, ni, (double*)yi, nullptr, (double*)dydx, extrap_val)
             : plan1_host<float>(p, (const float*)xi, ni, (float*)yi, nullptr, (float*)dydx, (float)extrap_val);
}

int b200_interp1_grad_dev(b200_interp1_plan* p, const void* xi_dev, size_t ni, void* yi_dev, void* dydx_dev,
                          double extrap_val, void* stream) {
  if (!p || (ni && (!xi_dev || !yi_dev || !dydx_dev))) return fail(B200_ERR_INVALID_ARG, "interp1_grad_dev: NULL argument");
  DeviceScope on_plan_device(p->device);
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == B200_F64
             ? plan1_launch<double>(p, (const double*)xi_dev, ni, (double*)yi_dev, nullptr, (double*)dydx_dev, extrap_val, st)
             : plan1_launch<float>(p, (const float*)xi_dev, ni, (float*)yi_dev, nullptr, (float*)dydx_dev, (float)extrap_val, st);
}

int b200_interp1_adjoint_workspace(const b200_interp1_plan* p, size_t ni, size_t* bytes) {
  if (!p || !bytes) return fail(B200_ERR_INVALID_ARG, "interp1_adjoint_workspace: NULL argument");
  if (ni > (size_t)INT32_MAX) return fail(B200_ERR_INVALID_ARG, "interp1_adjoint: %zu queries exceed 2^31-1", ni);
  DeviceScope on_plan_device(p->device);
  Adjoint1Ws w;
  B200_TRY(adjoint1_ws(p, ni, w));
  *bytes = w.s.total;
  return B200_OK;
}

int b200_interp1_adjoint_dev(b200_interp1_plan* p, const void* xi_dev, const void* g_dev, size_t ni, void* G_dev,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (!p || !G_dev || !workspace || (ni && (!xi_dev || !g_dev)))
    return fail(B200_ERR_INVALID_ARG, "interp1_adjoint_dev: NULL argument");
  size_t need = 0;
  B200_TRY(b200_interp1_adjoint_workspace(p, ni, &need));
  if (workspace_bytes < need)
    return fail(B200_ERR_INVALID_ARG, "interp1_adjoint_dev: workspace of %zu bytes is below the %zu required",
                workspace_bytes, need);
  DeviceScope on_plan_device(p->device);
  Adjoint1Ws w;
  B200_TRY(adjoint1_ws(p, ni, w));
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == B200_F64
             ? plan1_adjoint_launch<double>(p, (const double*)xi_dev, (const double*)g_dev, ni, (double*)G_dev, workspace, w, st)
             : plan1_adjoint_launch<float>(p, (const float*)xi_dev, (const float*)g_dev, ni, (float*)G_dev, workspace, w, st);
}

int b200_interp1_adjoint(b200_interp1_plan* p, const void* xi, const void* g, size_t ni, void* G) {
  if (!p || !G || (ni && (!xi || !g))) return fail(B200_ERR_INVALID_ARG, "interp1_adjoint: NULL argument");
  size_t need = 0;
  B200_TRY(b200_interp1_adjoint_workspace(p, ni, &need));
  DeviceScope on_plan_device(p->device);
  const size_t esz = p->dtype == B200_F64 ? 8 : 4;
  cudaStream_t st = p->stream[0];
  return adjoint_host({xi, g}, ni * esz, G, p->ng * esz, need, st,
                      [&](const std::vector<void*>& d, void* dG, void* ws) {
                        return b200_interp1_adjoint_dev(p, d[0], d[1], ni, dG, ws, need, st);
                      });
}

int b200_interp1_f64(const double* xg, const double* yg, size_t ng, const double* xi, size_t ni,
                     double* yi, int32_t* idx_out, double extrap_val) {
  b200_interp1_plan* p = nullptr;
  B200_TRY(b200_interp1_plan_create(B200_F64, xg, yg, ng, &p));
  int rc = b200_interp1_exec(p, xi, ni, yi, idx_out, extrap_val);
  b200_interp1_plan_destroy(p);
  return rc;
}

int b200_interp1_f32(const float* xg, const float* yg, size_t ng, const float* xi, size_t ni,
                     float* yi, int32_t* idx_out, float extrap_val) {
  b200_interp1_plan* p = nullptr;
  B200_TRY(b200_interp1_plan_create(B200_F32, xg, yg, ng, &p));
  int rc = b200_interp1_exec(p, xi, ni, yi, idx_out, (double)extrap_val);
  b200_interp1_plan_destroy(p);
  return rc;
}

}  // extern "C"
