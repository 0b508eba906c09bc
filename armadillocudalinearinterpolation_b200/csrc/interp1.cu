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
#include "interp_common.cuh"
#include "host_staging.cuh"

namespace b200 {
namespace {

// ------------------------------------------------------------------ interp1 ----
template <typename T> struct Loader1;
template <> struct Loader1<double> { using type = LoadSeg1D; };
template <> struct Loader1<float> { using type = LoadSeg1F; };

template <typename T>
__device__ __forceinline__ T interp1_one(const AxisDev<T>& ax, const typename Loader1<T>::type& ld, T q, T extrap,
                                         int32_t& idx) {
  if (!(q >= ax.x0 && q <= ax.xmax)) {  // out of range -> extrap_val; NaN query -> NaN
    idx = -1;
    return (q != q) ? qnan<T>() : extrap;
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
      idx = k;
      return blend((T)div_rn_fast(a_err, sum), sg.ya, sg.yb);
    }
  }
  idx = find_bracket(ax, ld, q, sg);
  return blend(weight_of(sg.xa, sg.xb, q), sg.ya, sg.yb);
}

template <typename T>
__device__ __forceinline__ typename Loader1<T>::type make_loader1(const T* seg);
template <> __device__ __forceinline__ LoadSeg1D make_loader1<double>(const double* seg) { return {seg}; }
template <> __device__ __forceinline__ LoadSeg1F make_loader1<float>(const float* seg) { return {seg, l2_policy_evict_last()}; }

// Vector kernel: each thread owns 32 bytes of queries per iteration (4 doubles / 8 floats),
// i.e. V independent gather chains in flight.  Requires 32-byte aligned xi / yi.
// (Affine axes could gather the 16-byte value pair instead of the 32-byte record; measured within +-2 %
// of this kernel at 1e7 and 1e8 queries — the gather RATE bounds it, not the bytes — and not kept.)
template <typename T, bool WANT_IDX>
__global__ void __launch_bounds__(kThreads)
interp1_vec_kernel(AxisDev<T> ax, const T* __restrict__ seg, const T* __restrict__ xi, T* __restrict__ yi,
                   int32_t* __restrict__ idx, size_t nvec, T extrap) {
  constexpr int V = Vec256<T>::n;
  // programmatic dependent launch (plan1_launch): this grid may have been scheduled while the previous kernel of
  // the stream was still draining; nothing is read or written before that kernel has completed and flushed
  // (a no-op for an ordinary launch), and the next launch of the stream may be scheduled from now on
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;");
  const auto ld = make_loader1<T>(seg);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    T q[V], y[V];
    int32_t id[V];
    ld_stream_256(xi + i * V, q);
#pragma unroll
    for (int j = 0; j < V; ++j) y[j] = interp1_one<T>(ax, ld, q[j], extrap, id[j]);
    st_stream_256(yi + i * V, y);
    if (WANT_IDX) {
      if (V == 8) {
        st_stream_256(idx + i * V, reinterpret_cast<const int32_t(&)[8]>(id));
      } else {
        st_stream_128(idx + i * V, reinterpret_cast<const int32_t(&)[4]>(id));
      }
    }
  }
}

// Scalar kernel: tails and unaligned buffers.
template <typename T, bool WANT_IDX>
__global__ void __launch_bounds__(kThreads)
interp1_scalar_kernel(AxisDev<T> ax, const T* __restrict__ seg, const T* __restrict__ xi, T* __restrict__ yi,
                      int32_t* __restrict__ idx, size_t begin, size_t end, T extrap) {
  const auto ld = make_loader1<T>(seg);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = begin + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += stride) {
    int32_t id;
    yi[i] = interp1_one<T>(ax, ld, xi[i], extrap, id);
    if (WANT_IDX) idx[i] = id;
  }
}

// ---- small grids: the whole grid staged in shared memory ----
// The "coarse profile -> fine ensemble" case (a few thousand knots, millions of queries): persistent
// CTAs copy the knots, the values and (for non-uniform knots) the bucket table into shared memory
// once with TMA bulk copies and then stream queries; the bracket lookup and the two value reads never
// leave the SM, so HBM carries exactly 16 bytes (f64) per query.  Affine knots (linspace) are recomputed
// instead of staged: half the shared memory, half the bank-conflicted look-ups (0.79 vs 0.74 of peak).
constexpr int kSmem1Threads = 512;

template <typename T, bool WANT_IDX>
__global__ void __launch_bounds__(kSmem1Threads)
interp1_smem_kernel(AxisDev<T> ax, const T* __restrict__ yg, const T* __restrict__ xi, T* __restrict__ yi,
                    int32_t* __restrict__ idx, size_t nvec, T extrap) {
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
    int32_t id[V];
    ld_stream_256(xi + i * V, q);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const T qq = q[j];
      if (!(qq >= A.x0 && qq <= A.xmax)) { id[j] = -1; y[j] = (qq != qq) ? qnan<T>() : extrap; }
      else {
        T xa, xb;
        const int a = find_bracket_s(A, qq, xa, xb);
        id[j] = a;
        y[j] = blend(weight_of(xa, xb, qq), sy[a], sy[min(a + 1, A.n - 1)]);
      }
    }
    st_stream_256(yi + i * V, y);
    if (WANT_IDX) {
      if (V == 8) st_stream_256(idx + i * V, reinterpret_cast<const int32_t(&)[8]>(id));
      else st_stream_128(idx + i * V, reinterpret_cast<const int32_t(&)[4]>(id));
    }
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
  // staging for host-buffer execution (allocated on first use)
  void* st_in[2] = {nullptr, nullptr};
  void* st_out[2] = {nullptr, nullptr};
  int32_t* st_idx[2] = {nullptr, nullptr};
  size_t st_cap = 0;  // queries per slot
  StagePool pool;     // pinned ring for pageable host buffers
  cudaEvent_t ev[2] = {nullptr, nullptr};
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
  B200_CUDA(cudaEventCreateWithFlags(&p->ev[0], cudaEventDisableTiming));
  B200_CUDA(cudaEventCreateWithFlags(&p->ev[1], cudaEventDisableTiming));
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

// Launch on device buffers.  Vector path when xi/yi(/idx) are 32-byte aligned.
template <typename T>
int plan1_launch(b200_interp1_plan* p, const T* xi, size_t ni, T* yi, int32_t* idx, T extrap,
                 cudaStream_t st) {
  if (ni == 0) return B200_OK;
  constexpr int V = Vec256<T>::n;
  const AxisDev<T>& ax = axis_of<T>(p).dev;
  const T* seg = (const T*)p->seg;
  const bool aligned = (((uintptr_t)xi | (uintptr_t)yi) % 32 == 0) &&
                       (!idx || ((uintptr_t)idx % (V == 8 ? 32 : 16) == 0));
  size_t nvec = aligned ? ni / V : 0;
  if (nvec && p->smem_bytes && nvec >= 4096) {
    auto launch = [&](auto kern) -> int {
      unsigned grid = 0;
      B200_TRY(persistent_grid(kern, kSmem1Threads, p->smem_bytes, p->device, (nvec + kSmem1Threads - 1) / kSmem1Threads, grid));
      kern<<<grid, kSmem1Threads, p->smem_bytes, B200_CNT(st)>>>(ax, (const T*)p->yg, xi, yi, idx, nvec, extrap);
      return B200_OK;
    };
    if (idx) B200_TRY(launch(interp1_smem_kernel<T, true>));
    else B200_TRY(launch(interp1_smem_kernel<T, false>));
  } else if (nvec) {
    // a few waves of 8 resident CTAs per SM, grid-stride beyond that
    size_t blocks = (nvec + kThreads - 1) / kThreads;
    // measured: 1e7 queries 37.0 us with 16 CTAs per SM vs 38.9 us with 64; 1e8 queries 0.304 ms with 64 vs 0.316 ms with 16
    const size_t mult = blocks > (size_t)148 * 256 ? 64 : 16;
    int grid = (int)(blocks < (size_t)148 * mult ? blocks : (size_t)148 * mult);
    // back-to-back calls on one stream (a caller that batches, the chunks of the host-buffer pipeline): with the
    // programmatic-stream-serialization attribute the next grid is scheduled while this one drains and starts the
    // moment it has completed — no launch bubble between 30-60 us kernels
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = 0; cfg.stream = B200_CNT(st);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int32_t* no_idx = nullptr;
    if (idx) B200_CUDA(cudaLaunchKernelEx(&cfg, interp1_vec_kernel<T, true>, ax, seg, xi, yi, idx, nvec, extrap));
    else B200_CUDA(cudaLaunchKernelEx(&cfg, interp1_vec_kernel<T, false>, ax, seg, xi, yi, no_idx, nvec, extrap));
  }
  size_t done = nvec * V;
  if (done < ni) {
    size_t rem = ni - done;
    size_t blocks = (rem + kThreads - 1) / kThreads;
    int grid = (int)(blocks < (size_t)148 * 64 ? blocks : (size_t)148 * 64);
    if (idx) interp1_scalar_kernel<T, true><<<grid, kThreads, 0, B200_CNT(st)>>>(ax, seg, xi, yi, idx, done, ni, extrap);
    else interp1_scalar_kernel<T, false><<<grid, kThreads, 0, B200_CNT(st)>>>(ax, seg, xi, yi, nullptr, done, ni, extrap);
  }
  B200_CUDA(cudaGetLastError());
  return B200_OK;
}

constexpr size_t kChunk = (size_t)1 << 22;  // queries per pipeline slot

template <typename T>
int plan1_ensure_staging(b200_interp1_plan* p, size_t ni, bool want_idx) {
  size_t cap = ni < kChunk ? ni : kChunk;
  if (cap > p->st_cap) {
    for (int s = 0; s < 2; ++s) {
      cudaFree(p->st_in[s]); cudaFree(p->st_out[s]); cudaFree(p->st_idx[s]);
      p->st_in[s] = p->st_out[s] = nullptr; p->st_idx[s] = nullptr;
    }
    p->st_cap = 0;
    for (int s = 0; s < 2; ++s) {
      B200_CUDA(cudaMalloc(&p->st_in[s], cap * sizeof(T)));
      B200_CUDA(cudaMalloc(&p->st_out[s], cap * sizeof(T)));
    }
    p->st_cap = cap;
  }
  if (want_idx && !p->st_idx[0]) {
    for (int s = 0; s < 2; ++s) B200_CUDA(cudaMalloc(&p->st_idx[s], p->st_cap * sizeof(int32_t)));
  }
  return B200_OK;
}

// Host buffers: two slots, each on its own stream: H2D(chunk) -> kernel -> D2H(chunk);
// slot s+1's upload overlaps slot s's kernel and download (PCIe is full duplex).
template <typename T>
int plan1_exec_host(b200_interp1_plan* p, const T* xi, size_t ni, T* yi, int32_t* idx, T extrap) {
  if (ni == 0) return B200_OK;
  NvtxRange nvtx_call("interp1:exec_host");
  if (ni >= ((size_t)1 << 21) && (host_pageable(xi) || host_pageable(yi) || host_pageable(idx))) {
    // ordinary (pageable) arma::vec memory: pinned ring + copier threads (host_staging.cuh), same kernels
    std::vector<StageArray> arrays = {{xi, nullptr, sizeof(T)}, {nullptr, yi, sizeof(T)}};
    if (idx) arrays.push_back({nullptr, idx, sizeof(int32_t)});
    return staged_run(p->pool, p->device, arrays, ni, [&](const std::vector<void*>& d, size_t n, cudaStream_t st) {
      return plan1_launch<T>(p, (const T*)d[0], n, (T*)d[1], idx ? (int32_t*)d[2] : nullptr, extrap, st);
    });
  }
  B200_TRY(plan1_ensure_staging<T>(p, ni, idx != nullptr));
  const size_t cap = p->st_cap;
  int slot = 0;
  for (size_t off = 0; off < ni; off += cap, slot ^= 1) {
    size_t n = ni - off < cap ? ni - off : cap;
    cudaStream_t st = p->stream[slot];
    NvtxRange nvtx_slot(slot ? "interp1:slot1 h2d+kernel+d2h" : "interp1:slot0 h2d+kernel+d2h");
    B200_CUDA(cudaMemcpyAsync(p->st_in[slot], xi + off, n * sizeof(T), cudaMemcpyHostToDevice, st));
    B200_TRY(plan1_launch<T>(p, (const T*)p->st_in[slot], n, (T*)p->st_out[slot],
                             idx ? p->st_idx[slot] : nullptr, extrap, st));
    B200_CUDA(cudaMemcpyAsync(yi + off, p->st_out[slot], n * sizeof(T), cudaMemcpyDeviceToHost, st));
    if (idx)
      B200_CUDA(cudaMemcpyAsync(idx + off, p->st_idx[slot], n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  }
  B200_CUDA(cudaStreamSynchronize(p->stream[0]));
  B200_CUDA(cudaStreamSynchronize(p->stream[1]));
  return B200_OK;
}

void plan1_free(b200_interp1_plan* p) {
  p->ax64.release();
  p->ax32.release();
  cudaFree(p->yg);
  cudaFree(p->seg);
  for (int s = 0; s < 2; ++s) {
    cudaFree(p->st_in[s]); cudaFree(p->st_out[s]); cudaFree(p->st_idx[s]);
    if (p->stream[s]) cudaStreamDestroy(p->stream[s]);
    if (p->ev[s]) cudaEventDestroy(p->ev[s]);
  }
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
             ? plan1_exec_host<double>(p, (const double*)xi, ni, (double*)yi, idx_out, extrap_val)
             : plan1_exec_host<float>(p, (const float*)xi, ni, (float*)yi, idx_out, (float)extrap_val);
}

int b200_interp1_exec_dev(b200_interp1_plan* p, const void* xi_dev, size_t ni, void* yi_dev,
                          int32_t* idx_dev, double extrap_val, void* stream) {
  if (!p || (ni && (!xi_dev || !yi_dev))) return fail(B200_ERR_INVALID_ARG, "interp1_exec_dev: NULL argument");
  DeviceScope on_plan_device(p->device);
  cudaStream_t st = (cudaStream_t)stream;
  return p->dtype == B200_F64
             ? plan1_launch<double>(p, (const double*)xi_dev, ni, (double*)yi_dev, idx_dev, extrap_val, st)
             : plan1_launch<float>(p, (const float*)xi_dev, ni, (float*)yi_dev, idx_dev, (float)extrap_val, st);
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
