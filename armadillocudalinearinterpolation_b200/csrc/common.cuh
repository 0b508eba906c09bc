// common.cuh — shared plumbing of the C-ABI library (error text, CUDA call checking,
// cache-hinted 128/256-bit memory accessors for sm_100a).
//
// Replaces the reference's CUDA_CALL / CUDA_CHECK_ERROR / CURAND_CALL macros
// (EventDrivenMap.cu:12-54), which print and exit(-1): here every failure becomes a
// status code plus a thread-local message (b200_last_error()).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stddef.h>
#include <stdint.h>
#include "b200_common.h"

namespace b200 {

// NVTX range (header-only NVTX3: a no-op unless a profiler is attached) around host-side phases: the map's
// lift / evolve / reduce / all-gather (edm.cu) and the host-buffer calls of the interpolation plans (host_staging.cuh)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

// Entry points run on the device their plan / handle lives on and hand the caller's current device back on
// every exit path (dev < 0: only restore — for functions that switch between several devices themselves).
struct DeviceScope {
  int prev = -1;
  bool restore = false;
  explicit DeviceScope(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); return; }
    if (dev < 0) { restore = true; return; }
    if (dev != prev) { cudaSetDevice(dev); restore = true; }
  }
  ~DeviceScope() { if (restore) cudaSetDevice(prev); }
  DeviceScope(const DeviceScope&) = delete;
  DeviceScope& operator=(const DeviceScope&) = delete;
};

int fail(int status, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
// B200_OK if the current device is a compute-capability 10.x GPU (there is no CPU path).
int require_device();

#define B200_CUDA(call)                                                         \
  do {                                                                          \
    cudaError_t e__ = (call);                                                   \
    if (e__ != cudaSuccess) return ::b200::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)
// every kernel launch of the library goes through B200_CNT(stream) in its launch configuration, so
// b200_launch_count() (include/b200_common.h) is an exact count of this library's own launches
unsigned long long count_launch();
inline cudaStream_t counted_stream(cudaStream_t s) { count_launch(); return s; }
#define B200_CNT(stream) ::b200::counted_stream(stream)
#define B200_TRY(call)                \
  do {                                \
    int s__ = (call);                 \
    if (s__ != B200_OK) return s__;   \
  } while (0)

// Grow-only device scratch: reserve() keeps the allocation when it holds `need` bytes and replaces it otherwise.  A
// failed allocation leaves the buffer empty (p == nullptr, bytes == 0), never with a capacity it does not have.
struct DeviceBuffer {
  void* p = nullptr;
  size_t bytes = 0;
  int reserve(size_t need) {
    if (need <= bytes) return B200_OK;
    release();
    void* q = nullptr;
    B200_CUDA(cudaMalloc(&q, need));
    p = q;
    bytes = need;
    return B200_OK;
  }
  void release() { cudaFree(p); p = nullptr; bytes = 0; }
};

#ifdef __CUDACC__
// ---- streaming (touch-once) 256-bit accessors: bypass L1, first to leave L2 ----
__device__ __forceinline__ void ld_stream_256(const double* p, double (&v)[4]) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];"
               : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}
__device__ __forceinline__ void ld_stream_256(const float* p, float (&v)[8]) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
               : "l"(p));
}
__device__ __forceinline__ void st_stream_256(double* p, const double (&v)[4]) {
  asm volatile("st.global.L1::no_allocate.L2::evict_first.v4.f64 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "d"(v[0]), "d"(v[1]), "d"(v[2]), "d"(v[3]) : "memory");
}
__device__ __forceinline__ void st_stream_256(float* p, const float (&v)[8]) {
  asm volatile("st.global.L1::no_allocate.L2::evict_first.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ void st_stream_256(int32_t* p, const int32_t (&v)[8]) {
  asm volatile("st.global.L1::no_allocate.L2::evict_first.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               :: "l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void st_stream_128(int32_t* p, const int32_t (&v)[4]) {
  asm volatile("st.global.cs.v4.b32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
}
// ---- resident-table gathers: keep in L2 (evict_last) ----
__device__ __forceinline__ void ld_keep_256(const double* p, double (&v)[4]) {
  asm volatile("ld.global.nc.L2::evict_last.v4.f64 {%0,%1,%2,%3}, [%4];"
               : "=d"(v[0]), "=d"(v[1]), "=d"(v[2]), "=d"(v[3]) : "l"(p));
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void ld_keep_128(const double* p, double (&v)[2], uint64_t pol) {
  asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0,%1}, [%2], %3;"
               : "=d"(v[0]), "=d"(v[1]) : "l"(p), "l"(pol));
}
__device__ __forceinline__ void ld_keep_128(const float* p, float (&v)[4], uint64_t pol) {
  asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
               : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "l"(p), "l"(pol));
}
__device__ __forceinline__ void ld_keep_64(const float* p, float (&v)[2], uint64_t pol) {
  asm volatile("ld.global.nc.L2::cache_hint.v2.f32 {%0,%1}, [%2], %3;"
               : "=f"(v[0]), "=f"(v[1]) : "l"(p), "l"(pol));
}

// individually rounded arithmetic (never contracted into FMA): the interp blend must be
// bit-identical to Armadillo compiled without contraction (oracle: -ffp-contract=off)
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
#endif  // __CUDACC__

}  // namespace b200
