// interp2_banded.cuh — scattered interp2 for tables that do not fit L2: the L2-banded pipeline.
// Included by interp2.cu inside namespace b200::{anonymous}, after Plan2Dev / AxisSmem / BW.
//
// Why.  On B200 an L2 miss fills a whole 128-byte line, so 1e8 uniformly random 32-byte record gathers
// from a 512 MiB table move >= 10.8 GB of DRAM and cannot run faster than ~4.5e10 gathers/s
// (profiles/interp2_scattered_r1.md).  The 126 MB L2 is the way round it: cut the table into K column
// BANDS, visit the queries band by band, and the record gathers become L2 hits.  All DRAM traffic then
// is sequential:
//
//   B  band_bin      : a CTA takes a CHUNK of consecutive queries, finds the band of each (its
//                      x-bracket >> shift), partitions the chunk by band inside shared memory (rank =
//                      one shared-memory atomic per query) and writes (xq, yq) back as one contiguous
//                      block whose K segments are listed in a small table; pos16[i] = where query i
//                      went inside its chunk
//   C  band_interp   : one warp per (band, chunk) segment, in BAND-MAJOR order, so at any time the
//                      whole GPU gathers from one band: brackets, weights, record gather, three blends
//                      (a cp.async-pipelined variant of this pass was measured and was slower: the pass
//                      is bound by FP64 dependency chains at 24 warps/SM, not by bytes in flight)
//   D  band_unpermute: chunk by chunk, results back into query order through shared memory
//
// Arithmetic is the per-point restatement used everywhere else in this file (same weight_of/blend,
// individually rounded), so the results are bit-identical to the direct kernels and to the oracle.
#pragma once

constexpr int kBandThreads = 512;   // 4 consecutive queries per thread and round, 128 per warp
constexpr int kBandQ = 4;
constexpr int kBandRound = kBandThreads * kBandQ;   // 2048 queries per round; a chunk is 1 or 2 rounds
constexpr int kBandMaxK = 64;
constexpr size_t kBandBytes = (size_t)32 << 20;   // records per band (sweep: 64 MiB 2.52, 32 MiB 2.27, 16 MiB 2.27, 8 MiB 2.75 ms; profiles/interp2_banded_r1.md)

struct BandDev {
  int shift;          // band = ax >> shift
  int K;              // number of bands
  uint32_t nchunks;   // chunks in this slab
  uint32_t chunk;     // queries per chunk (2048 or 4096)
};

// four consecutive queries of a thread: one 256-bit (f64) / 128-bit (f32) streaming load when the
// array is 32-byte aligned and the four are inside the slab, guarded scalar loads otherwise
__device__ __forceinline__ void band_load4(const double* p, size_t i, size_t nq, bool vec, double (&v)[4]) {
  if (vec && i + 4 <= nq) { ld_stream_256(p + i, v); return; }
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = i + j < nq ? __ldcs(p + i + j) : 0.0;
}
__device__ __forceinline__ void band_load4(const float* p, size_t i, size_t nq, bool vec, float (&v)[4]) {
  if (vec && i + 4 <= nq) {
    const float4 t = __ldcs(reinterpret_cast<const float4*>(p + i));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    return;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) v[j] = i + j < nq ? __ldcs(p + i + j) : 0.f;
}
__device__ __forceinline__ void band_store4(double* p, size_t i, size_t nq, bool vec, const double (&v)[4]) {
  if (vec && i + 4 <= nq) { st_stream_256(p + i, v); return; }
#pragma unroll
  for (int j = 0; j < 4; ++j) if (i + j < nq) __stcs(p + i + j, v[j]);
}
__device__ __forceinline__ void band_store4(float* p, size_t i, size_t nq, bool vec, const float (&v)[4]) {
  if (vec && i + 4 <= nq) { __stcs(reinterpret_cast<float4*>(p + i), make_float4(v[0], v[1], v[2], v[3])); return; }
#pragma unroll
  for (int j = 0; j < 4; ++j) if (i + j < nq) __stcs(p + i + j, v[j]);
}

// ---- B: partition each chunk by band ----
// seg table: seg[b * nchunks + c] = start of band b inside chunk c (b = 0..K; entry K = chunk length)
template <typename T, int ROUNDS>
__global__ void __launch_bounds__(kBandThreads, 2)
band_bin_kernel(Plan2Dev<T> p, BandDev bd, const T* __restrict__ xq, const T* __restrict__ yq, size_t nq, int vec,
                uint16_t* __restrict__ seg, T* __restrict__ b_x, T* __restrict__ b_y, uint16_t* __restrict__ pos16) {
  constexpr int CHUNK = ROUNDS * kBandRound;
  extern __shared__ __align__(128) unsigned char smem2[];
  AxisSmem<T> X, Y;
  unsigned char* rest = stage_axes_smem<T>(p.X, p.Y, smem2, false, X, Y);
  T* img_x = reinterpret_cast<T*>(rest);
  T* img_y = img_x + CHUNK;
  uint32_t* hist = reinterpret_cast<uint32_t*>(img_y + CHUNK);   // [kBandMaxK] running count of each band
  uint32_t* segstart = hist + kBandMaxK;                         // [kBandMaxK + 1]
  const unsigned tid = threadIdx.x;
  if (tid < kBandMaxK) hist[tid] = 0;
  __syncthreads();
  for (uint32_t c = blockIdx.x; c < bd.nchunks; c += gridDim.x) {
    const size_t c0 = (size_t)c * CHUNK;
    T x[ROUNDS][kBandQ], y[ROUNDS][kBandQ];
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const size_t i0 = c0 + r * kBandRound + (size_t)tid * kBandQ;
      band_load4(xq, i0, nq, vec != 0, x[r]);
      band_load4(yq, i0, nq, vec != 0, y[r]);
    }
    uint32_t rank[ROUNDS][kBandQ];
    int band[ROUNDS][kBandQ];
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r)
#pragma unroll
      for (int j = 0; j < kBandQ; ++j) {
        const T q = x[r][j];
        int b = 0;   // out-of-range and NaN xi need no record: any band will do
        if (!((q < X.x0) || (q > X.xmax) || (q != q))) {
          T xa, xb;
          b = find_bracket_s(X, q, xa, xb) >> bd.shift;
        }
        band[r][j] = b;
        rank[r][j] = 0;
        if (c0 + r * kBandRound + (size_t)tid * kBandQ + j < nq) rank[r][j] = atomicAdd(&hist[b], 1u);
      }
    __syncthreads();
    if (tid < 32) {
      // K <= 64: two bands per lane, warp-level exclusive scan of the counts; reset them for the next chunk
      const uint32_t n0 = (int)(2 * tid) < bd.K ? hist[2 * tid] : 0, n1 = (int)(2 * tid + 1) < bd.K ? hist[2 * tid + 1] : 0;
      uint32_t inc = n0 + n1;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (tid >= (unsigned)d) inc += t;
      }
      const uint32_t ex = inc - n0 - n1;
      if ((int)(2 * tid) < bd.K) { segstart[2 * tid] = ex; seg[(size_t)(2 * tid) * bd.nchunks + c] = (uint16_t)ex; }
      if ((int)(2 * tid + 1) < bd.K) { segstart[2 * tid + 1] = ex + n0; seg[(size_t)(2 * tid + 1) * bd.nchunks + c] = (uint16_t)(ex + n0); }
      if (tid == 31) { segstart[bd.K] = inc; seg[(size_t)bd.K * bd.nchunks + c] = (uint16_t)inc; }   // chunk length
      hist[2 * tid] = 0;
      hist[2 * tid + 1] = 0;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const size_t i0 = c0 + r * kBandRound + (size_t)tid * kBandQ;
      uint16_t pos[kBandQ];
#pragma unroll
      for (int j = 0; j < kBandQ; ++j) {
        pos[j] = 0;
        if (i0 + j < nq) {
          const uint32_t q = segstart[band[r][j]] + rank[r][j];
          img_x[q] = x[r][j];
          img_y[q] = y[r][j];
          pos[j] = (uint16_t)q;
        }
      }
      if (i0 + kBandQ <= nq) {
        __stcs(reinterpret_cast<uint2*>(pos16 + i0), make_uint2((uint32_t)pos[0] | ((uint32_t)pos[1] << 16),
                                                                  (uint32_t)pos[2] | ((uint32_t)pos[3] << 16)));
      } else {
#pragma unroll
        for (int j = 0; j < kBandQ; ++j) if (i0 + j < nq) pos16[i0 + j] = pos[j];
      }
    }
    __syncthreads();
    // the partitioned chunk goes out as one contiguous block (the arrays are padded to whole chunks)
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const size_t o = c0 + r * kBandRound + (size_t)tid * kBandQ;
      T a[kBandQ], b[kBandQ];
#pragma unroll
      for (int j = 0; j < kBandQ; ++j) { a[j] = img_x[r * kBandRound + tid * kBandQ + j]; b[j] = img_y[r * kBandRound + tid * kBandQ + j]; }
      band_store4(b_x, o, o + kBandQ, true, a);
      band_store4(b_y, o, o + kBandQ, true, b);
    }
    // no barrier here: the next chunk writes the image only after two more barriers
  }
}

// ---- C: the interpolation, one warp per (band, chunk) segment in band-major order ----
__device__ __forceinline__ void ld_cell_keep(const double* p, double (&c)[4]) { ld_keep_256(p, c); }
__device__ __forceinline__ void ld_cell_keep(const float* p, float (&c)[4]) { ld_keep_128(p, c, l2_policy_evict_last()); }

// One query, split so that a thread can have several record gathers in flight: prepare() does the
// bracket lookups and weights and names the record; finish() blends (same case analysis as interp2_point_s:
// two_pass_special / two_pass).
template <typename T>
struct BandPrep { uint32_t cell; int fx, fy; T wx, wy; };

template <typename T>
__device__ __forceinline__ BandPrep<T> band_prepare(const AxisSmem<T>& X, const AxisSmem<T>& Y, T xq, T yq) {
  BandPrep<T> r;
  const BW<T> bx = bracket_weight_s<T>(X, xq);
  const BW<T> by = bracket_weight_s<T>(Y, yq);
  r.fx = bx.flag; r.fy = by.flag;
  r.wx = bx.w; r.wy = by.w;
  r.cell = (bx.flag | by.flag) ? 0u : (uint32_t)bx.a * (uint32_t)Y.n + (uint32_t)by.a;
  return r;
}
template <typename T>
__device__ __forceinline__ T band_finish(int yfirst, const BandPrep<T>& r, const T (&c)[4], T extrap) {
  T out;
  if (two_pass_special<T>(yfirst, r.fx, r.fy, r.wx, r.wy, extrap, out)) return out;
  return two_pass<T>(yfirst, r.wx, r.wy, c[0], c[1], c[2], c[3]);
}

constexpr int kBandCThreads = 256;

template <typename T>
__global__ void __launch_bounds__(kBandCThreads)
band_interp_kernel(Plan2Dev<T> p, BandDev bd, const uint16_t* __restrict__ seg, const T* __restrict__ b_x,
                   const T* __restrict__ b_y, T* __restrict__ res, T extrap) {
  extern __shared__ __align__(128) unsigned char smem2[];
  AxisSmem<T> X, Y;
  stage_axes_smem<T>(p.X, p.Y, smem2, true, X, Y);
  const unsigned lane = threadIdx.x & 31;
  const size_t nwarps = (size_t)gridDim.x * (kBandCThreads / 32);
  const size_t nitems = (size_t)bd.K * bd.nchunks;
  size_t item = (size_t)blockIdx.x * (kBandCThreads / 32) + (threadIdx.x >> 5);
  uint32_t s0 = 0, s1 = 0;
  if (item < nitems) { s0 = __ldg(seg + item); s1 = __ldg(seg + item + bd.nchunks); }
  for (; item < nitems; item += nwarps) {
    const uint32_t c = (uint32_t)(item % bd.nchunks);
    const size_t base = (size_t)c * bd.chunk;
    const uint32_t e0 = s0, e1 = s1;
    if (item + nwarps < nitems) {   // the next segment's bounds travel while this one is processed
      s0 = __ldg(seg + item + nwarps);
      s1 = __ldg(seg + item + nwarps + bd.nchunks);
    }
    for (uint32_t k0 = e0; k0 < e1; k0 += 128) {
      T x[4], y[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t k = k0 + j * 32 + lane;
        const bool on = k < e1;
        x[j] = on ? __ldcs(b_x + base + k) : qnan<T>();
        y[j] = on ? __ldcs(b_y + base + k) : qnan<T>();
      }
      BandPrep<T> pr[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) pr[j] = band_prepare<T>(X, Y, x[j], y[j]);
      // all four record gathers go out before the first blend (special cases gather record 0 and drop it)
      T q[4][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) ld_cell_keep(p.cells + 4 * (size_t)pr[j].cell, q[j]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t k = k0 + j * 32 + lane;
        const T v = band_finish<T>(p.yfirst, pr[j], q[j], extrap);
        if (k < e1) __stcs(res + base + k, v);
      }
    }
  }
}

// ---- D: results back into query order ----
template <typename T, int ROUNDS>
__global__ void __launch_bounds__(kBandThreads)
band_unpermute_kernel(uint32_t nchunks, const T* __restrict__ res, const uint16_t* __restrict__ pos16,
                      T* __restrict__ zq, size_t nq, int vec) {
  constexpr int CHUNK = ROUNDS * kBandRound;
  __shared__ __align__(32) T img[CHUNK];
  const unsigned tid = threadIdx.x;
  for (uint32_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
    const size_t c0 = (size_t)c * CHUNK;
    uint16_t pos[ROUNDS][kBandQ];
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const size_t i0 = c0 + r * kBandRound + (size_t)tid * kBandQ;
      if (i0 + kBandQ <= nq) {
        const uint2 t = __ldcs(reinterpret_cast<const uint2*>(pos16 + i0));
        pos[r][0] = (uint16_t)(t.x & 0xffff); pos[r][1] = (uint16_t)(t.x >> 16);
        pos[r][2] = (uint16_t)(t.y & 0xffff); pos[r][3] = (uint16_t)(t.y >> 16);
      } else {
#pragma unroll
        for (int j = 0; j < kBandQ; ++j) pos[r][j] = i0 + j < nq ? pos16[i0 + j] : (uint16_t)0;
      }
      T v[kBandQ];
      band_load4(res, i0, i0 + kBandQ, true, v);   // padded to whole chunks
#pragma unroll
      for (int j = 0; j < kBandQ; ++j) img[r * kBandRound + tid * kBandQ + j] = v[j];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const size_t i0 = c0 + r * kBandRound + (size_t)tid * kBandQ;
      T v[kBandQ];
#pragma unroll
      for (int j = 0; j < kBandQ; ++j) v[j] = img[pos[r][j]];
      band_store4(zq, i0, nq, vec != 0, v);
    }
    __syncthreads();
  }
}
