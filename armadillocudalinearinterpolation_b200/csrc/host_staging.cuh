// host_staging.cuh — host_run(), the one runner of every host-buffer query call of the interpolation plans
// (b200_interp1_exec / _grad, b200_interp2_scattered / _scattered_grad).
//
// Pinned (or small) buffers go through a two-slot pipeline on the plan's two streams: H2D chunk -> kernel -> D2H
// chunk, the upload of one slot overlapping the kernel and download of the other (PCIe is full duplex).
// A plain arma::vec (or numpy array) is pageable memory: cudaMemcpyAsync on it is staged by the driver on the
// calling thread, does not overlap with anything, and measured 5.5x slower end to end than pinned buffers
// (profiles/r2_e2e.md).  Large pageable batches therefore go through staged_run() instead: a few worker threads,
// each owning a stream and two slots of pinned + device chunk buffers, take the chunks round-robin — memcpy the
// chunk's inputs into the pinned slot, H2D, kernel, D2H into the pinned slot, and copy the previous chunk's outputs
// back to the caller while the GPU works on this one.
// Both run the device path's own kernels on the same values: results are bit-identical.
#pragma once
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>
#include "common.cuh"

namespace b200 {

inline bool host_pageable(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
  return a.type == cudaMemoryTypeUnregistered;
}

struct StageArray { const void* in; void* out; size_t elem; };   // exactly one of in / out is set

struct StagePool {
  static constexpr int kSlots = 2;
  struct Worker {
    cudaStream_t st = nullptr;
    cudaEvent_t ev[kSlots] = {nullptr, nullptr};
    std::vector<void*> pin[kSlots], dev[kSlots];
  };
  std::vector<Worker> workers;
  std::vector<size_t> elems;     // element size of every array the buffers were sized for
  size_t chunk = 0;
  int device = -1;

  void release() {
    if (device >= 0) cudaSetDevice(device);
    for (Worker& w : workers) {
      for (int s = 0; s < kSlots; ++s) {
        for (void* p : w.pin[s]) cudaFreeHost(p);
        for (void* p : w.dev[s]) cudaFree(p);
        if (w.ev[s]) cudaEventDestroy(w.ev[s]);
      }
      if (w.st) cudaStreamDestroy(w.st);
    }
    workers.clear(); elems.clear(); chunk = 0;
  }
  ~StagePool() { release(); }

  int ensure(int dev_id, int nworkers, size_t chunk_elems, const std::vector<StageArray>& arrays) {
    bool same = device == dev_id && (int)workers.size() == nworkers && chunk == chunk_elems && elems.size() == arrays.size();
    for (size_t a = 0; same && a < arrays.size(); ++a) same = elems[a] == arrays[a].elem;
    if (same) return B200_OK;
    release();
    const int rc = build(dev_id, nworkers, chunk_elems, arrays);
    if (rc != B200_OK) release();   // never leave a half-built pool behind: the next call would take it for complete
    return rc;
  }

  int build(int dev_id, int nworkers, size_t chunk_elems, const std::vector<StageArray>& arrays) {
    device = dev_id;
    chunk = chunk_elems;
    for (const StageArray& a : arrays) elems.push_back(a.elem);
    workers.resize(nworkers);
    for (Worker& w : workers) {
      B200_CUDA(cudaStreamCreateWithFlags(&w.st, cudaStreamNonBlocking));
      for (int s = 0; s < kSlots; ++s) {
        B200_CUDA(cudaEventCreateWithFlags(&w.ev[s], cudaEventDisableTiming));
        for (size_t e : elems) {
          void *hp = nullptr, *dp = nullptr;
          B200_CUDA(cudaHostAlloc(&hp, chunk * e, cudaHostAllocDefault));
          w.pin[s].push_back(hp);
          B200_CUDA(cudaMalloc(&dp, chunk * e));
          w.dev[s].push_back(dp);
        }
      }
    }
    return B200_OK;
  }
};

// launch(dev_ptrs (one per array, in the order of `arrays`), count, stream) -> status
template <class Launch>
int staged_run(StagePool& pool, int device, const std::vector<StageArray>& arrays, size_t n, Launch launch) {
  if (n == 0) return B200_OK;
  constexpr size_t kChunkElems = (size_t)1 << 20;
  unsigned hw = std::thread::hardware_concurrency();
  int nworkers = (int)(hw >= 16 ? 8 : (hw >= 4 ? hw / 2 : 1));
  const size_t nchunks = (n + kChunkElems - 1) / kChunkElems;
  if ((size_t)nworkers > nchunks) nworkers = (int)nchunks;
  B200_TRY(pool.ensure(device, nworkers, kChunkElems, arrays));
  std::vector<int> status(nworkers, B200_OK);
  std::vector<std::string> text(nworkers);
  auto body = [&](int t) {
    auto run = [&]() -> int {
      B200_CUDA(cudaSetDevice(device));
      StagePool::Worker& w = pool.workers[t];
      bool pending[StagePool::kSlots] = {false, false};
      size_t p_off[StagePool::kSlots] = {0, 0}, p_cnt[StagePool::kSlots] = {0, 0};
      auto drain = [&](int s) -> int {
        if (!pending[s]) return B200_OK;
        B200_CUDA(cudaEventSynchronize(w.ev[s]));
        for (size_t a = 0; a < arrays.size(); ++a)
          if (arrays[a].out) memcpy((char*)arrays[a].out + p_off[s] * arrays[a].elem, w.pin[s][a], p_cnt[s] * arrays[a].elem);
        pending[s] = false;
        return B200_OK;
      };
      int slot = 0;
      for (size_t c = (size_t)t; c < nchunks; c += (size_t)nworkers, slot ^= 1) {
        const size_t off = c * kChunkElems, cnt = n - off < kChunkElems ? n - off : kChunkElems;
        B200_TRY(drain(slot));
        NvtxRange nvtx_chunk("staged:chunk memcpy+h2d+kernel+d2h");
        for (size_t a = 0; a < arrays.size(); ++a)
          if (arrays[a].in) {
            memcpy(w.pin[slot][a], (const char*)arrays[a].in + off * arrays[a].elem, cnt * arrays[a].elem);
            B200_CUDA(cudaMemcpyAsync(w.dev[slot][a], w.pin[slot][a], cnt * arrays[a].elem, cudaMemcpyHostToDevice, w.st));
          }
        B200_TRY(launch(w.dev[slot], cnt, w.st));
        for (size_t a = 0; a < arrays.size(); ++a)
          if (arrays[a].out)
            B200_CUDA(cudaMemcpyAsync(w.pin[slot][a], w.dev[slot][a], cnt * arrays[a].elem, cudaMemcpyDeviceToHost, w.st));
        B200_CUDA(cudaEventRecord(w.ev[slot], w.st));
        pending[slot] = true; p_off[slot] = off; p_cnt[slot] = cnt;
      }
      for (int s = 0; s < StagePool::kSlots; ++s) B200_TRY(drain(s));
      return B200_OK;
    };
    status[t] = run();
    if (status[t] != B200_OK) text[t] = b200_last_error();   // the error text is thread-local: carry it over
  };
  std::vector<std::thread> th;
  bool spawn_failed = false;
  try {
    for (int t = 1; t < nworkers; ++t) th.emplace_back(body, t);
  } catch (...) {   // no exception may cross the C ABI; the chunks of the missing workers are not done -> the call fails
    spawn_failed = true;
  }
  body(0);
  for (std::thread& x : th) x.join();
  if (spawn_failed) return fail(B200_ERR_CUDA, "staged copy: could not start the worker threads");
  for (int t = 0; t < nworkers; ++t)
    if (status[t] != B200_OK) return fail(status[t], "%s", text[t].c_str());
  return B200_OK;
}

// Device buffers of the two-slot pipeline, one per slot and array position.  They only grow, so a plan whose calls
// alternate between array lists (value, value + index, gradient) keeps them: position 2 holds the int32 index of one
// call and the slope of the next.
struct HostSlots {
  std::vector<DeviceBuffer> buf[2];
  void release() {
    for (std::vector<DeviceBuffer>& s : buf)
      for (DeviceBuffer& b : s) b.release();
  }
};

// n queries in host memory: `arrays` (inputs and outputs, n elements each) through staged_run when any of them is
// pageable and n >= 2^21, else through the two-slot pipeline in chunks of 2^22 queries on `streams`; returns after
// both streams have finished.  `launch` as for staged_run.
template <class Launch>
int host_run(HostSlots& slots, cudaStream_t streams[2], StagePool& pool, int device, const char* label,
             const std::vector<StageArray>& arrays, size_t n, Launch launch) {
  if (n == 0) return B200_OK;
  NvtxRange nvtx_call(label);
  bool pageable = false;
  if (n >= ((size_t)1 << 21))
    for (const StageArray& a : arrays) pageable = pageable || host_pageable(a.in ? a.in : a.out);
  if (pageable) return staged_run(pool, device, arrays, n, launch);
  constexpr size_t kChunk = (size_t)1 << 22;
  const size_t cap = n < kChunk ? n : kChunk;
  std::vector<void*> d[2];
  for (int s = 0; s < 2; ++s) {
    if (slots.buf[s].size() < arrays.size()) slots.buf[s].resize(arrays.size());
    for (size_t a = 0; a < arrays.size(); ++a) {
      B200_TRY(slots.buf[s][a].reserve(cap * arrays[a].elem));
      d[s].push_back(slots.buf[s][a].p);
    }
  }
  int slot = 0;
  for (size_t off = 0; off < n; off += cap, slot ^= 1) {
    const size_t cnt = n - off < cap ? n - off : cap;
    cudaStream_t st = streams[slot];
    NvtxRange nvtx_slot(slot ? "slot1 h2d+kernel+d2h" : "slot0 h2d+kernel+d2h");
    for (size_t a = 0; a < arrays.size(); ++a)
      if (arrays[a].in)
        B200_CUDA(cudaMemcpyAsync(d[slot][a], (const char*)arrays[a].in + off * arrays[a].elem, cnt * arrays[a].elem,
                                  cudaMemcpyHostToDevice, st));
    B200_TRY(launch(d[slot], cnt, st));
    for (size_t a = 0; a < arrays.size(); ++a)
      if (arrays[a].out)
        B200_CUDA(cudaMemcpyAsync((char*)arrays[a].out + off * arrays[a].elem, d[slot][a], cnt * arrays[a].elem,
                                  cudaMemcpyDeviceToHost, st));
  }
  B200_CUDA(cudaStreamSynchronize(streams[0]));
  B200_CUDA(cudaStreamSynchronize(streams[1]));
  return B200_OK;
}

}  // namespace b200
