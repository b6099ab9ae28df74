// Pieces shared by the VarDCT batch (batch.cc) and the Modular batch (modular_batch.cc): error plumbing, pooled
// device buffers, the pinned staging arena and the per-device context.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/jxg.h"

namespace jxgpu {
namespace detail {

extern thread_local std::string g_error;
inline int set_error(int code, const std::string& what) {
  g_error = what;
  return code;
}
#define CUDA_TRY(expr)                                                                        \
  do {                                                                                        \
    cudaError_t e__ = (expr);                                                                 \
    if (e__ != cudaSuccess) return set_error(JXG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    if (cudaMalloc(&p, want) != cudaSuccess) return set_error(JXG_ERR_CUDA, "cudaMalloc of " + std::to_string(want) + " bytes failed");
    cap = want;
    return 0;
  }
  ~DevBuf() {
    if (p) cudaFree(p);
  }
};

// Growable pinned host arena: the batch blob is assembled directly in pinned
// memory so that the upload is one cudaMemcpyAsync.
struct PinnedArena {
  uint8_t* p = nullptr;
  size_t size = 0, cap = 0;
  ~PinnedArena() {
    if (p) cudaFreeHost(p);
  }
  bool reserve(size_t want) {
    if (want <= cap) return true;
    size_t ncap = std::max(want, cap * 2);
    ncap = std::max<size_t>(ncap, 1 << 20);
    uint8_t* np = nullptr;
    if (cudaHostAlloc(reinterpret_cast<void**>(&np), ncap, cudaHostAllocDefault) != cudaSuccess) return false;
    if (p) {
      memcpy(np, p, size);
      cudaFreeHost(p);
    }
    p = np;
    cap = ncap;
    return true;
  }
  // Deferred mode (jxg_batch_set_deferred_copy): large copies are only recorded here and executed by
  // flush() on several host threads right before the upload; sources must stay valid until then.
  struct Pending {
    size_t off;
    const void* src;
    size_t bytes;
  };
  std::vector<Pending> pending;
  int deferred_threads = 0;
  // returns offset; pads with zeros up to `align`, appends `bytes` (+ `tail_zero` zero bytes)
  int64_t append(const void* src, size_t bytes, size_t align = 16, size_t tail_zero = 0) {
    size_t off = (size + align - 1) / align * align;
    size_t end = off + bytes + tail_zero;
    if (!reserve(end)) return -1;
    memset(p + size, 0, off - size);
    if (bytes) {
      if (deferred_threads > 0 && bytes >= 4096) pending.push_back(Pending{off, src, bytes});
      else memcpy(p + off, src, bytes);
    }
    if (tail_zero) memset(p + off + bytes, 0, tail_zero);
    size = end;
    return int64_t(off);
  }
  void flush() {
    if (pending.empty()) return;
    const int nt = std::max(1, std::min<int>(deferred_threads, int(pending.size())));
    std::atomic<size_t> next{0};
    auto work = [&] {
      for (;;) {
        const size_t i = next.fetch_add(8);
        if (i >= pending.size()) return;
        for (size_t j = i; j < std::min(i + 8, pending.size()); j++) memcpy(p + pending[j].off, pending[j].src, pending[j].bytes);
      }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nt; t++) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    pending.clear();
  }
};

// One D2H stream for all contexts of the device: output copies leave in launch order. With a copy stream per context
// the copies of all batches in flight share the host link evenly, so they all end together, all contexts come free
// together and the next batches start together: a convoy that leaves the SMs idle for the length of the D2H tail
// (profiles/r02l_e2e_convoy.log). First in, first out retires the oldest batch early and keeps the launches staggered.
// Created by the first jxg_init on the device; nullptr if that failed.
cudaStream_t device_d2h_stream(int device);

struct Context {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t d2h_stream = nullptr;  // device_d2h_stream (not owned): D2H of finished frame ranges overlaps the
                                      // filtering of later ranges
  static constexpr int kMaxRanges = 8;
  cudaEvent_t range_done[kMaxRanges] = {nullptr}, copy_done = nullptr;
  DevBuf dequant_default, dequant_default_off, natural_orders, natural_order_off;
  // Pools reused by successive batches (one live batch per context): device
  // intermediates and the pinned staging arena survive jxg_batch_end so that a
  // steady-state decode loop does no cudaMalloc / cudaHostAlloc.
  PinnedArena blob;
  DevBuf d_blob, d_coeffs, d_block_off, d_nz, d_planes_a, d_status, d_out, d_lean_desc, d_lean_nblk, d_orient, d_lzwin;
  bool batch_live = false;
  // pinned status readback buffer, owned by the context: cudaHostAlloc / cudaFreeHost synchronise the whole
  // device, so they must not happen per batch when batches of several contexts are in flight
  int32_t* status_host = nullptr;
  size_t status_cap = 0;
};


template <typename T>
int upload(DevBuf& b, const std::vector<T>& v, cudaStream_t s, uint64_t* counter) {
  if (int r = b.ensure(std::max<size_t>(v.size() * sizeof(T), 16))) return r;
  if (!v.empty()) CUDA_TRY(cudaMemcpyAsync(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  if (counter) *counter += v.size() * sizeof(T);
  return 0;
}

}  // namespace detail
}  // namespace jxgpu
