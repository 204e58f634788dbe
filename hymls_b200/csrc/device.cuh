// Small device/host helpers shared by the .cu files.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/hymls_b200.h"
#include "params.hpp"

namespace hymls {

#define HY_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      throw ::hymls::Error(HYMLS_B200_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + \
                                                    " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

// device memory held by the DevBuf and DeviceArena allocations of this process (hymls_b200_stats::device_bytes)
extern std::atomic<int64_t> g_deviceBytes;

// Bump allocator for the index arrays of one level.  A level holds ~100 immutable device arrays, sized once per
// sparsity pattern; cudaMalloc costs 3-10 ms a call on a 180 GB device (measured: 7 small allocations = 68 ms), so
// Initialize takes them from 256 MB slabs instead.  Memory goes back when the level is destroyed.
struct DeviceArena {
  size_t SLAB, DIRECT;  // slab size; requests of at least DIRECT bytes get an allocation of their own
  std::vector<void*> slabs;
  char* cur = nullptr;
  size_t left = 0;
  size_t held = 0;  // bytes of the slabs (counted in g_deviceBytes)
  explicit DeviceArena(size_t slab = (size_t)256 << 20, size_t direct = (size_t)64 << 20) : SLAB(slab), DIRECT(direct) {}
  DeviceArena(const DeviceArena&) = delete;
  DeviceArena& operator=(const DeviceArena&) = delete;
  ~DeviceArena() {
    for (void* p : slabs) cudaFree(p);
    g_deviceBytes -= (int64_t)held;
  }
  void* take(size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    void* p = nullptr;
    if (bytes >= DIRECT) {  // large arrays get their own allocation (still owned by the arena)
      HY_CUDA(cudaMalloc(&p, bytes));
      slabs.push_back(p);
      held += bytes;
      g_deviceBytes += (int64_t)bytes;
      return p;
    }
    if (bytes > left) {
      const size_t slab = bytes > SLAB ? bytes : SLAB;
      HY_CUDA(cudaMalloc(&p, slab));
      slabs.push_back(p);
      held += slab;
      g_deviceBytes += (int64_t)slab;
      cur = (char*)p;
      left = slab;
    }
    p = cur;
    cur += bytes;
    left -= bytes;
    return p;
  }
  // bump-allocate from memory somebody else owns first (e.g. the Compute workspace, idle during Initialize)
  void adopt(void* p, size_t bytes) {
    cur = (char*)p;
    left = bytes;
  }
  // a buffer that is re-allocated (grown) returns its memory: direct allocations are freed, slab pieces stay
  void giveBack(void* p, size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes < DIRECT) return;
    for (size_t k = 0; k < slabs.size(); ++k)
      if (slabs[k] == p) {
        cudaFree(p);
        held -= bytes;
        g_deviceBytes -= (int64_t)bytes;
        slabs.erase(slabs.begin() + k);
        return;
      }
  }
};
extern thread_local DeviceArena* g_arena;  // set by ArenaScope: DevBuf allocations of this thread come from it
struct ArenaScope {
  DeviceArena* prev;
  explicit ArenaScope(DeviceArena* a) : prev(g_arena) { g_arena = a; }
  ~ArenaScope() { g_arena = prev; }
};

// RAII device buffer (cudaMallocAsync-free: plain cudaMalloc or the level's arena, sized once per pattern)
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;    // elements in use
  size_t cap = 0;  // elements allocated (grow-only: cudaMalloc/cudaFree of GB-sized buffers stall for 100s of ms)
  DeviceArena* owner = nullptr;  // set when the memory came from an arena (which must outlive the buffer)
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p && owner) {
      owner->giveBack(p, cap * sizeof(T));
    } else if (p) {
      cudaFree(p);
      g_deviceBytes -= (int64_t)(cap * sizeof(T));
    }
    p = nullptr;
    n = 0;
    cap = 0;
    owner = nullptr;
  }
  void alloc(size_t count) {
    if (p && count <= cap) {
      n = count;
      return;
    }
    release();
    n = cap = count;
    if (!count) return;
    if (g_arena) {
      p = (T*)g_arena->take(count * sizeof(T));
      owner = g_arena;
    } else {
      HY_CUDA(cudaMalloc((void**)&p, count * sizeof(T)));
      g_deviceBytes += (int64_t)(count * sizeof(T));
    }
  }
  void upload(const std::vector<T>& h, cudaStream_t s) {
    alloc(h.size());
    if (!h.empty()) HY_CUDA(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  size_t bytes() const { return n * sizeof(T); }
};

// "largest opt-in dynamic shared memory size requested so far" of one kernel, tracked PER DEVICE: function
// attributes belong to the device/context, so a process-wide flag is wrong once a process drives two devices
struct PerDeviceLimit {
  size_t v[64];
  PerDeviceLimit() { for (size_t& x : v) x = 48 * 1024; }
  bool raise(size_t want) {  // true: the attribute has to be (re)set on the current device
    int d = 0;
    cudaGetDevice(&d);
    d &= 63;
    if (want <= v[d]) return false;
    v[d] = want;
    return true;
  }
};

}  // namespace hymls
