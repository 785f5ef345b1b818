// Shared host-side helpers of libmcre_b200: error reporting, launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <vector>
#include "../../include/mcre.h"

namespace mcre {

extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;
extern std::atomic<long long> g_h2d_bytes;   // bytes this library copied host -> device (mcre_h2d_bytes)
#define MCRE_H2D(bytes) mcre::g_h2d_bytes.fetch_add((long long)(bytes), std::memory_order_relaxed)

inline int fail(int code, const char *fmt, const char *a = "", long long b = 0) {
  snprintf(g_err, sizeof(g_err), fmt, a, b);
  return code;
}
inline int cuda_fail(cudaError_t e, const char *what) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return (int)e;
}
#define MCRE_CUDA(call)                                      \
  do {                                                       \
    cudaError_t e__ = (call);                                \
    if (e__ != cudaSuccess) return mcre::cuda_fail(e__, #call); \
  } while (0)
#define MCRE_LAUNCHED()                                           \
  do {                                                            \
    mcre::g_launches.fetch_add(1, std::memory_order_relaxed);     \
    cudaError_t e__ = cudaGetLastError();                         \
    if (e__ != cudaSuccess) return mcre::cuda_fail(e__, "kernel launch"); \
  } while (0)

// One device allocation + one host-to-device copy for all tables of a plan: cudaMalloc / cudaFree
// cost ~0.1 ms each and a plan has ~40 tables, which showed up as several ms per run_simulation()
// call.  While an arena is open (ArenaScope) DevArray::upload stages into it; commit() allocates,
// copies once and patches every staged array's device pointer.
// Plan arenas come from a small process-wide cache of device blocks (power-of-two size classes): books of thousands
// of products create and destroy hundreds of plans and temporary tables per run, and cudaFree / cudaMalloc cost
// milliseconds each once the process holds GBs of device memory (measured: 5 - 50 ms per call in the large-book runs).
// A block goes back to the cache only after the device has drained (what cudaFree would have waited for, too).
int arena_cache_get(size_t bytes, void **out, size_t *cap);
void arena_cache_put(void *p, size_t cap);

struct DevArena {
  struct Item { void **slot; size_t off; };
  std::vector<unsigned char> stage;
  std::vector<Item> items;
  void *base = nullptr;
  void add(const void *host, size_t bytes, void **slot) {
    const size_t off = (stage.size() + 255) & ~(size_t)255;
    stage.resize(off + bytes);
    memcpy(stage.data() + off, host, bytes);
    items.push_back({slot, off});
  }
  size_t cap = 0;
  int commit() {
    if (stage.empty()) return 0;
    const int rc = arena_cache_get(stage.size(), &base, &cap);
    if (rc) return rc;
    MCRE_CUDA(cudaMemcpy(base, stage.data(), stage.size(), cudaMemcpyHostToDevice));
    MCRE_H2D(stage.size());
    for (const Item &it : items) *it.slot = (unsigned char *)base + it.off;
    std::vector<unsigned char>().swap(stage);
    items.clear();
    return 0;
  }
  void release() { if (base) arena_cache_put(base, cap); base = nullptr; cap = 0; }
};
extern thread_local DevArena *g_arena;
struct ArenaScope {
  explicit ArenaScope(DevArena *a) { g_arena = a; }
  ~ArenaScope() { g_arena = nullptr; }
};

// Device buffer filled from a host array (staged into the open arena, else its own allocation).
template <typename T>
struct DevArray {
  T *p = nullptr;
  size_t n = 0;
  bool owned = false;
  int upload(const T *host, size_t count) {
    n = count;
    if (count == 0 || host == nullptr) { p = nullptr; n = 0; return 0; }
    if (g_arena) { g_arena->add(host, count * sizeof(T), (void **)&p); return 0; }
    MCRE_CUDA(cudaMalloc((void **)&p, count * sizeof(T)));
    owned = true;
    MCRE_CUDA(cudaMemcpy(p, host, count * sizeof(T), cudaMemcpyHostToDevice));
    MCRE_H2D(count * sizeof(T));
    return 0;
  }
  void release() { if (p && owned) cudaFree(p); p = nullptr; n = 0; owned = false; }
};

int sm_count();
int smem_optin_limit();   // cudaDevAttrMaxSharedMemoryPerBlockOptin of the current device (cached)

}  // namespace mcre
