// Library-wide utilities: error state, launch accounting, the fixed-order tree reduction
// of per-chunk partial sums, and the FP64 FMA peak probe used as roofline denominator.
#include "common.cuh"
#include <algorithm>
#include <map>
#include <mutex>
#include <utility>

namespace mcre {
thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};
std::atomic<long long> g_h2d_bytes{0};
thread_local DevArena *g_arena = nullptr;

int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
    if (cached <= 0) cached = 148;
  }
  return cached;
}

int smem_optin_limit() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&cached, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (cached <= 0) cached = 48 * 1024;
  }
  return cached;
}

// Balanced pairwise sum over chunks, defined by a binary-counter stack: element i is pushed at
// level 0 and equal-level neighbours are merged immediately; leftover levels (non power-of-two
// counts) fold from the most recent to the oldest.  For a power-of-two count this is exactly the
// balanced binary tree over chunk indices, so a rank that owns an aligned power-of-two block of
// chunks produces a node of the global tree and the result is independent of how many GPUs the
// chunks were spread over.
//
// The tree is evaluated level by level, 32 elements at a time, so the loads of one thread are
// independent (the first version walked the chunks serially per slot: 2 ms of dependent-load
// latency per 4096-chunk reduction).  A full group of 32 aligned elements is a balanced subtree
// -> one element of the next level; the ragged tail of a level is the most recent part of the
// stack and is folded into the running `carry` before any older block, level by level.
constexpr int TREE_G = 32;

__device__ __forceinline__ double counter_fold(const double *v, int cnt, double carry, bool carry_valid) {
  double stack[8];
  int top = 0;
  for (int c = 0; c < cnt; ++c) {
    double x = v[c];
    int idx = c + 1;
    while ((idx & 1) == 0) { x = stack[--top] + x; idx >>= 1; }
    stack[top++] = x;
  }
  double s = carry;
  bool first = !carry_valid;
  while (top > 0) {
    const double x = stack[--top];
    s = first ? x : x + s;
    first = false;
  }
  return s;
}

// in: [n_in][n_slots].  Groups g < n_full: balanced sum of 32 rows -> next[g][slot].
// Group n_full (launched when there is a tail, or as the last level with n_full = 0):
// counter-fold of rows [32 n_full, n_in) with the incoming carry -> carry[slot].
__global__ void __launch_bounds__(128) tree_level_kernel(const double *in, long long n_in, long long n_slots,
                                                         long long n_full, double *next, double *carry,
                                                         int carry_valid) {
  const long long slot = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= n_slots) return;
  const long long g = blockIdx.y;
  double v[2 * TREE_G];
  if (g < n_full) {
#pragma unroll
    for (int i = 0; i < TREE_G; ++i) v[i] = in[(g * TREE_G + i) * n_slots + slot];
#pragma unroll
    for (int w = 1; w < TREE_G; w <<= 1)
#pragma unroll
      for (int i = 0; i < TREE_G; i += 2 * w) v[i] = v[i] + v[i + w];
    next[g * n_slots + slot] = v[0];
    return;
  }
  const int cnt = (int)(n_in - n_full * TREE_G);   // < 2 * TREE_G
#pragma unroll
  for (int i = 0; i < 2 * TREE_G; ++i) v[i] = i < cnt ? in[(n_full * TREE_G + i) * n_slots + slot] : 0.0;
  carry[slot] = counter_fold(v, cnt, carry_valid ? carry[slot] : 0.0, carry_valid != 0);
}

// sum(x - c), sum((x - c)^2) of rows of x [n_rows][n] with c = shift[row]: per-chunk block sums in a fixed order
// (the same chunks as the simulation kernels), combined by mcre_tree_reduce.  partial: [chunk][n_rows][2].
// mode 0: x, 1: max(x, 0), 2: -max(-x, 0)   (EPE / ENE integrands of spilled exposures)
__global__ void __launch_bounds__(256) sum_stats_kernel(const double *__restrict__ x, long long n, int n_rows, int chunk,
                                                        const double *__restrict__ shift, int mode,
                                                        double *__restrict__ partial) {
  __shared__ double stage[2 * 8];
  const long long ch = blockIdx.x;
  const int row = blockIdx.y;
  const double c = shift[row];
  double s1 = 0.0, s2 = 0.0;
  for (int it = threadIdx.x; it < chunk; it += blockDim.x) {
    const long long p = ch * chunk + it;
    if (p < n) {
      double v = x[(size_t)row * n + p];
      if (mode == 1) v = fmax(v, 0.0); else if (mode == 2) v = -fmax(-v, 0.0);
      const double d = v - c; s1 += d; s2 += d * d;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, off);
    s2 += __shfl_xor_sync(0xffffffffu, s2, off);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (lane == 0) { stage[warp * 2] = s1; stage[warp * 2 + 1] = s2; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += stage[w * 2 + threadIdx.x];
    partial[((size_t)ch * n_rows + row) * 2 + threadIdx.x] = t;
  }
}

// Register-resident DFMA chains: 16 independent accumulators per thread.
__global__ void dfma_peak_kernel(double *sink, int iters, double a, double b) {
  double x[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = (double)(threadIdx.x + i) * 1e-3;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) x[i] = fma(x[i], a, b);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i];
  if (s == 12345.6789) sink[0] = s;  // never true; keeps the chains alive
}
}  // namespace mcre

using namespace mcre;

namespace mcre {
namespace {
std::mutex g_arena_mu;
std::map<std::pair<int, size_t>, std::vector<void *>> g_arena_free;   // (device, size class) -> blocks
size_t g_arena_cached = 0;
constexpr size_t ARENA_CACHE_MAX = (size_t)1 << 30;                  // keep at most 1 GiB of idle blocks
}  // namespace

// A released block may still be read by kernels queued on some stream.  Instead of draining the whole device (which
// serialised every stream of the process and broke the asynchronous-on-the-caller's-stream contract of the entry
// points), the block is parked with an event recorded on the legacy default stream - which orders after the work
// queued so far on all blocking streams of the device, what the library's callers use - and goes back to the free list
// only once that event has completed (checked, without waiting, on later get / put calls).
namespace {
struct Parked { void *p; size_t cap; int dev; cudaEvent_t ev; };
std::vector<Parked> g_arena_parked;

void arena_cache_collect_locked() {
  size_t w = 0;
  for (size_t i = 0; i < g_arena_parked.size(); ++i) {
    Parked &k = g_arena_parked[i];
    if (cudaEventQuery(k.ev) == cudaSuccess) {
      cudaEventDestroy(k.ev);
      if (g_arena_cached + k.cap > ARENA_CACHE_MAX) cudaFree(k.p);
      else { g_arena_free[std::make_pair(k.dev, k.cap)].push_back(k.p); g_arena_cached += k.cap; }
    } else {
      cudaGetLastError();   // cudaErrorNotReady is not an error
      g_arena_parked[w++] = k;
    }
  }
  g_arena_parked.resize(w);
}
}  // namespace

int arena_cache_get(size_t bytes, void **out, size_t *cap) {
  size_t c = 4096;
  while (c < bytes) c <<= 1;
  int dev = 0;
  MCRE_CUDA(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lock(g_arena_mu);
    arena_cache_collect_locked();
    auto it = g_arena_free.find(std::make_pair(dev, c));
    if (it != g_arena_free.end() && !it->second.empty()) {
      *out = it->second.back();
      it->second.pop_back();
      g_arena_cached -= c;
      *cap = c;
      return 0;
    }
  }
  cudaError_t e = cudaMalloc(out, c);
  if (e != cudaSuccess) {
    // out of memory with idle blocks around: hand them back and retry once
    cudaGetLastError();
    cudaDeviceSynchronize();
    {
      std::lock_guard<std::mutex> lock(g_arena_mu);
      arena_cache_collect_locked();
      for (auto &kv : g_arena_free)
        for (void *p : kv.second) cudaFree(p);
      g_arena_free.clear();
      g_arena_cached = 0;
    }
    MCRE_CUDA(cudaMalloc(out, c));
  }
  *cap = c;
  return 0;
}

void arena_cache_put(void *p, size_t cap) {
  if (!p) return;
  int dev = 0;
  if (cap == 0 || cudaGetDevice(&dev) != cudaSuccess) { cudaFree(p); return; }
  cudaEvent_t ev;
  if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(ev, 0) != cudaSuccess) {
    cudaGetLastError();
    cudaDeviceSynchronize();
    cudaFree(p);
    return;
  }
  std::lock_guard<std::mutex> lock(g_arena_mu);
  g_arena_parked.push_back(Parked{p, cap, dev, ev});
  arena_cache_collect_locked();
}
}  // namespace mcre

// Level buffers of mcre_tree_reduce: one grow-only device buffer per (device, stream); work queued on a
// stream is ordered, so consecutive reductions on it can share the buffer.  (cudaMallocAsync was tried and
// cost more than the reduction: the default pool hands its memory back at every synchronisation.)
static int tree_scratch(cudaStream_t st, size_t bytes, double **out) {
  struct Buf { void *p = nullptr; size_t cap = 0; };
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, Buf> bufs;
  int dev = 0;
  MCRE_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  Buf &b = bufs[std::make_pair(dev, st)];
  if (b.cap < bytes) {
    if (b.p) { MCRE_CUDA(cudaStreamSynchronize(st)); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    const size_t cap = std::max(bytes, (size_t)4 << 20);
    MCRE_CUDA(cudaMalloc(&b.p, cap));
    b.cap = cap;
  }
  *out = (double *)b.p;
  return 0;
}

extern "C" int mcre_tree_reduce(const double *d_partial, int64_t n_chunks, int64_t n_slots, double *d_out,
                                void *stream) {
  if (!d_partial || !d_out) return fail(-1, "null argument%s", "");
  if (n_slots <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (n_chunks <= 0) { MCRE_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n_slots * sizeof(double), st)); return 0; }
  const int threads = 128;
  const unsigned bx = (unsigned)((n_slots + threads - 1) / threads);
  // level buffers: n/32 + n/1024 + ... rows, from a grow-only scratch kept per stream
  double *scratch = nullptr;
  size_t rows = 0;
  for (long long n = n_chunks; n >= 2 * TREE_G; n /= TREE_G) rows += (size_t)(n / TREE_G);
  if (rows) {
    const int rc = tree_scratch(st, rows * (size_t)n_slots * sizeof(double), &scratch);
    if (rc) return rc;
  }
  const double *in = d_partial;
  double *next = scratch;
  long long n = n_chunks;
  int carry_valid = 0;
  while (true) {
    const bool last = n < 2 * TREE_G;
    const long long n_full = last ? 0 : n / TREE_G;
    const bool tail = last || (n % TREE_G) != 0;
    dim3 grid(bx, (unsigned)(n_full + (tail ? 1 : 0)));
    tree_level_kernel<<<grid, threads, 0, st>>>(in, n, n_slots, n_full, next, d_out, carry_valid);
    MCRE_LAUNCHED();
    if (tail) carry_valid = 1;
    if (last) break;
    in = next;
    next += (size_t)n_full * n_slots;
    n = n_full;
  }
  return 0;
}

extern "C" int mcre_sum_stats(const double *d_x, int64_t n, int32_t n_rows, int32_t chunk_paths, const double *d_shift,
                              int32_t mode, double *d_partial, double *d_out, void *stream) {
  if (!d_x || !d_shift || !d_partial || !d_out) return fail(-1, "null argument%s", "");
  if (n_rows <= 0 || chunk_paths <= 0 || chunk_paths % 32 != 0) return fail(-2, "sum_stats: bad shape%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) { MCRE_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n_rows * 2 * sizeof(double), st)); return 0; }
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  dim3 grid((unsigned)n_chunks, (unsigned)n_rows);
  sum_stats_kernel<<<grid, 256, 0, st>>>(d_x, n, n_rows, chunk_paths, d_shift, mode, d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, (int64_t)n_rows * 2, d_out, stream);
}

extern "C" int mcre_dfma_peak(double *tflops_out, void *stream) {
  if (!tflops_out) return fail(-1, "null argument%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  double *sink = nullptr;
  MCRE_CUDA(cudaMalloc((void **)&sink, 8));
  const int threads = 256, blocks = sm_count() * 8, iters = 1 << 14;
  cudaEvent_t e0, e1;
  MCRE_CUDA(cudaEventCreate(&e0));
  MCRE_CUDA(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    MCRE_CUDA(cudaEventRecord(e0, st));
    dfma_peak_kernel<<<blocks, threads, 0, st>>>(sink, iters, 1.0000001, 1e-9);
    MCRE_LAUNCHED();
    MCRE_CUDA(cudaEventRecord(e1, st));
    MCRE_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    MCRE_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 16.0 * (double)iters * threads * blocks;
    const double tf = flops / (ms * 1e-3) * 1e-12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  *tflops_out = best;
  return 0;
}

extern "C" int64_t mcre_launch_count(void) { return g_launches.load(); }
extern "C" int64_t mcre_h2d_bytes(void) { return g_h2d_bytes.load(); }
extern "C" const char *mcre_last_error(void) { return g_err; }
extern "C" int mcre_abi_version(void) { return MCRE_ABI_VERSION; }
