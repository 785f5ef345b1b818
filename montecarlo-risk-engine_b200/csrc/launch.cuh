// Host-side helpers shared by the entry points: path-shard descriptor, RNG descriptor
// conversion and validation (include/mcre.h: mcre_rng, mcre_shard).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace mcre {

struct ShardDev {
  long long path_begin, n_paths;
  int chunk;
};

inline RngDev make_rng(const mcre_rng *r) {
  RngDev d;
  d.mode = r->mode; d.k0 = (uint32_t)r->seed; d.k1 = (uint32_t)r->stream;
  d.z = r->d_z; d.u = r->d_u; d.n_total = r->n_paths_total;
  return d;
}
inline int check_shard(const mcre_shard *s) {
  if (!s || s->n_paths < 0 || s->chunk_paths <= 0 || s->chunk_paths % 256 != 0)
    return fail(-2, "invalid shard: chunk_paths must be a positive multiple of 256%s", "");
  if (s->path_begin % s->chunk_paths != 0) return fail(-2, "invalid shard: path_begin not chunk aligned%s", "");
  return 0;
}

// Dynamic shared memory of a launch of kernel k.  Above the 32 KB that every kernel gets without asking, the request
// is checked against the per-block opt-in limit (static shared memory included) before the attribute is set: a plan
// that cannot fit is refused with -3 and `what`, and the runtime is left without a pending error.
inline int set_dynamic_smem(const void *k, size_t smem, const char *what) {
  if (smem <= 32 * 1024) return 0;
  cudaFuncAttributes fa;
  MCRE_CUDA(cudaFuncGetAttributes(&fa, k));
  if (smem + fa.sharedSizeBytes > (size_t)smem_optin_limit()) return fail(-3, what, "", (long long)smem);
  MCRE_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return 0;
}
#define MCRE_SMEM(k, smem, what)                                 \
  do {                                                           \
    const int rc__ = mcre::set_dynamic_smem((const void *)(k), (smem), (what)); \
    if (rc__) return rc__;                                       \
  } while (0)

inline double pack2(int lo, int hi) {
  long long v = ((long long)(unsigned int)hi << 32) | (unsigned int)lo;
  double d;
  memcpy(&d, &v, 8);
  return d;
}

}  // namespace mcre
