// Longstaff-Schwartz backward induction on spilled pre-simulation arrays.
//
// The reference regresses, for every regression date t_k (latest first), the deflated
// future cashflows of the product under the exercise policy already fitted for later dates
// (src/controller/controller.py:294-383): it rolls compute_normalized_cashflows over the
// product dates [t_next, last) for every starting state with float32 accumulators, adds
// the cached tail, and solves a tall least-squares problem in [1, x, x^2].
// For single-right exercise products (BermudanOption / AmericanOption,
// src/products/bermudan_option.py:93-188) state 0 (exercised) never carries value, so the
// roll collapses to one float32 running value V per path:
//     V <- fp32( fp32(ex ? imm_i / N_i : 0) + (ex ? 0 : V) ),   ex = imm_i > phi(x_i) . coef_i
// and the tall least squares to 8 moments per date.  One fused launch per regression date:
// HBM-bound, 5 coalesced f64 streams + the f32 value array (36 B / path / date).
#include "common.cuh"
#include "reduce.cuh"
#include "solve3.cuh"
#include <map>
#include <mutex>
#include <utility>

namespace mcre {

constexpr int LSM_MAX_RIGHTS = MCRE_LSM_MAX_RIGHTS;

struct LsmCoef { double c[LSM_MAX_RIGHTS][3]; };

// R exercise rights (1: Bermudan / American, up to 6: FlexiCall, src/products/flexicall.py:56-160).  The
// product state is the number of rights left; the roll keeps one float32 running value per path and state
// s = 1..R (value[s-1][n]; state 0 carries nothing).  Exercise update of product date i:
//     ex_s = imm_i + cont_i(s-1) > cont_i(s)                       (hard indicator, cont(0) = 0)
//     V_s <- fp32( fp32(ex_s ? imm_i / N_i : 0) + (ex_s ? V_{s-1} : V_s) )
// then the moments of regression date k: sum u^0..u^4 and per state sum u^0..u^2 N_k V_s  (5 + 3R).
// One (chunk) work item of the step: shared by the per-product kernel and the batched one, so both produce the same
// bits.  out: NV partial sums of this chunk.
template <int R>
__device__ __forceinline__ void lsm_step_item(const double *__restrict__ xk, const double *__restrict__ nk, double shift_k,
                                              double scale_k, const double *__restrict__ xi, const double *__restrict__ ni,
                                              const double *__restrict__ imm, int has_coef, const LsmCoef &cf, double shift_i,
                                              double scale_i, float *__restrict__ value, long long n, int chunk, long long ch,
                                              double *acc, double *stage, double *__restrict__ out) {
  constexpr int NV = 5 + 3 * R;
  if (threadIdx.x < NV) acc[threadIdx.x] = 0.0;
  __syncthreads();
  int parity = 0;
  // each thread first sums its own paths of the chunk (stride blockDim), the block reduces once
  double vals[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) vals[i] = 0.0;
  for (int it = 0; it < chunk; it += blockDim.x) {
    const long long p = ch * chunk + it + threadIdx.x;
    if (it + (int)threadIdx.x < chunk && p < n) {
      float v[R];
#pragma unroll
      for (int s = 0; s < R; ++s) v[s] = value[(size_t)s * n + p];
      if (imm) {
        const double im = imm[p];
        double cont[R + 1];
        cont[0] = 0.0;
        const double ui = has_coef ? (xi[p] - shift_i) * scale_i : 0.0;
#pragma unroll
        for (int s = 0; s < R; ++s) cont[s + 1] = has_coef ? cf.c[s][0] + ui * (cf.c[s][1] + ui * cf.c[s][2]) : 0.0;
        const double pay = im / ni[p];
        float nv[R];
#pragma unroll
        for (int s = 0; s < R; ++s) {
          const bool ex = im + cont[s] > cont[s + 1];
          // float32 step value updated with a float64 cashflow, then float32 + float32
          // (controller.py:330-349)
          const float step = (float)(ex ? pay : 0.0);
          const float prev = s > 0 ? v[s - 1] : 0.0f;
          nv[s] = step + (ex ? prev : v[s]);
        }
#pragma unroll
        for (int s = 0; s < R; ++s) { v[s] = nv[s]; value[(size_t)s * n + p] = nv[s]; }
      }
      const double u = (xk[p] - shift_k) * scale_k;
      const double u2 = u * u;
      vals[0] += 1.0; vals[1] += u; vals[2] += u2; vals[3] += u2 * u; vals[4] += u2 * u2;
#pragma unroll
      for (int s = 0; s < R; ++s) {
        const double y = nk[p] * (double)v[s];   // numeraire * total cashflows (controller.py:368)
        vals[5 + 3 * s] += y; vals[6 + 3 * s] += y * u; vals[7 + 3 * s] += y * u2;
      }
    }
  }
  block_accumulate<NV>(vals, acc, 0, stage, NV, parity);
  __syncthreads();
  if (threadIdx.x < NV) out[threadIdx.x] = acc[threadIdx.x];
  __syncthreads();
}

template <int R>
__global__ void __launch_bounds__(256) lsm_step_kernel(const double *__restrict__ xk, const double *__restrict__ nk,
                                                       double shift_k, double scale_k, const double *__restrict__ xi,
                                                       const double *__restrict__ ni, const double *__restrict__ imm,
                                                       int has_coef, LsmCoef cf, double shift_i,
                                                       double scale_i, float *__restrict__ value, long long n, int chunk,
                                                       double *__restrict__ partial) {
  constexpr int NV = 5 + 3 * R;
  __shared__ double acc[NV];
  __shared__ double stage[2 * 8 * NV];
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x)
    lsm_step_item<R>(xk, nk, shift_k, scale_k, xi, ni, imm, has_coef, cf, shift_i, scale_i, value, n, chunk, ch, acc, stage,
                     partial + ch * NV);
}

// Single-right step with the continuation coefficients of product date i read from DEVICE memory (d_coef, 3 doubles,
// or NULL): the backward induction of one Bermudan option then runs as a stream of kernels - step, tree reduction,
// (all-reduce,) 3x3 solve - without reading the moments back per date (mcre/lsm.py:backward_induction_device).
__global__ void __launch_bounds__(256) lsm_step_dev_kernel(const double *__restrict__ xk, const double *__restrict__ nk,
                                                           double shift_k, double scale_k, const double *__restrict__ xi,
                                                           const double *__restrict__ ni, const double *__restrict__ imm,
                                                           const double *__restrict__ d_coef, double shift_i, double scale_i,
                                                           float *__restrict__ value, long long n, int chunk,
                                                           double *__restrict__ partial) {
  constexpr int NV = 8;
  __shared__ double acc[NV];
  __shared__ double stage[2 * 8 * NV];
  LsmCoef cf;
#pragma unroll
  for (int s = 0; s < LSM_MAX_RIGHTS; ++s)
#pragma unroll
    for (int q = 0; q < 3; ++q) cf.c[s][q] = (d_coef && s == 0) ? d_coef[q] : 0.0;
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x)
    lsm_step_item<1>(xk, nk, shift_k, scale_k, xi, ni, imm, d_coef != nullptr, cf, shift_i, scale_i, value, n, chunk, ch, acc,
                     stage, partial + ch * NV);
}

// coefficients of one regression date from its 8 moments (sum u^0..u^4, sum u^0..u^2 Y)
__global__ void lsm_solve_dev_kernel(const double *__restrict__ moments, double *__restrict__ coef) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double c[3];
    solve_normal_equations_dev(moments, moments + 5, c);
    coef[0] = c[0]; coef[1] = c[1]; coef[2] = c[2];
  }
}

// The steps of MANY exercise products in one launch (the lock-step backward inductions of a book: one job per
// product and round).  Work item = (job, chunk); the moments of every job sit in a row of LSM_NV_MAX doubles
// (unused tail zero).  partial: [chunk][job][LSM_NV_MAX].
constexpr int LSM_NV_MAX = 5 + 3 * LSM_MAX_RIGHTS;
struct LsmStepJob {
  int n_rights, has_coef;
  const double *xk, *nk;
  double shift_k, scale_k;
  const double *xi, *ni, *imm;
  double coef[3 * LSM_MAX_RIGHTS];
  double shift_i, scale_i;
  float *value;
};
__global__ void __launch_bounds__(256) lsm_step_batch_kernel(const LsmStepJob *__restrict__ jobs, long long n_jobs, long long n,
                                                             int chunk, double *__restrict__ partial) {
  __shared__ double acc[LSM_NV_MAX];
  __shared__ double stage[2 * 8 * LSM_NV_MAX];
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long w = blockIdx.x; w < n_jobs * n_chunks; w += gridDim.x) {
    const long long j = w / n_chunks, ch = w - j * n_chunks;
    const LsmStepJob *job = jobs + j;
    LsmCoef cf;
#pragma unroll
    for (int s = 0; s < LSM_MAX_RIGHTS; ++s)
#pragma unroll
      for (int q = 0; q < 3; ++q) cf.c[s][q] = job->coef[s * 3 + q];
    double *out = partial + ((size_t)ch * n_jobs + j) * LSM_NV_MAX;
    const int R = job->n_rights;
    if (threadIdx.x >= 5 + 3 * R && threadIdx.x < LSM_NV_MAX) out[threadIdx.x] = 0.0;
#define LSM_ITEM(RV) lsm_step_item<RV>(job->xk, job->nk, job->shift_k, job->scale_k, job->xi, job->ni, job->imm, job->has_coef, \
                                       cf, job->shift_i, job->scale_i, job->value, n, chunk, ch, acc, stage, out)
    if (R == 1) LSM_ITEM(1); else if (R == 2) LSM_ITEM(2); else if (R == 3) LSM_ITEM(3); else if (R == 4) LSM_ITEM(4);
    else if (R == 5) LSM_ITEM(5); else LSM_ITEM(6);
#undef LSM_ITEM
  }
}

// Moments of many (product, regression date) pairs in ONE launch: books of thousands of products on ~1000
// pre-simulation paths are launch-bound when every pair costs a kernel + a tree reduction (380k launches for the
// reference's 5000-product exposure book).  Work item = (job, chunk); per item exactly the arithmetic of
// lsm_step_kernel<1> without an exercise update and with a constant numeraire, so the sums are bit-identical to
// the per-job calls.  partial: [chunk][job][8].
struct LsmJob { const double *x; const float *v; double nk, shift, scale; };
__global__ void __launch_bounds__(256) lsm_moments_batch_kernel(const LsmJob *__restrict__ jobs, long long n_jobs, long long n,
                                                                int chunk, double *__restrict__ partial) {
  constexpr int NV = 8;
  __shared__ double acc[NV];
  __shared__ double stage[2 * 8 * NV];
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long w = blockIdx.x; w < n_jobs * n_chunks; w += gridDim.x) {
    const long long j = w / n_chunks, ch = w - j * n_chunks;
    const LsmJob job = jobs[j];
    if (threadIdx.x < NV) acc[threadIdx.x] = 0.0;
    __syncthreads();
    int parity = 0;
    double vals[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) vals[i] = 0.0;
    for (int it = 0; it < chunk; it += blockDim.x) {
      const long long p = ch * chunk + it + threadIdx.x;
      if (it + (int)threadIdx.x < chunk && p < n) {
        const double u = (job.x[p] - job.shift) * job.scale;
        const double u2 = u * u;
        vals[0] += 1.0; vals[1] += u; vals[2] += u2; vals[3] += u2 * u; vals[4] += u2 * u2;
        const double y = job.nk * (double)job.v[p];
        vals[5] += y; vals[6] += y * u; vals[7] += y * u2;
      }
    }
    block_accumulate<NV>(vals, acc, 0, stage, NV, parity);
    __syncthreads();
    if (threadIdx.x < NV) partial[((size_t)ch * n_jobs + j) * NV + threadIdx.x] = acc[threadIdx.x];
    __syncthreads();
  }
}

// Tangent companion of lsm_step_kernel<R> for R = 2..6 rights (R = 1: lsm_step_tan_kernel, csrc/irc_tan.cu), run after
// the value step of the same regression date.  For parameter blockIdx.y it recomputes the exercise decisions with the
// double expressions of lsm_step_item<R> (so they are the value pass's decisions) and applies them to the running
// tangents, every state from the values before the update:
//     dV_s <- ex_s ? d(imm_i / N_i) + dV_{s-1} : dV_s,   d(imm / N) = (dimm - (imm / N) dN) / N,   dV_0 = 0
// then accumulates the tangent moments of date k with Y_s = N_k V_s, dY_s = dN_k V_s + N_k dV_s (V_s the float32 value
// the value step has already written): [0..3] sum u^m du (shared by the states), per state s at 4 + 5 s:
// sum dY, u dY, u^2 dY, du Y, 2 u du Y.  dvalue: [R][nt][n] f64; partial: [chunk][nt][4 + 5 R].
template <int R>
__global__ void __launch_bounds__(256) lsm_step_states_tan_kernel(
    int nt, const double *__restrict__ xk, const double *__restrict__ nk, const double *__restrict__ dxk,
    const double *__restrict__ dnk, double shift_k, double scale_k, const double *__restrict__ xi,
    const double *__restrict__ ni, const double *__restrict__ imm, const double *__restrict__ dni,
    const double *__restrict__ dimm, int has_coef, LsmCoef cf, double shift_i, double scale_i,
    const float *__restrict__ value, double *__restrict__ dvalue, long long n, int chunk, double *__restrict__ partial) {
  constexpr int NV = 4 + 5 * R;
  __shared__ double acc[NV];
  __shared__ double stage[2 * 8 * NV];
  const int ip = blockIdx.y;
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    if (threadIdx.x < NV) acc[threadIdx.x] = 0.0;
    __syncthreads();
    int parity = 0;
    double vals[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) vals[j] = 0.0;
    for (int it = 0; it < chunk; it += blockDim.x) {
      const long long p = ch * chunk + it + threadIdx.x;
      if (it + (int)threadIdx.x < chunk && p < n) {
        double dv[R];
#pragma unroll
        for (int s = 0; s < R; ++s) dv[s] = dvalue[((size_t)s * nt + ip) * n + p];
        if (imm) {
          const double im = imm[p];
          double cont[R + 1];
          cont[0] = 0.0;
          const double ui = has_coef ? (xi[p] - shift_i) * scale_i : 0.0;
#pragma unroll
          for (int s = 0; s < R; ++s) cont[s + 1] = has_coef ? cf.c[s][0] + ui * (cf.c[s][1] + ui * cf.c[s][2]) : 0.0;
          const double inv = 1.0 / ni[p];
          const double dpay = (dimm[(size_t)ip * n + p] - im * inv * dni[(size_t)ip * n + p]) * inv;
          double nd[R];
#pragma unroll
          for (int s = 0; s < R; ++s) {
            const bool ex = im + cont[s] > cont[s + 1];
            nd[s] = ex ? dpay + (s > 0 ? dv[s - 1] : 0.0) : dv[s];
          }
#pragma unroll
          for (int s = 0; s < R; ++s) { dv[s] = nd[s]; dvalue[((size_t)s * nt + ip) * n + p] = nd[s]; }
        }
        const double uu = (xk[p] - shift_k) * scale_k, du = dxk[(size_t)ip * n + p] * scale_k;
        const double u2 = uu * uu, nkp = nk[p], dnkp = dnk[(size_t)ip * n + p];
        vals[0] += du; vals[1] += uu * du; vals[2] += u2 * du; vals[3] += u2 * uu * du;
#pragma unroll
        for (int s = 0; s < R; ++s) {
          const double V = (double)value[(size_t)s * n + p];
          const double Y = nkp * V, dY = dnkp * V + nkp * dv[s];
          double *o = vals + 4 + 5 * s;
          o[0] += dY; o[1] += uu * dY; o[2] += u2 * dY; o[3] += du * Y; o[4] += 2.0 * uu * du * Y;
        }
      }
    }
    block_accumulate<NV>(vals, acc, 0, stage, NV, parity);
    __syncthreads();
    if (threadIdx.x < NV) partial[((size_t)ch * nt + ip) * NV + threadIdx.x] = acc[threadIdx.x];
    __syncthreads();
  }
}

// Pathwise tangents of the arrays of mcre_lsm_prepare_equity from the tangent spill of the pre-simulation
// (mcre_eq_presim_tangents, dx [n_rows][A][nt][n]): blockIdx.y = output row (n_reg regression dates, then n_ex exercise
// dates), threads over paths.
//   dxs[k][j]  = dx[reg_row[k]][x_asset][j]                 (tangent of the explanatory spot)
//   dnum[k][j] = j == rate_slot ? reg_dnum[k] : 0           (the deterministic numeraire moves with the rate only)
//   dimm[i][j] = imm[i] > 0 ? sign dx[ex_row[i]][u_asset][j] : 0
__global__ void __launch_bounds__(256) lsm_prepare_equity_tan_kernel(const double *__restrict__ dx, long long n, int A, int nt,
                                                                     int n_reg, const int *__restrict__ reg_row,
                                                                     const double *__restrict__ reg_dnum, int rate_slot,
                                                                     int x_asset, int n_ex, const int *__restrict__ ex_row,
                                                                     int u_asset, double sign, const double *__restrict__ imm,
                                                                     double *__restrict__ dxs, double *__restrict__ dnum,
                                                                     double *__restrict__ dimm) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int k = blockIdx.y;
  if (k < n_reg) {
    const double *src = dx + ((size_t)reg_row[k] * A + x_asset) * nt * n;
    for (int j = 0; j < nt; ++j) {
      dxs[((size_t)k * nt + j) * n + p] = src[(size_t)j * n + p];
      dnum[((size_t)k * nt + j) * n + p] = j == rate_slot ? reg_dnum[k] : 0.0;
    }
  } else {
    const int i = k - n_reg;
    const double *src = dx + ((size_t)ex_row[i] * A + u_asset) * nt * n;
    const bool itm = imm[(size_t)i * n + p] > 0.0;
    for (int j = 0; j < nt; ++j) dimm[((size_t)i * nt + j) * n + p] = itm ? sign * src[(size_t)j * n + p] : 0.0;
  }
}

// Gathers the regression / exercise inputs of an equity exercise product from materialised paths
// [n_paths][n_dates][state_dim]: blockIdx.y = output row (n_reg regression dates, then n_ex exercise dates), threads
// over paths: date-major outputs (coalesced writes) and enough threads in flight for books on ~1000 paths (one
// thread per path walking all dates was latency bound: 8 ms per product).
__global__ void __launch_bounds__(256) lsm_prepare_equity_kernel(const double *__restrict__ paths, long long n, int n_dates,
                                                                 int state_dim, int n_reg, const int *__restrict__ reg_date,
                                                                 const double *__restrict__ reg_num, int n_ex,
                                                                 const int *__restrict__ ex_date, int x_col, int x_is_log,
                                                                 int n_under, const int *__restrict__ ucol,
                                                                 const double *__restrict__ uw, const int *__restrict__ ulog,
                                                                 double strike, const double *__restrict__ ex_strike,
                                                                 double sign, double *__restrict__ x, double *__restrict__ num,
                                                                 double *__restrict__ imm) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const double *row = paths + (size_t)p * n_dates * state_dim;
  const int k = blockIdx.y;
  if (k < n_reg) {
    const double v = row[(size_t)reg_date[k] * state_dim + x_col];
    x[(size_t)k * n + p] = x_is_log ? exp(v) : v;
    num[(size_t)k * n + p] = reg_num[k];
  } else {
    const int i = k - n_reg;
    const double *st = row + (size_t)ex_date[i] * state_dim;
    double U = 0.0;
    for (int j = 0; j < n_under; ++j) {
      const double v = st[ucol[j]];
      U += uw[j] * (ulog[j] ? exp(v) : v);
    }
    imm[(size_t)i * n + p] = fmax((U - (ex_strike ? ex_strike[i] : strike)) * sign, 0.0);
  }
}

}  // namespace mcre

using namespace mcre;

extern "C" int mcre_lsm_prepare_equity(const double *d_paths, int64_t n_paths, int32_t n_dates, int32_t state_dim,
                                       int32_t n_reg, const int32_t *reg_date, const double *reg_numeraire, int32_t n_ex,
                                       const int32_t *ex_date, int32_t x_col, int32_t x_is_log, int32_t n_under,
                                       const int32_t *under_col, const double *under_w, const int32_t *under_is_log,
                                       double strike, const double *ex_strike, double sign, double *d_x, double *d_n,
                                       double *d_imm, void *stream) {
  if (!d_paths || !reg_date || !reg_numeraire || !ex_date || !under_col || !under_w || !under_is_log || !d_x || !d_n || !d_imm)
    return fail(-1, "null argument%s", "");
  if (n_paths <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DevArray<int> rd, ed, uc, ul;
  DevArray<double> rn, uw, xs;
  DevArena arena;   // the index tables travel in one allocation + one copy
  ArenaScope arena_scope(&arena);
  int rc = rd.upload(reg_date, n_reg);
  if (!rc && ex_strike) rc = xs.upload(ex_strike, n_ex);
  if (!rc) rc = ed.upload(ex_date, n_ex);
  if (!rc) rc = uc.upload(under_col, n_under);
  if (!rc) rc = ul.upload(under_is_log, n_under);
  if (!rc) rc = rn.upload(reg_numeraire, n_reg);
  if (!rc) rc = uw.upload(under_w, n_under);
  if (!rc) rc = arena.commit();
  if (!rc) {
    lsm_prepare_equity_kernel<<<dim3((unsigned)((n_paths + 255) / 256), (unsigned)(n_reg + n_ex)), 256, 0, st>>>(
        d_paths, n_paths, n_dates, state_dim, n_reg, rd.p, rn.p, n_ex, ed.p, x_col, x_is_log, n_under, uc.p, uw.p, ul.p,
        strike, xs.p, sign, d_x, d_n, d_imm);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "kernel launch");
    else cudaStreamSynchronize(st);   // the temporary index tables are freed below
  }
  rd.release(); ed.release(); uc.release(); ul.release(); rn.release(); uw.release(); xs.release();
  arena.release();
  return rc;
}

extern "C" int mcre_lsm_prepare_equity_tangents(const double *d_dx, int64_t n_paths, int32_t n_assets, int32_t nt,
                                                int32_t n_reg, const int32_t *reg_row, const double *reg_dnum,
                                                int32_t rate_slot, int32_t x_asset, int32_t n_ex, const int32_t *ex_row,
                                                int32_t u_asset, double sign, const double *d_imm, double *d_dxs,
                                                double *d_dnum, double *d_dimm, void *stream) {
  if (!d_dx || !reg_row || !reg_dnum || !ex_row || !d_imm || !d_dxs || !d_dnum || !d_dimm) return fail(-1, "null argument%s", "");
  if (nt < 1 || n_assets < 1 || x_asset < 0 || x_asset >= n_assets || u_asset < 0 || u_asset >= n_assets)
    return fail(-1, "lsm prepare tangents: asset or parameter count out of range%s", "");
  if (n_paths <= 0 || n_reg + n_ex <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DevArray<int> rr, er;
  DevArray<double> rd;
  DevArena arena;
  ArenaScope arena_scope(&arena);
  int rc = rr.upload(reg_row, n_reg);
  if (!rc) rc = er.upload(ex_row, n_ex);
  if (!rc) rc = rd.upload(reg_dnum, n_reg);
  if (!rc) rc = arena.commit();
  if (!rc) {
    lsm_prepare_equity_tan_kernel<<<dim3((unsigned)((n_paths + 255) / 256), (unsigned)(n_reg + n_ex)), 256, 0, st>>>(
        d_dx, n_paths, n_assets, nt, n_reg, rr.p, rd.p, rate_slot, x_asset, n_ex, er.p, u_asset, sign, d_imm, d_dxs, d_dnum,
        d_dimm);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "kernel launch");
    else cudaStreamSynchronize(st);   // the temporary index tables are freed below
  }
  rr.release(); er.release(); rd.release();
  arena.release();
  return rc;
}

extern "C" int mcre_lsm_step_states_tangents(int32_t n_rights, int32_t nt, const double *d_xk, const double *d_nk,
                                             const double *d_dxk, const double *d_dnk, double shift_k, double scale_k,
                                             const double *d_xi, const double *d_ni, const double *d_imm,
                                             const double *d_dni, const double *d_dimm, const double *coef_i,
                                             double shift_i, double scale_i, const float *d_value, double *d_dvalue,
                                             int64_t n, int32_t chunk_paths, double *d_partial, double *d_tmoments,
                                             void *stream) {
  if (n_rights < 1 || n_rights > LSM_MAX_RIGHTS) return fail(-3, "lsm: 1..6 exercise rights are supported%s", "");
  if (n_rights == 1)   // one right: the rate family's kernel, bit for bit
    return mcre_lsm_step_tangents(nt, d_xk, d_nk, d_dxk, d_dnk, shift_k, scale_k, d_xi, d_ni, d_imm, d_dni, d_dimm, coef_i,
                                  shift_i, scale_i, d_value, d_dvalue, n, chunk_paths, d_partial, d_tmoments, stream);
  if (!d_xk || !d_nk || !d_dxk || !d_dnk || !d_value || !d_dvalue || !d_partial || !d_tmoments)
    return fail(-1, "null argument%s", "");
  if (nt < 1) return fail(-1, "lsm tangents: nt must be positive%s", "");
  if (d_imm && (!d_xi || !d_ni || !d_dni || !d_dimm)) return fail(-1, "lsm tangents: exercise update needs its arrays%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  const int nv = 4 + 5 * n_rights;
  if (n <= 0) {
    MCRE_CUDA(cudaMemsetAsync(d_tmoments, 0, (size_t)nt * nv * sizeof(double), st));
    return 0;
  }
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long gx = (long long)sm_count() * 4;
  if (gx > n_chunks) gx = n_chunks;
  dim3 grid((unsigned)gx, (unsigned)nt);
  LsmCoef cf;
  for (int s = 0; s < LSM_MAX_RIGHTS; ++s)
    for (int j = 0; j < 3; ++j) cf.c[s][j] = (coef_i && s < n_rights) ? coef_i[s * 3 + j] : 0.0;
#define LSM_TAN_LAUNCH(RV)                                                                                              \
  lsm_step_states_tan_kernel<RV><<<grid, 256, 0, st>>>(nt, d_xk, d_nk, d_dxk, d_dnk, shift_k, scale_k, d_xi, d_ni, d_imm, \
                                                       d_dni, d_dimm, coef_i != nullptr, cf, shift_i, scale_i, d_value,  \
                                                       d_dvalue, n, chunk_paths, d_partial)
  if (n_rights == 2) LSM_TAN_LAUNCH(2); else if (n_rights == 3) LSM_TAN_LAUNCH(3); else if (n_rights == 4) LSM_TAN_LAUNCH(4);
  else if (n_rights == 5) LSM_TAN_LAUNCH(5); else LSM_TAN_LAUNCH(6);
#undef LSM_TAN_LAUNCH
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, (int64_t)nt * nv, d_tmoments, stream);
}

extern "C" int mcre_lsm_step_states(int32_t n_rights, const double *d_xk, const double *d_nk, double shift_k,
                                    double scale_k, const double *d_xi, const double *d_ni, const double *d_imm,
                                    const double *coef_i, double shift_i, double scale_i, float *d_value, int64_t n,
                                    int32_t chunk_paths, double *d_partial, double *d_moments, void *stream) {
  if (!d_xk || !d_nk || !d_value || !d_partial || !d_moments) return fail(-1, "null argument%s", "");
  if (n_rights < 1 || n_rights > LSM_MAX_RIGHTS) return fail(-3, "lsm: 1..6 exercise rights are supported%s", "");
  if (d_imm && (!d_xi || !d_ni)) return fail(-1, "lsm: exercise update needs x_i and N_i%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  const int nv = 5 + 3 * n_rights;
  if (n <= 0) {   // a rank without pre-simulation paths contributes zero moments
    MCRE_CUDA(cudaMemsetAsync(d_moments, 0, nv * sizeof(double), st));
    return 0;
  }
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long grid = (long long)sm_count() * 8;
  if (grid > n_chunks) grid = n_chunks;
  LsmCoef cf;
  for (int s = 0; s < LSM_MAX_RIGHTS; ++s)
    for (int j = 0; j < 3; ++j) cf.c[s][j] = (coef_i && s < n_rights) ? coef_i[s * 3 + j] : 0.0;
#define LSM_LAUNCH(RV)                                                                                          \
  lsm_step_kernel<RV><<<(unsigned)grid, 256, 0, st>>>(d_xk, d_nk, shift_k, scale_k, d_xi, d_ni, d_imm,          \
                                                      coef_i != nullptr, cf, shift_i, scale_i, d_value, n,     \
                                                      chunk_paths, d_partial)
  if (n_rights == 1) LSM_LAUNCH(1); else if (n_rights == 2) LSM_LAUNCH(2); else if (n_rights == 3) LSM_LAUNCH(3);
  else if (n_rights == 4) LSM_LAUNCH(4); else if (n_rights == 5) LSM_LAUNCH(5); else LSM_LAUNCH(6);
#undef LSM_LAUNCH
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, nv, d_moments, stream);
}

extern "C" int mcre_lsm_step_dev(const double *d_xk, const double *d_nk, double shift_k, double scale_k, const double *d_xi,
                                 const double *d_ni, const double *d_imm, const double *d_coef_i, double shift_i,
                                 double scale_i, float *d_value, int64_t n, int32_t chunk_paths, double *d_partial,
                                 double *d_moments, void *stream) {
  if (!d_xk || !d_nk || !d_value || !d_partial || !d_moments) return fail(-1, "null argument%s", "");
  if (d_imm && (!d_xi || !d_ni)) return fail(-1, "lsm: exercise update needs x_i and N_i%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) {   // a rank without pre-simulation paths contributes zero moments
    MCRE_CUDA(cudaMemsetAsync(d_moments, 0, 8 * sizeof(double), st));
    return 0;
  }
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long grid = (long long)sm_count() * 8;
  if (grid > n_chunks) grid = n_chunks;
  lsm_step_dev_kernel<<<(unsigned)grid, 256, 0, st>>>(d_xk, d_nk, shift_k, scale_k, d_xi, d_ni, d_imm, d_coef_i, shift_i,
                                                      scale_i, d_value, n, chunk_paths, d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, 8, d_moments, stream);
}

extern "C" int mcre_lsm_solve_dev(const double *d_moments, double *d_coef, void *stream) {
  if (!d_moments || !d_coef) return fail(-1, "null argument%s", "");
  lsm_solve_dev_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(d_moments, d_coef);
  MCRE_LAUNCHED();
  return 0;
}

// Job tables of the batched launches: one grow-only device buffer per (device, stream); the upload is ordered on
// the stream after the previous launch that read the buffer.
static int job_scratch(cudaStream_t st, size_t bytes, void **out) {
  struct Buf { void *p = nullptr; size_t cap = 0; };
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, Buf> bufs;
  int dev = 0;
  MCRE_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  Buf &b = bufs[std::make_pair(dev, st)];
  if (b.cap < bytes) {
    if (b.p) { MCRE_CUDA(cudaStreamSynchronize(st)); cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t cap = (size_t)1 << 20;
    while (cap < bytes) cap <<= 1;
    MCRE_CUDA(cudaMalloc(&b.p, cap));
    b.cap = cap;
  }
  *out = b.p;
  return 0;
}

extern "C" int mcre_lsm_step_batch(int64_t n_jobs, const mcre_lsm_step_job *jobs, int64_t n, int32_t chunk_paths,
                                   double *d_partial, double *d_moments, void *stream) {
  if (n_jobs <= 0) return 0;
  if (!jobs || !d_partial || !d_moments) return fail(-1, "null argument%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  static_assert(sizeof(LsmStepJob) == sizeof(mcre_lsm_step_job), "job record layout");
  for (int64_t j = 0; j < n_jobs; ++j) {
    if (jobs[j].n_rights < 1 || jobs[j].n_rights > LSM_MAX_RIGHTS) return fail(-3, "lsm: 1..6 exercise rights are supported%s", "");
    if (!jobs[j].xk || !jobs[j].nk || !jobs[j].value) return fail(-1, "lsm batch: null job array%s", "");
    if (jobs[j].imm && (!jobs[j].xi || !jobs[j].ni)) return fail(-1, "lsm: exercise update needs x_i and N_i%s", "");
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) {
    MCRE_CUDA(cudaMemsetAsync(d_moments, 0, (size_t)n_jobs * LSM_NV_MAX * sizeof(double), st));
    return 0;
  }
  void *d_jobs = nullptr;
  int rc = job_scratch(st, (size_t)n_jobs * sizeof(LsmStepJob), &d_jobs);
  if (rc) return rc;
  MCRE_CUDA(cudaMemcpyAsync(d_jobs, jobs, (size_t)n_jobs * sizeof(LsmStepJob), cudaMemcpyHostToDevice, st));
  MCRE_H2D((size_t)n_jobs * sizeof(LsmStepJob));
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long grid = (long long)sm_count() * 8;
  if (grid > n_jobs * n_chunks) grid = n_jobs * n_chunks;
  lsm_step_batch_kernel<<<(unsigned)grid, 256, 0, st>>>((const LsmStepJob *)d_jobs, n_jobs, n, chunk_paths, d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, n_jobs * LSM_NV_MAX, d_moments, stream);
}

extern "C" int mcre_lsm_moments_batch(int64_t n_jobs, const mcre_lsm_job *jobs, int64_t n, int32_t chunk_paths,
                                      double *d_partial, double *d_moments, void *stream) {
  if (n_jobs <= 0) return 0;
  if (!jobs || !d_partial || !d_moments) return fail(-1, "null argument%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  static_assert(sizeof(LsmJob) == sizeof(mcre_lsm_job), "job record layout");
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) {
    MCRE_CUDA(cudaMemsetAsync(d_moments, 0, (size_t)n_jobs * 8 * sizeof(double), st));
    return 0;
  }
  void *d_jobs_v = nullptr;
  int rc = job_scratch(st, (size_t)n_jobs * sizeof(LsmJob), &d_jobs_v);
  if (rc) return rc;
  LsmJob *d_jobs = (LsmJob *)d_jobs_v;
  MCRE_CUDA(cudaMemcpyAsync(d_jobs, jobs, (size_t)n_jobs * sizeof(LsmJob), cudaMemcpyHostToDevice, st));
  MCRE_H2D((size_t)n_jobs * sizeof(LsmJob));
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long grid = (long long)sm_count() * 8;
  if (grid > n_jobs * n_chunks) grid = n_jobs * n_chunks;
  lsm_moments_batch_kernel<<<(unsigned)grid, 256, 0, st>>>(d_jobs, n_jobs, n, chunk_paths, d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, n_jobs * 8, d_moments, stream);
}

extern "C" int mcre_lsm_step(const double *d_xk, const double *d_nk, double shift_k, double scale_k, const double *d_xi,
                             const double *d_ni, const double *d_imm, const double *coef_i, double shift_i,
                             double scale_i, float *d_value, int64_t n, int32_t chunk_paths, double *d_partial,
                             double *d_moments, void *stream) {
  return mcre_lsm_step_states(1, d_xk, d_nk, shift_k, scale_k, d_xi, d_ni, d_imm, coef_i, shift_i, scale_i, d_value, n,
                              chunk_paths, d_partial, d_moments, stream);
}
