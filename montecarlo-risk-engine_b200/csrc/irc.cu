// Interest-rate / credit family: fused path generation + cashflows + exposure + metrics.
//
// One thread owns one path for its whole life: the Vasicek (and CIR++) state lives in
// registers, normals come from Philox in registers (or from the reference's injected
// draws), and at every simulation date the thread evaluates the netted cashflows, the
// regression-proxy exposure, threshold / MPoR collateral and the metric integrands.
// Only block-reduced sums ever reach HBM.  See include/mcre.h for what each entry point
// replaces in the reference.
#include <algorithm>
#include <cstdlib>
#include "irc_main.cuh"
#include "irc_value.cuh"

namespace mcre {


// =====================================================================================
// Pre-simulation pass A: forward simulation, spills per regression date the explanatory
// variable, the numeraire and the FP32 window sums of each unit's discounted cashflows.
// scratch: x [n_reg][n] f64 | N [n_reg][n] f64 | W [n_units][n_reg][n] f32
//
// Round 2: lock-step like the main kernels (PP paths per thread, every operation interleaved over them - the
// round-1 version ran one path per thread on libdevice exp and took 3.4 ms of the 4.5 ms pre-simulation of the
// headline config).  Only the short rate and the numeraire integral are stepped: rate products read nothing else,
// the credit factor's normal is skipped (Philox is counter based: no stream to keep aligned; the injected stream is
// indexed).  NU = regression units of the launch (window accumulators per path).
// =====================================================================================
constexpr int PRE_PP = 4;
template <bool CIR, int SCHEME, int NU>
__global__ void __launch_bounds__(128, 4) irc_presim_forward_kernel(IrcDev P, RngDev rng, ShardDev sh, double *xbuf,
                                                                   double *nbuf, float *wbuf) {
  constexpr int PP = PRE_PP;
  fm_tables_init();
  const long long n = sh.n_paths;
  const long long base = (long long)blockIdx.x * (128 * PP) + threadIdx.x;
  if (base - threadIdx.x >= n) return;
  long long lpath[PP], gpath[PP];
  bool live[PP];
  MCRE_VP {
    lpath[p] = base + p * 128;
    live[p] = lpath[p] < n;
    gpath[p] = sh.path_begin + (live[p] ? lpath[p] : 0);
  }
  NormalStreamV<PP> nsv;
  nsv.init(rng, gpath);
  const bool inject = rng.mode == MCRE_RNG_INJECT;
  const double r0 = __ldg(P.vas + 0), sigma = __ldg(P.vas + 1), theta = __ldg(P.vas + 2), a = __ldg(P.vas + 3);
  // correlated noise of the short rate: row vas_noise of the lower Cholesky factor (model.py:46-48)
  const bool second = CIR && P.vas_noise == 1;
  const double l0 = CIR ? __ldg(P.chol + (second ? 2 : 0)) : __ldg(P.chol + 0);
  const double l1 = second ? __ldg(P.chol + 3) : 0.0;
  double r[PP], logB[PP], zb[PP];
  float W[PP][NU];
  MCRE_VP {
    r[p] = r0; logB[p] = 0.0; zb[p] = 0.0;
#pragma unroll
    for (int u = 0; u < NU; ++u) W[p][u] = 0.0f;
  }

  auto eval_date = [&](int di) {
    const int flags = __ldg(P.date_flags + di);
    if (!(flags & (MCRE_DATE_HAS_CASHFLOW | MCRE_DATE_HAS_REGRESSION))) return;
    double numeraire[PP];
    fm_exp_tv<PP>(logB, numeraire);                    // vasicek.py:154-156
    if (flags & MCRE_DATE_HAS_CASHFLOW) {
      double cf[PP][NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        const double fx = u < P.n_units ? __ldg(P.unit_fix + (size_t)u * P.n_dates + di) : 0.0;
        MCRE_VP cf[p][u] = fx;
      }
      const int j0 = __ldg(P.date_float_off + di), j1 = __ldg(P.date_float_off + di + 1);
      for (int j = j0; j < j1; ++j) {
        // LIBOR from the zero bond at the payment date's own short rate: (1 / P - 1) / tau with
        // 1 / P = exp(B r - alpha) (bond.py:55-66, vasicek.py:114-128)
        const double alpha = __ldg(P.float_coef + j * 2), B = __ldg(P.float_coef + j * 2 + 1);
        const double inv_tau = __ldg(P.float_inv_tau + j);
        double xa[PP], ip[PP];
        MCRE_VP xa[p] = fma(B, r[p], -alpha);
        fm_exp_tv<PP>(xa, ip);
        MCRE_VP ip[p] = (ip[p] - 1.0) * inv_tau;
#pragma unroll
        for (int u = 0; u < NU; ++u) {
          if (u < P.n_units) {
            const double wgt = __ldg(P.unit_float + (size_t)u * P.n_float + j);
            MCRE_VP cf[p][u] = fma(ip[p], wgt, cf[p][u]);
          }
        }
      }
      // FP32 accumulator updated with an FP64 addend: W <- fp32(fp64(W) + cf / N)
      // (controller.py:330,341: float32 step_value += float64 cashflows)
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        MCRE_VP W[p][u] = (float)((double)W[p][u] + fm_div(cf[p][u], numeraire[p]));
      }
    }
    if (flags & MCRE_DATE_HAS_REGRESSION) {
      const int k = __ldg(P.date_reg + di);
      MCRE_VP {
        if (live[p]) {
          xbuf[(size_t)k * n + lpath[p]] = r[p];
          nbuf[(size_t)k * n + lpath[p]] = numeraire[p];
        }
      }
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        MCRE_VP {
          if (u < P.n_units && k > 0 && live[p]) wbuf[((size_t)u * P.n_reg + (k - 1)) * n + lpath[p]] = W[p][u];
          W[p][u] = 0.0f;  // cashflows at or before the first regression date never enter a window
        }
      }
    }
  };
  for (int di = 0; di < P.n_pre_dates; ++di) eval_date(di);
#pragma unroll 1
  for (int is = 0; is < P.n_sub; ++is) {
    const double dt = __ldg(P.step_dt + is);
    const double sv0 = __ldg(P.step_vas + is * 2), sv1 = __ldg(P.step_vas + is * 2 + 1);
    double z0[PP], z1[PP];
    if (inject) {
      MCRE_VP {
        const double *zp = rng.z + ((size_t)is * rng.n_total + gpath[p]) * (CIR ? 2 : 1);
        z0[p] = zp[0];
        z1[p] = CIR ? zp[1] : 0.0;
      }
    } else if (CIR) {
      nsv.next2(z0, z1);                               // normals 2 is, 2 is + 1 of the path
    } else {
      // one normal per step: a Box-Muller pair serves two steps
      if ((is & 1) == 0) nsv.next2(z0, zb);
      else { MCRE_VP z0[p] = zb[p]; }
      MCRE_VP z1[p] = 0.0;
    }
    MCRE_VP logB[p] = fma(P.ext_num ? P.ext_rate : r[p], dt, logB[p]);          // left Riemann sum with the pre-step rate (vasicek.py:80,107)
    if (SCHEME == MCRE_SCHEME_ANALYTICAL) {
      // exact OU transition; the 1x1 Cholesky factor of the step covariance is sv1 (vasicek.py:52-86)
      MCRE_VP r[p] = fma(sv1, z0[p], fma(r[p] - theta, sv0, theta));
    } else {
      // r + a (theta_t - r) dt + sigma sqrt(dt) w   (vasicek.py:88-112)
      const double adt = a * dt, ssq = sigma * sqrt(dt);
      const double k0 = ssq * l0, k1 = ssq * l1;
      MCRE_VP r[p] = fma(k0, z0[p], fma(sv0 - r[p], adt, r[p]));
      if (second) { MCRE_VP r[p] = fma(k1, z1[p], r[p]); }
    }
    const int di = __ldg(P.step_date + is);
    if (di >= 0) eval_date(di);
  }
#pragma unroll
  for (int u = 0; u < NU; ++u) {
    MCRE_VP {
      if (u < P.n_units && P.n_reg > 0 && live[p]) wbuf[((size_t)u * P.n_reg + (P.n_reg - 1)) * n + lpath[p]] = W[p][u];
    }
  }
}

// Pre-simulation of Bermudan units, forward pass: spills per regression date the explanatory
// variable and the numeraire, and per exercise record the immediate exercise value.
// scratch: x [n_reg][n] | N [n_reg][n] | imm [n_ex][n], all f64
// Lock-step like irc_presim_forward_kernel (PRE_PP paths per thread; the zero-bond exponentials of the underlying,
// ~20 per exercise date of a 10y swap, are evaluated PP-wide on the table-driven exp).
template <bool CIR, int SCHEME>
__global__ void __launch_bounds__(128, 4) irc_lsm_forward_kernel(IrcDev P, RngDev rng, ShardDev sh, double *xbuf,
                                                                 double *nbuf, double *ibuf) {
  constexpr int PP = PRE_PP;
  fm_tables_init();
  const long long n = sh.n_paths;
  const long long base = (long long)blockIdx.x * (128 * PP) + threadIdx.x;
  if (base - threadIdx.x >= n) return;
  long long lpath[PP], gpath[PP];
  bool live[PP];
  MCRE_VP {
    lpath[p] = base + p * 128;
    live[p] = lpath[p] < n;
    gpath[p] = sh.path_begin + (live[p] ? lpath[p] : 0);
  }
  NormalStreamV<PP> nsv;
  nsv.init(rng, gpath);
  const bool inject = rng.mode == MCRE_RNG_INJECT;
  const double r0 = __ldg(P.vas + 0), sigma = __ldg(P.vas + 1), theta = __ldg(P.vas + 2), a = __ldg(P.vas + 3);
  const bool second = CIR && P.vas_noise == 1;
  const double l0 = CIR ? __ldg(P.chol + (second ? 2 : 0)) : __ldg(P.chol + 0);
  const double l1 = second ? __ldg(P.chol + 3) : 0.0;
  double r[PP], logB[PP], zb[PP];
  MCRE_VP { r[p] = r0; logB[p] = 0.0; zb[p] = 0.0; }
  auto eval_date = [&](int di) {
    const int flags = __ldg(P.date_flags + di);
    if (flags & MCRE_DATE_HAS_REGRESSION) {
      const int k = __ldg(P.date_reg + di);
      double numeraire[PP];
      fm_exp_tv<PP>(logB, numeraire);
      MCRE_VP {
        if (live[p]) {
          xbuf[(size_t)k * n + lpath[p]] = r[p];
          nbuf[(size_t)k * n + lpath[p]] = numeraire[p];
        }
      }
    }
    if (flags & MCRE_DATE_HAS_EXERCISE) {
      const int x0 = __ldg(P.date_ex_off + di), x1 = __ldg(P.date_ex_off + di + 1);
      for (int x = x0; x < x1; ++x) {
        // underlying = const + sum_j w_j P(t, T_j; r), P = exp(alpha_j - B_j r); immediate value max(sign (U - K), 0)
        // (bond.py:115-163, swap.py:129-140, bermudan_option.py:60-70) - same arithmetic as irc_exercise_value
        const int t0 = __ldg(P.ex_term_off + x), t1 = __ldg(P.ex_term_off + x + 1), b = __ldg(P.ex_unit + x);
        double U[PP];
        MCRE_VP U[p] = __ldg(P.ex_const + x);
        for (int t = t0; t < t1; ++t) {
          const double alpha = __ldg(P.term_coef + 2 * t), B = __ldg(P.term_coef + 2 * t + 1), wgt = __ldg(P.term_w + t);
          double xa[PP], e[PP];
          MCRE_VP xa[p] = alpha - B * r[p];
          fm_exp_tv<PP>(xa, e);
          MCRE_VP U[p] = U[p] + e[p] * wgt;
        }
        const double K = __ldg(P.berm_strike + b), sg = __ldg(P.berm_sign + b);
        MCRE_VP { if (live[p]) ibuf[(size_t)x * n + lpath[p]] = fmax((U[p] - K) * sg, 0.0); }
      }
    }
  };
  for (int di = 0; di < P.n_pre_dates; ++di) eval_date(di);
#pragma unroll 1
  for (int is = 0; is < P.n_sub; ++is) {
    const double dt = __ldg(P.step_dt + is);
    const double sv0 = __ldg(P.step_vas + is * 2), sv1 = __ldg(P.step_vas + is * 2 + 1);
    double z0[PP], z1[PP];
    if (inject) {
      MCRE_VP {
        const double *zp = rng.z + ((size_t)is * rng.n_total + gpath[p]) * (CIR ? 2 : 1);
        z0[p] = zp[0];
        z1[p] = CIR ? zp[1] : 0.0;
      }
    } else if (CIR) {
      nsv.next2(z0, z1);
    } else {
      if ((is & 1) == 0) nsv.next2(z0, zb);
      else { MCRE_VP z0[p] = zb[p]; }
      MCRE_VP z1[p] = 0.0;
    }
    MCRE_VP logB[p] = fma(P.ext_num ? P.ext_rate : r[p], dt, logB[p]);
    if (SCHEME == MCRE_SCHEME_ANALYTICAL) {
      MCRE_VP r[p] = fma(sv1, z0[p], fma(r[p] - theta, sv0, theta));
    } else {
      const double adt = a * dt, ssq = sigma * sqrt(dt);
      const double k0 = ssq * l0, k1 = ssq * l1;
      MCRE_VP r[p] = fma(k0, z0[p], fma(sv0 - r[p], adt, r[p]));
      if (second) { MCRE_VP r[p] = fma(k1, z1[p], r[p]); }
    }
    const int di = __ldg(P.step_date + is);
    if (di >= 0) eval_date(di);
  }
}

// Pre-simulation pass B: backward FP32 suffix sums + Gram / right-hand-side moments.
// slot layout: [n_reg][5 + 3*NU] = sum u^0..u^4, then per unit sum u^0..u^2 * Y
// Each thread owns MOM_IT paths of the block's chunk (stride blockDim) and keeps their running
// FP32 tails in registers; per regression date it sums its own paths first and the block
// reduces once - 16x fewer shuffle / barrier rounds than reducing every 256 paths, and the
// loads of one date stay coalesced.  HBM-bound: 20 B per (path, date).
// The loads of date k-1 are issued before the block reduction of date k (software pipeline): the first
// version waited for memory and for the barrier in turn with 8 warps per SM (175 registers, one block per SM,
// 1.1 TB/s; profiles/r01_other_kernels_ncu_summary.md).
// (paths per thread: 8 with one regression unit; fewer with more units, whose per-path window sums and tails would
// otherwise spill - the two-unit build ran at 2.1 TB/s with 120 bytes of spills, profiles/r02_other_kernels.md)
template <int NU>
__global__ void __launch_bounds__(256, 2) irc_presim_moments_kernel(IrcDev P, ShardDev sh, const double *__restrict__ xbuf,
                                                                    const double *__restrict__ nbuf,
                                                                    const float *__restrict__ wbuf,
                                                                    double *__restrict__ partial) {
  constexpr int NV = 5 + 3 * NU;
  constexpr int MOM_IT = NU == 1 ? 8 : (NU == 2 ? 4 : 2);
  extern __shared__ double smem[];
  const int nw = blockDim.x >> 5;
  const int n_slots = P.n_reg * NV;
  double *acc = smem;
  double *stage = smem + n_slots;
  const long long n = sh.n_paths;
  const long long n_chunks = (n + sh.chunk - 1) / sh.chunk;
  for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) acc[i] = 0.0;
    __syncthreads();
    int parity = 0;
    for (int base = 0; base < sh.chunk; base += MOM_IT * (int)blockDim.x) {
      float S[MOM_IT][NU];
      long long path[MOM_IT];
      bool live[MOM_IT];
#pragma unroll
      for (int i = 0; i < MOM_IT; ++i) {
        const int in_chunk = base + i * (int)blockDim.x + (int)threadIdx.x;
        const long long lp = chunk * sh.chunk + in_chunk;
        live[i] = in_chunk < sh.chunk && lp < n;
        path[i] = live[i] ? lp : 0;
#pragma unroll
        for (int u = 0; u < NU; ++u) S[i][u] = 0.0f;
      }
      double xc[MOM_IT], nc[MOM_IT], xn[MOM_IT], nn[MOM_IT];
      float wc[MOM_IT][NU], wn[MOM_IT][NU];
      auto load = [&](int k, double (&x)[MOM_IT], double (&num)[MOM_IT], float (&w)[MOM_IT][NU]) {
#pragma unroll
        for (int i = 0; i < MOM_IT; ++i) {
          x[i] = __ldg(xbuf + (size_t)k * n + path[i]);
          num[i] = __ldg(nbuf + (size_t)k * n + path[i]);
#pragma unroll
          for (int u = 0; u < NU; ++u)
            w[i][u] = u < P.n_units ? __ldg(wbuf + ((size_t)u * P.n_reg + k) * n + path[i]) : 0.0f;
        }
      };
      load(P.n_reg - 1, xc, nc, wc);
      for (int k = P.n_reg - 1; k >= 0; --k) {
        if (k > 0) load(k - 1, xn, nn, wn);
        const double bs = __ldg(P.reg_basis + k * 2), bc = __ldg(P.reg_basis + k * 2 + 1);
        double vals[NV];
#pragma unroll
        for (int j = 0; j < NV; ++j) vals[j] = 0.0;
#pragma unroll
        for (int i = 0; i < MOM_IT; ++i) {
          const double keep = live[i] ? 1.0 : 0.0;
          const double uu = (xc[i] - bs) * bc;
          const double u1 = keep * uu, u2 = u1 * uu;
          vals[0] += keep; vals[1] += u1; vals[2] += u2; vals[3] += u2 * uu; vals[4] += u2 * uu * uu;
#pragma unroll
          for (int u = 0; u < NU; ++u) {
            // total = step_value + tail_value, both float32 (controller.py:349)
            if (u < P.n_units) S[i][u] = wc[i][u] + S[i][u];
            const double Y = keep * (nc[i] * (double)S[i][u]);  // numeraire.unsqueeze(1) * total_cfs (controller.py:368)
            vals[5 + 3 * u] += Y; vals[6 + 3 * u] += Y * uu; vals[7 + 3 * u] += Y * uu * uu;
          }
        }
        block_accumulate<NV>(vals, acc, k * NV, stage, NV, parity);
#pragma unroll
        for (int i = 0; i < MOM_IT; ++i) {
          xc[i] = xn[i]; nc[i] = nn[i];
#pragma unroll
          for (int u = 0; u < NU; ++u) wc[i][u] = wn[i][u];
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) partial[(size_t)chunk * n_slots + i] = acc[i];
    __syncthreads();
  }
}

}  // namespace mcre

// =====================================================================================
// Host side of the C ABI
// =====================================================================================
using namespace mcre;

extern "C" int mcre_irc_create(const mcre_irc_desc *c, mcre_irc_plan **out) {
  if (!c || !out) return fail(-1, "null argument%s", "");
  if (c->nt != 0 && c->nt != 4 && c->nt != 8) return fail(-1, "irc: nt must be 0, 4 or 8%s", "");
  if (c->n_sets < 0 || c->n_sets > MCRE_IRC_MAX_SETS) return fail(-1, "irc: n_sets out of range%s", "");
  if (c->n_units < 0 || c->n_units > MCRE_IRC_MAX_UNITS) return fail(-1, "irc: n_units out of range%s", "");
  if (c->n_berm < 0 || c->n_berm > MCRE_IRC_MAX_BERM) return fail(-1, "irc: n_berm out of range%s", "");
  if (c->scheme != MCRE_SCHEME_EULER && c->scheme != MCRE_SCHEME_ANALYTICAL)
    return fail(-1, "irc: scheme must be EULER or ANALYTICAL%s", "");
  if (c->scheme == MCRE_SCHEME_ANALYTICAL && c->has_cir)
    return fail(-1, "irc: ANALYTICAL is not defined for the Vasicek+CIR++ hybrid (model_config.py:216-221)%s", "");
  mcre_irc_plan *p = new mcre_irc_plan();
  ArenaScope arena_scope(&p->arena);
  const int w = 1 + c->nt;
  const int n_float = c->date_float_off ? c->date_float_off[c->n_dates] : 0;
  int rc = 0;
#define UP(field, host, count) if (!rc) rc = p->field.upload(host, (size_t)(count))
  UP(vas, c->vas, 4 * w); UP(cir, c->cir, c->has_cir ? 4 * w : 0); UP(cir_init, c->cir_init, c->has_cir ? w : 0);
  UP(chol, c->chol, 4 * w);
  UP(step_dt, c->step_dt, c->n_sub); UP(step_date, c->step_date, c->n_sub);
  UP(step_vas, c->step_vas, (size_t)c->n_sub * 2 * w); UP(step_cir, c->step_cir, c->has_cir ? (size_t)c->n_sub * 2 * w : 0);
  UP(date_flags, c->date_flags, c->n_dates); UP(date_expo, c->date_expo, c->n_dates);
  UP(date_metric, c->date_metric, c->n_dates); UP(date_reg, c->date_reg, c->n_dates);
  UP(date_float_off, c->date_float_off, c->n_dates + 1);
  UP(float_coef, c->float_coef, (size_t)n_float * 2 * w); UP(float_inv_tau, c->float_inv_tau, n_float);
  UP(set_fix, c->set_fix, (size_t)c->n_sets * c->n_dates); UP(set_float, c->set_float, (size_t)c->n_sets * n_float);
  UP(set_threshold, c->set_threshold, c->n_sets); UP(set_flags, c->set_flags, c->n_sets);
  UP(set_lag, c->set_lag, (size_t)c->n_sets * c->n_metric);
  p->expo_coef_count = (size_t)c->n_expo * c->n_sets * 3 * w;
  UP(expo_coef, c->expo_coef, p->expo_coef_count); UP(expo_basis, c->expo_basis, (size_t)c->n_expo * 2);
  UP(cva_coef, c->cva_coef, (size_t)c->n_metric * 2 * w);
  UP(unit_fix, c->unit_fix, (size_t)c->n_units * c->n_dates); UP(unit_float, c->unit_float, (size_t)c->n_units * n_float);
  UP(reg_basis, c->reg_basis, (size_t)c->n_reg * 2);
  const int n_berm = c->n_berm;
  const int n_ex = (n_berm > 0 && c->date_ex_off) ? c->date_ex_off[c->n_dates] : 0;
  const int n_term = n_ex > 0 ? c->ex_term_off[n_ex] : 0;
  if (n_berm > 0) {
    UP(berm_set, c->berm_set, n_berm); UP(berm_strike, c->berm_strike, n_berm); UP(berm_sign, c->berm_sign, n_berm);
    UP(date_ex_off, c->date_ex_off, c->n_dates + 1); UP(ex_unit, c->ex_unit, n_ex); UP(ex_last, c->ex_last, n_ex);
    UP(ex_term_off, c->ex_term_off, n_ex + 1); UP(ex_const, c->ex_const, n_ex);
    UP(term_coef, c->term_coef, (size_t)n_term * 2 * w); UP(term_w, c->term_w, n_term);
    UP(ex_basis, c->ex_basis, (size_t)n_ex * 2);
    p->ex_coef_count = (size_t)n_ex * 3 * w;
    p->berm_expo_count = (size_t)c->n_expo * n_berm * 3 * w;
    std::vector<double> zeros(std::max(p->ex_coef_count, p->berm_expo_count) + 1, 0.0);
    UP(ex_coef, zeros.data(), p->ex_coef_count); UP(berm_expo_coef, zeros.data(), p->berm_expo_count);
  }
  {
    // packed per-step and per-date records of the main kernel (layout: STEP_HDR / DATE_HDR above)
    const int SR = STEP_HDR + 4 * w, DR = (DATE_HDR + 2 * w + 3 * w * c->n_sets + 1) & ~1;
    std::vector<double> srec((size_t)c->n_sub * SR + 2, 0.0);
    for (int s = 0; s < c->n_sub; ++s) {
      double *r = srec.data() + (size_t)s * SR;
      r[0] = c->step_dt[s]; r[1] = sqrt(c->step_dt[s]); r[2] = pack2(c->step_date[s], 0);
      for (int k = 0; k < 2 * w; ++k) r[STEP_HDR + k] = c->step_vas[(size_t)s * 2 * w + k];
      if (c->has_cir) for (int k = 0; k < 2 * w; ++k) r[STEP_HDR + 2 * w + k] = c->step_cir[(size_t)s * 2 * w + k];
    }
    p->h_date_rec.assign((size_t)c->n_dates * DR + 2, 0.0);
    p->h_date_expo.assign(c->date_expo, c->date_expo + c->n_dates);
    p->date_stride = DR;
    for (int di = 0; di < c->n_dates; ++di) {
      double *r = p->h_date_rec.data() + (size_t)di * DR;
      const int e = c->date_expo[di], m = c->date_metric[di];
      r[0] = pack2(c->date_flags[di], e + 1);
      r[1] = pack2(m + 1, c->date_float_off[di]);
      r[2] = pack2(c->date_float_off[di + 1] - c->date_float_off[di], 0);
      if (e >= 0) { r[4] = c->expo_basis[e * 2]; r[5] = c->expo_basis[e * 2 + 1]; }
      if (m >= 0 && c->cva_coef) for (int k = 0; k < 2 * w; ++k) r[DATE_HDR + k] = c->cva_coef[(size_t)m * 2 * w + k];
      if (e >= 0 && c->expo_coef)
        for (int k = 0; k < 3 * w * c->n_sets; ++k) r[DATE_HDR + 2 * w + k] = c->expo_coef[(size_t)e * 3 * w * c->n_sets + k];
    }
    UP(step_rec, srec.data(), srec.size());
    UP(date_rec, p->h_date_rec.data(), p->h_date_rec.size());
    for (int k = 0; k < c->n_sets; ++k) p->any_collateral = p->any_collateral || (c->set_flags[k] & 1);
    // "CVA only" kernel (irc_cva.cu): one set, CVA the only accumulator, no threshold / collateral, stochastic
    // intensity started above zero; everything else runs the general kernel
    p->cva_only = !c->ext_numeraire && c->has_cir && c->nt == 0 && c->n_sets == 1 && c->acc_flags == MCRE_ACC_CVA && n_berm == 0 &&
                  c->set_threshold[0] == 0.0 && (c->set_flags[0] & 1) == 0 && (c->set_flags[0] & 2) != 0 &&
                  !c->cir_deterministic && c->cir_init[0] > 0.0 && c->scheme == MCRE_SCHEME_EULER;
    if (p->cva_only) {
      CvaHost &h = p->cva;
      h.n_sub = c->n_sub; h.n_pre_dates = c->n_pre_dates; h.n_metric = c->n_metric;
      h.vas_noise = c->vas_noise; h.cir_noise = c->cir_noise;
      for (int k = 0; k < 4; ++k) { h.vas[k] = c->vas[k]; h.chol[k] = c->chol[k]; }
      for (int k = 0; k < 3; ++k) h.cir[k] = c->cir[k];
      h.y0 = c->cir_init[0]; h.lgd = c->lgd;
      h.step_dt.assign(c->step_dt, c->step_dt + c->n_sub);
      h.step_date.assign(c->step_date, c->step_date + c->n_sub);
      h.step_theta.resize(c->n_sub); h.step_psi.resize(c->n_sub);
      for (int s = 0; s < c->n_sub; ++s) { h.step_theta[s] = c->step_vas[(size_t)s * 2]; h.step_psi[s] = c->step_cir[(size_t)s * 2]; }
      h.date_flags.assign(c->date_flags, c->date_flags + c->n_dates);
      h.date_metric.assign(c->date_metric, c->date_metric + c->n_dates);
      irc_cva_fill_static(p);
      std::vector<int> zsync(4, 0);
      UP(cva_rec, p->cva_rec_host.data(), p->cva_rec_host.size());
      UP(cva_sync, zsync.data(), zsync.size());
    }
  }
#undef UP
  if (!rc) rc = p->arena.commit();
  if (rc) { mcre_irc_destroy(p); return rc; }
  IrcDev &d = p->d;
  d.nt = c->nt; d.scheme = c->scheme; d.has_cir = c->has_cir; d.cir_det = c->cir_deterministic;
  d.vas_noise = c->vas_noise; d.cir_noise = c->cir_noise;
  d.ext_num = c->ext_numeraire; d.ext_rate = c->ext_rate; d.ext_slot = c->ext_numeraire ? c->ext_slot : -1; d.pv_spill = nullptr;
  d.vas = p->vas.p; d.cir = p->cir.p; d.cir_init = p->cir_init.p; d.chol = p->chol.p;
  d.n_sub = c->n_sub; d.n_dates = c->n_dates; d.n_pre_dates = c->n_pre_dates;
  d.step_dt = p->step_dt.p; d.step_date = p->step_date.p; d.step_vas = p->step_vas.p; d.step_cir = p->step_cir.p;
  d.date_flags = p->date_flags.p; d.date_expo = p->date_expo.p; d.date_metric = p->date_metric.p;
  d.date_reg = p->date_reg.p; d.date_float_off = p->date_float_off.p;
  d.float_coef = p->float_coef.p; d.float_inv_tau = p->float_inv_tau.p; d.n_float = n_float;
  d.n_sets = c->n_sets; d.n_expo = c->n_expo; d.n_metric = c->n_metric; d.acc_flags = c->acc_flags;
  d.set_fix = p->set_fix.p; d.set_float = p->set_float.p; d.set_threshold = p->set_threshold.p;
  d.set_flags = p->set_flags.p; d.set_lag = p->set_lag.p;
  {
    int max_lag = 0;
    for (size_t k = 0; k < (size_t)c->n_sets * c->n_metric; ++k) max_lag = std::max(max_lag, (int)c->set_lag[k]);
    // the general template keeps MCRE_IRC_MAX_LAG exposures per path in registers; the value-only kernel a ring in shared memory
    const bool general = c->nt != 0 || n_berm != 0;
    if (max_lag >= (general ? MCRE_IRC_MAX_LAG : 64)) { mcre_irc_destroy(p); return fail(-3, "irc: MPoR look-back of %s%lld exposure dates is too long for this plan", "", max_lag); }
    p->max_lag = max_lag;
    d.ring_depth = 2;
    while (d.ring_depth <= max_lag) d.ring_depth *= 2;
    if (general && d.ring_depth < MCRE_IRC_MAX_LAG) d.ring_depth = MCRE_IRC_MAX_LAG;
  }
  d.expo_coef = p->expo_coef.p; d.expo_basis = p->expo_basis.p; d.cva_coef = p->cva_coef.p; d.lgd = c->lgd;
  d.n_units = c->n_units; d.n_reg = c->n_reg;
  d.unit_fix = p->unit_fix.p; d.unit_float = p->unit_float.p; d.reg_basis = p->reg_basis.p;
  d.step_rec = p->step_rec.p; d.date_rec = p->date_rec.p;
  d.n_berm = n_berm; d.n_ex = n_ex;
  d.berm_set = p->berm_set.p; d.berm_strike = p->berm_strike.p; d.berm_sign = p->berm_sign.p;
  d.date_ex_off = p->date_ex_off.p; d.ex_unit = p->ex_unit.p; d.ex_term_off = p->ex_term_off.p; d.ex_last = p->ex_last.p;
  d.ex_const = p->ex_const.p; d.term_coef = p->term_coef.p; d.term_w = p->term_w.p; d.ex_basis = p->ex_basis.p;
  d.ex_coef = p->ex_coef.p; d.berm_expo_coef = p->berm_expo_coef.p;
  d.path_list = nullptr; d.tan_spill = nullptr;
  p->cva_rec_dev = p->cva_rec.p; p->cva_sync_dev = (unsigned *)p->cva_sync.p;
  *out = p;
  return 0;
}

extern "C" void mcre_irc_destroy(mcre_irc_plan *p) {
  if (!p) return;
  p->vas.release(); p->cir.release(); p->cir_init.release(); p->chol.release(); p->step_dt.release();
  p->step_vas.release(); p->step_cir.release(); p->float_coef.release(); p->float_inv_tau.release();
  p->set_fix.release(); p->set_float.release(); p->set_threshold.release(); p->expo_coef.release();
  p->expo_basis.release(); p->cva_coef.release(); p->unit_fix.release(); p->unit_float.release();
  p->reg_basis.release(); p->step_date.release(); p->date_flags.release(); p->date_expo.release();
  p->date_metric.release(); p->date_reg.release(); p->date_float_off.release(); p->set_flags.release();
  p->set_lag.release(); p->step_rec.release(); p->date_rec.release();
  p->berm_set.release(); p->date_ex_off.release(); p->ex_unit.release(); p->ex_last.release(); p->ex_term_off.release();
  p->berm_strike.release(); p->berm_sign.release(); p->ex_const.release(); p->term_coef.release(); p->term_w.release();
  p->ex_basis.release(); p->ex_coef.release(); p->berm_expo_coef.release();
  p->cva_rec.release(); p->cva_sync.release();
  p->arena.release();
  delete p;
}

static int nu_template(int n_units) { return n_units <= 1 ? 1 : (n_units <= 2 ? 2 : 4); }

extern "C" int64_t mcre_irc_main_slots(const mcre_irc_plan *p) {
  return (int64_t)(p->d.n_metric + 1) * ns_template(p->d.n_sets) * (4 + 2 * p->d.nt);
}
extern "C" int64_t mcre_irc_presim_slots(const mcre_irc_plan *p) {
  return (int64_t)p->d.n_reg * (5 + 3 * nu_template(p->d.n_units));
}
extern "C" int64_t mcre_irc_presim_scratch_bytes(const mcre_irc_plan *p, int64_t n_paths) {
  // value buffers, then (plans with tangents) dx, dN, dW: see irc_tan.cu
  const int64_t tangents = (int64_t)p->d.n_reg * p->d.nt * n_paths * 8 * (2 + (int64_t)p->d.n_units);
  return (int64_t)p->d.n_reg * n_paths * (16 + 4 * (int64_t)p->d.n_units) + tangents + 256;
}
extern "C" int64_t mcre_irc_partial_bytes(const mcre_irc_plan *p, int64_t n_paths, int32_t chunk, int presim) {
  int64_t n_chunks = (n_paths + chunk - 1) / chunk;
  int64_t slots = presim ? mcre_irc_presim_slots(p) : mcre_irc_main_slots(p);
  if (presim && p->d.nt > 0) slots = std::max<int64_t>(slots, mcre_irc_presim_tangent_slots(p));
  int64_t doubles = n_chunks * slots;
  if (!presim && p->cva_only) doubles = std::max<int64_t>(doubles, irc_cva_units(n_paths) * 4);   // per-pass partials
  return doubles * 8;
}

extern "C" int mcre_irc_set_coefficients(mcre_irc_plan *p, const double *coef, void *stream) {
  if (!p || (!coef && p->expo_coef_count)) return fail(-1, "null argument%s", "");
  if (p->expo_coef_count == 0) return 0;
  MCRE_CUDA(cudaMemcpyAsync(p->d.expo_coef, coef, p->expo_coef_count * sizeof(double), cudaMemcpyHostToDevice,
                            (cudaStream_t)stream));
  MCRE_H2D(p->expo_coef_count * sizeof(double) + p->h_date_rec.size() * sizeof(double));
  const int w = 1 + p->d.nt, per_date = 3 * w * p->d.n_sets, DR = p->date_stride;
  for (int di = 0; di < p->d.n_dates; ++di) {
    const int e = p->h_date_expo[di];
    if (e < 0) continue;
    double *r = p->h_date_rec.data() + (size_t)di * DR + DATE_HDR + 2 * w;
    for (int k = 0; k < per_date; ++k) r[k] = coef[(size_t)e * per_date + k];
    if (p->cva_only) {
      // the CVA-only kernel mode evaluates the polynomial in the raw basis [1, r, r^2]:
      // c(u) with u = (r - shift) * scale  ->  c'(r)
      const double sh = p->h_date_rec[(size_t)di * DR + 4], sc = p->h_date_rec[(size_t)di * DR + 5];
      irc_raw_basis(r[0], r[1], r[2], sh, sc, r);
    }
  }
  MCRE_CUDA(cudaMemcpyAsync((void *)p->d.date_rec, p->h_date_rec.data(), p->h_date_rec.size() * sizeof(double),
                            cudaMemcpyHostToDevice, (cudaStream_t)stream));
  if (p->cva_only) {
    const int rc = irc_cva_apply_coefficients(p, (cudaStream_t)stream);
    if (rc) return rc;
  }
  MCRE_CUDA(cudaStreamSynchronize((cudaStream_t)stream));  // host staging buffers may be reused by the caller
  return 0;
}

extern "C" int mcre_irc_set_exercise_coefficients(mcre_irc_plan *p, const double *ex_coef, const double *expo_coef,
                                                  void *stream) {
  if (!p) return fail(-1, "null argument%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  if (p->ex_coef_count && ex_coef)
    MCRE_CUDA(cudaMemcpyAsync(p->d.ex_coef, ex_coef, p->ex_coef_count * sizeof(double), cudaMemcpyHostToDevice, st));
  MCRE_H2D((p->ex_coef_count && ex_coef ? p->ex_coef_count : 0) * sizeof(double) +
           (p->berm_expo_count && expo_coef ? p->berm_expo_count : 0) * sizeof(double));
  if (p->berm_expo_count && expo_coef)
    MCRE_CUDA(cudaMemcpyAsync(p->d.berm_expo_coef, expo_coef, p->berm_expo_count * sizeof(double),
                              cudaMemcpyHostToDevice, st));
  MCRE_CUDA(cudaStreamSynchronize(st));  // host staging buffers may be reused by the caller
  return 0;
}

extern "C" int mcre_irc_set_path_replay(mcre_irc_plan *p, const int64_t *d_paths, double *d_tan_spill) {
  if (!p) return fail(-1, "null argument%s", "");
  if ((d_paths == nullptr) != (d_tan_spill == nullptr)) return fail(-1, "path replay needs both the path list and the output%s", "");
  if (d_paths && p->d.nt == 0) return fail(-1, "path replay writes tangents: the plan has none%s", "");
  p->d.path_list = (const long long *)d_paths;
  p->d.tan_spill = d_tan_spill;
  return 0;
}

extern "C" int64_t mcre_irc_lsm_scratch_bytes(const mcre_irc_plan *p, int64_t n_paths) {
  // x, N, imm and (plans with tangents) dx, dN, dimm: see irc_tan.cu
  return ((int64_t)2 * p->d.n_reg + p->d.n_ex) * n_paths * 8 * (1 + p->d.nt) + 256;
}

// defined in irc_tan.cu
int irc_lsm_forward_tangent_pass(mcre_irc_plan *p, const mcre::RngDev &r, const mcre::ShardDev &sh, void *d_scratch,
                                 cudaStream_t st);

extern "C" int mcre_irc_lsm_forward(mcre_irc_plan *p, const mcre_rng *rng, const mcre_shard *shard, void *d_scratch,
                                    void *stream) {
  if (!p || !rng || !d_scratch) return fail(-1, "null argument%s", "");
  int rc = check_shard(shard);
  if (rc) return rc;
  if (p->d.n_berm < 1) return fail(-1, "irc lsm: plan has no exercise unit%s", "");
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  const IrcDev &d = p->d;
  if (shard->n_paths == 0) return 0;
  RngDev r = make_rng(rng);
  ShardDev sh{shard->path_begin, shard->n_paths, shard->chunk_paths};
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = sh.n_paths;
  double *xbuf = (double *)d_scratch;
  double *nbuf = xbuf + (size_t)d.n_reg * n;
  double *ibuf = nbuf + (size_t)d.n_reg * n;
  if (d.nt != 0) return irc_lsm_forward_tangent_pass(p, r, sh, d_scratch, st);
  const int threads = 128;
  const unsigned blocks = (unsigned)((n + threads * PRE_PP - 1) / (threads * PRE_PP));
  if (d.has_cir) irc_lsm_forward_kernel<true, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, ibuf);
  else if (d.scheme == MCRE_SCHEME_ANALYTICAL)
    irc_lsm_forward_kernel<false, MCRE_SCHEME_ANALYTICAL><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, ibuf);
  else irc_lsm_forward_kernel<false, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, ibuf);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_irc_set_pv_spill(mcre_irc_plan *p, double *d_pv) {
  if (!p) return fail(-1, "null argument%s", "");
  if (p->cva_only) return fail(-3, "pv spill: not available on the CVA-only plan%s", "");
  if (p->d.n_berm != 0) return fail(-3, "pv spill: plans of linear products%s", "");
  p->d.pv_spill = d_pv;
  return 0;
}

extern "C" int mcre_irc_mainsim(mcre_irc_plan *p, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                                double *d_acc, double *d_shift, double *d_spill, void *stream) {
  if (!p || !rng || !d_partial || !d_acc || !d_shift) return fail(-1, "null argument%s", "");
  int rc = check_shard(shard);
  if (rc) return rc;
  if ((p->d.acc_flags & MCRE_ACC_SPILL) && !d_spill && !p->d.tan_spill) return fail(-1, "spill requested but d_spill is null%s", "");
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  RngDev r = make_rng(rng);
  ShardDev sh{shard->path_begin, shard->n_paths, shard->chunk_paths};
  cudaStream_t st = (cudaStream_t)stream;
  if (p->cva_only) {
    // per-pass partials of the tail row only: [pass][pv, pv^2, cva, cva^2]; the date rows of the accumulator stay 0
    const int64_t slots = mcre_irc_main_slots(p);
    rc = irc_cva_launch(p, r, sh, d_partial, d_shift, st);
    if (rc) return rc;
    MCRE_CUDA(cudaMemsetAsync(d_acc, 0, (size_t)slots * sizeof(double), st));
    return mcre_tree_reduce(d_partial, irc_cva_units(sh.n_paths), 4, d_acc + (slots - 4), stream);
  }
  // value-only plans without exercise units: the lean kernel of irc_value.cuh (MCRE_IRC_GENERIC=1: the general template)
  static const bool force_generic = getenv("MCRE_IRC_GENERIC") && getenv("MCRE_IRC_GENERIC")[0] == '1';
  if (p->d.nt == 0 && p->d.n_berm == 0 && !p->d.path_list && !force_generic) {
    const int ns = ns_template(p->d.n_sets);
    rc = ns == 1 ? launch_value<1>(p, r, sh, d_partial, d_spill, d_shift, st)
       : ns == 2 ? launch_value<2>(p, r, sh, d_partial, d_spill, d_shift, st)
                 : launch_value<4>(p, r, sh, d_partial, d_spill, d_shift, st);
    if (rc) return rc;
    const long long n_chunks_v = (sh.n_paths + sh.chunk - 1) / sh.chunk;
    return mcre_tree_reduce(d_partial, n_chunks_v, mcre_irc_main_slots(p), d_acc, stream);
  }
  if (p->max_lag >= MCRE_IRC_MAX_LAG) return fail(-3, "irc: MPoR look-back too long for the general kernel%s", "");
  rc = p->d.n_berm > 0 ? irc_dispatch_main_berm(p, r, sh, d_partial, d_spill, d_shift, st)
                       : irc_dispatch_main<false>(p, r, sh, d_partial, d_spill, d_shift, st);
  if (rc) return rc;
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  return mcre_tree_reduce(d_partial, n_chunks, mcre_irc_main_slots(p), d_acc, stream);
}

// defined in irc_tan.cu
int irc_presim_tangent_fit(const mcre_irc_plan *p);
int irc_presim_tangent_pass(mcre_irc_plan *p, const mcre::RngDev &r, const mcre::ShardDev &sh, void *d_scratch,
                            double *d_partial, double *d_tmoments, cudaStream_t st);

template <int NU>
static int irc_presim_moments_launch(const IrcDev &d, const ShardDev &sh, size_t smem, const double *xbuf,
                                     const double *nbuf, const float *wbuf, double *d_partial, cudaStream_t st) {
  const int threads = 256;
  auto k = irc_presim_moments_kernel<NU>;
  int per_sm = 1;
  MCRE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem));
  if (per_sm < 1) return fail(-3, "irc presim kernel does not fit: too many regression dates%s", "");
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  long long grid = (long long)sm_count() * per_sm;
  if (grid > n_chunks) grid = n_chunks;
  k<<<(unsigned)grid, threads, smem, st>>>(d, sh, xbuf, nbuf, wbuf, d_partial);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_irc_presim(mcre_irc_plan *p, const mcre_rng *rng, const mcre_shard *shard, void *d_scratch,
                               double *d_partial, double *d_moments, double *d_tmoments, void *stream) {
  if (!p || !rng || !d_scratch || !d_partial || !d_moments) return fail(-1, "null argument%s", "");
  int rc = check_shard(shard);
  if (rc) return rc;
  if (p->d.nt != 0 && !d_tmoments) return fail(-1, "irc presim: the plan carries tangents but d_tmoments is null%s", "");
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  const IrcDev &d = p->d;
  if (d.n_reg == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // the moment kernels keep every regression date's sums in shared memory: a plan with too many dates is refused here,
  // before anything is launched
  const int nu = nu_template(d.n_units);
  const int nv = 5 + 3 * nu, nw = 256 / 32;
  const size_t smem = ((size_t)d.n_reg * nv + 2 * nw * nv) * sizeof(double);
  const char *too_many = "irc presim kernel does not fit: too many regression dates (%s%lld bytes of shared memory)";
  if (nu == 1) MCRE_SMEM(irc_presim_moments_kernel<1>, smem, too_many);
  else if (nu == 2) MCRE_SMEM(irc_presim_moments_kernel<2>, smem, too_many);
  else MCRE_SMEM(irc_presim_moments_kernel<4>, smem, too_many);
  const bool tangents = d.nt != 0 && d.n_units > 0;
  if (tangents) {
    rc = irc_presim_tangent_fit(p);
    if (rc) return rc;
  }
  if (shard->n_paths == 0) {
    // a rank without pre-simulation paths contributes zero moments
    MCRE_CUDA(cudaMemsetAsync(d_moments, 0, (size_t)mcre_irc_presim_slots(p) * sizeof(double), st));
    if (tangents) MCRE_CUDA(cudaMemsetAsync(d_tmoments, 0, (size_t)mcre_irc_presim_tangent_slots(p) * sizeof(double), st));
    return 0;
  }
  RngDev r = make_rng(rng);
  ShardDev sh{shard->path_begin, shard->n_paths, shard->chunk_paths};
  const long long n = sh.n_paths;
  double *xbuf = (double *)d_scratch;
  double *nbuf = xbuf + (size_t)d.n_reg * n;
  float *wbuf = (float *)(nbuf + (size_t)d.n_reg * n);
  if (tangents) {
    // forward pass with tangents (fills the value buffers too) + tangent moments
    rc = irc_presim_tangent_pass(p, r, sh, d_scratch, d_partial, d_tmoments, st);
    if (rc) return rc;
  } else {
    const unsigned fblocks = (unsigned)((n + 128 * PRE_PP - 1) / (128 * PRE_PP));
    const int nuf = nu_template(d.n_units);
#define LAUNCHF(NUV)                                                                                          \
  do {                                                                                                        \
    if (d.has_cir) irc_presim_forward_kernel<true, MCRE_SCHEME_EULER, NUV><<<fblocks, 128, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf); \
    else if (d.scheme == MCRE_SCHEME_ANALYTICAL)                                                              \
      irc_presim_forward_kernel<false, MCRE_SCHEME_ANALYTICAL, NUV><<<fblocks, 128, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf); \
    else irc_presim_forward_kernel<false, MCRE_SCHEME_EULER, NUV><<<fblocks, 128, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf); \
  } while (0)
    if (nuf == 1) LAUNCHF(1); else if (nuf == 2) LAUNCHF(2); else LAUNCHF(4);
#undef LAUNCHF
    MCRE_LAUNCHED();
  }
  rc = nu == 1 ? irc_presim_moments_launch<1>(d, sh, smem, xbuf, nbuf, wbuf, d_partial, st)
     : nu == 2 ? irc_presim_moments_launch<2>(d, sh, smem, xbuf, nbuf, wbuf, d_partial, st)
               : irc_presim_moments_launch<4>(d, sh, smem, xbuf, nbuf, wbuf, d_partial, st);
  if (rc) return rc;
  const long long n_chunks = (n + sh.chunk - 1) / sh.chunk;
  return mcre_tree_reduce(d_partial, n_chunks, mcre_irc_presim_slots(p), d_moments, stream);
}
