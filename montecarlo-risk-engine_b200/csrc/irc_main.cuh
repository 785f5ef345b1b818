// Interest-rate / credit family: device plan tables + the fused main-simulation kernel.
// Shared by irc.cu (plain books) and irc_berm.cu (books with Bermudan exercise units) so
// the two sets of template instantiations compile in parallel.
#pragma once
#define MCRE_FAST_MATH 2
#include "common.cuh"
#include "philox.cuh"
#include "dual.cuh"
#include "reduce.cuh"
#include "launch.cuh"

namespace mcre {

struct IrcDev {
  int nt, scheme, has_cir, cir_det, vas_noise, cir_noise;
  const double *vas, *cir, *cir_init, *chol;
  int n_sub, n_dates, n_pre_dates;
  const double *step_dt; const int *step_date; const double *step_vas, *step_cir;
  const int *date_flags, *date_expo, *date_metric, *date_reg, *date_float_off;
  const double *float_coef, *float_inv_tau;
  int n_float;
  int n_sets, n_expo, n_metric, acc_flags;
  const double *set_fix, *set_float, *set_threshold; const int *set_flags, *set_lag;
  double *expo_coef;  // mutable: uploaded after the regression solve
  const double *expo_basis, *cva_coef;
  double lgd;
  int n_units, n_reg;
  const double *unit_fix, *unit_float; const double *reg_basis;
  const double *step_rec, *date_rec;  // packed records of the main kernel
  // Bermudan exercise units (bermudan_option.py:93-188): CSR of exercise records per date
  int n_berm, n_ex;
  const int *berm_set; const double *berm_strike, *berm_sign;
  const int *date_ex_off, *ex_unit, *ex_term_off, *ex_last;
  const double *ex_const, *term_coef, *term_w, *ex_basis;
  double *ex_coef;         // dual[n_ex][3] continuation coefficients (uploaded after the regression)
  double *berm_expo_coef;  // dual[n_expo][n_berm][3] alive-state exposure coefficients
  // path replay (mcre_irc_set_path_replay): simulate the listed global path ids instead of a contiguous
  // range and write the tangents of every unsecured exposure, [path][n_metric][n_sets][nt] - the gradient
  // of a PFE order statistic is the pathwise gradient of the selected path (pfe_metric.py:59-71 under autograd)
  const long long *path_list;
  double *tan_spill;
  // hybrid books (mcre/hybrid.py): the numeraire is another model's deterministic money-market account,
  // exp(ext_rate (t - t0)) (model_config.py:44-47, numeraire_model_idx), accumulated step by step like the path's own;
  // pv_spill [n_sets][n_paths]: per-path discounted cashflow totals (mcre_irc_set_pv_spill)
  int ring_depth;          // value-only kernel: slots of the exposure look-back ring (power of two > largest MPoR lag)
  int ext_num, ext_slot;   // ext_slot: tangent slot of the external rate (-1: none)
  double ext_rate;
  double *pv_spill;
};

// Underlying value of an exercise record at short rate r: const + sum_j w_j P(t, T_j; r) with
// P = exp(alpha_j - B_j r) (bond.py:115-163, swap.py:129-140), then the immediate exercise
// value max(sign (U - K), 0) (bermudan_option.py:60-70).
template <typename R>
__device__ __forceinline__ R irc_exercise_value(const IrcDev &P, int x, const R &r) {
  typedef RealTraits<R> T;
  const int t0 = __ldg(P.ex_term_off + x), t1 = __ldg(P.ex_term_off + x + 1), b = __ldg(P.ex_unit + x);
  R U = T::lift(__ldg(P.ex_const + x));
  for (int t = t0; t < t1; ++t) {
    const R alpha = T::load(P.term_coef, 2 * t), B = T::load(P.term_coef, 2 * t + 1);
    U = U + r_exp(alpha - B * r) * __ldg(P.term_w + t);
  }
  return r_max((U - __ldg(P.berm_strike + b)) * __ldg(P.berm_sign + b), 0.0);
}

// ---- per-path model state ---------------------------------------------------------
template <typename R>
struct IrcState {
  R r, logB, y, logBl;
};

template <typename R, bool CIR>
struct IrcParams {
  R r0, sigma, theta, a;        // Vasicek
  R kappa, ctheta, csigma, y0;  // CIR++
  R L10, L11;                   // Cholesky rows used by the second noise column
  R L00;
};

// One sub-step of the joint model (src/models/vasicek.py:52-112, cirpp.py:155-198,
// model_config.py:223-276).  z0/z1 are the independent draws; the correlated noise is
// z @ L^T with L the lower Cholesky factor (model.py:46-48).
// STEP_CIR = false: the credit factor is not advanced (the pre-simulations of rate products only read the short
// rate and the numeraire; its normal is still drawn so that the streams stay aligned).
template <typename R, bool CIR, int SCHEME, bool STEP_CIR = CIR>
__device__ __forceinline__ void irc_step(const IrcDev &P, const IrcParams<R, CIR> &mp, IrcState<R> &s, int is,
                                         double z0, double z1) {
  typedef RealTraits<R> T;
  const double dt = __ldg(P.step_dt + is);
  const double sq = sqrt(dt);
  R w0 = mp.L00 * z0;
  R w1 = T::zero();
  if (CIR) w1 = mp.L10 * z0 + mp.L11 * z1;
  const R wv = (CIR && P.vas_noise == 1) ? w1 : w0;
  // numeraire integral uses the pre-step rate (left Riemann sum)
  if (P.ext_num) {
    R e = T::lift(P.ext_rate);
    r_seed(e, P.ext_slot);
    s.logB = s.logB + e * dt;
  } else {
    s.logB = s.logB + s.r * dt;
  }
  if (SCHEME == MCRE_SCHEME_ANALYTICAL) {
    R decay = T::load(P.step_vas, is * 2 + 0), nstd = T::load(P.step_vas, is * 2 + 1);
    // exact OU transition; the 1x1 Cholesky factor of the step covariance is nstd (vasicek.py:52-86)
    s.r = mp.theta + (s.r - mp.theta) * decay + nstd * z0;
  } else {
    const R theta_t = T::load(P.step_vas, is * 2 + 0);  // mean level at t1 (constant for Vasicek)
    s.r = s.r + mp.a * (theta_t - s.r) * dt + mp.sigma * sq * wv;
  }
  if (CIR && STEP_CIR) {
    const R wc = (P.cir_noise == 1) ? w1 : w0;
    if (P.cir_det) {
      R lam1 = T::load(P.step_cir, is * 2 + 0), lam2 = T::load(P.step_cir, is * 2 + 1);
      s.logBl = s.logBl + lam1 * dt;
      s.y = lam2;
    } else {
      R psi = T::load(P.step_cir, is * 2 + 0);
      R ypos = r_relu(s.y);
      R yn = s.y + mp.kappa * (mp.ctheta - s.y) * dt + mp.csigma * r_sqrt(ypos) * sq * wc;
      s.logBl = s.logBl + (s.y + psi) * dt;
      s.y = r_max(yn, 1e-12);
    }
  }
}

template <typename R, bool CIR>
__device__ __forceinline__ void irc_load_params(const IrcDev &P, IrcParams<R, CIR> &mp) {
  typedef RealTraits<R> T;
  mp.r0 = T::load(P.vas, 0); mp.sigma = T::load(P.vas, 1); mp.theta = T::load(P.vas, 2); mp.a = T::load(P.vas, 3);
  mp.L00 = T::load(P.chol, 0);
  if (CIR) {
    mp.kappa = T::load(P.cir, 0); mp.ctheta = T::load(P.cir, 1); mp.csigma = T::load(P.cir, 2);
    mp.y0 = T::load(P.cir_init, 0);
    mp.L10 = T::load(P.chol, 2); mp.L11 = T::load(P.chol, 3);
  } else {
    mp.kappa = mp.ctheta = mp.csigma = mp.y0 = mp.L10 = mp.L11 = T::zero();
  }
}

template <typename R, bool CIR>
__device__ __forceinline__ void irc_draw(const RngDev &rng, NormalStream &ns, int is, long long lpath,
                                         long long gpath, double &z0, double &z1) {
  if (rng.mode == MCRE_RNG_INJECT) {
    const int d = CIR ? 2 : 1;
    const double *p = rng.z + ((size_t)is * rng.n_total + gpath) * d;
    z0 = p[0];
    z1 = CIR ? p[1] : 0.0;
  } else {
    if (CIR) ns.next2(z0, z1);
    else { z0 = ns.next(); z1 = 0.0; }
  }
}

// threshold dead-band (src/products/netting_set.py:48-72)
template <typename R>
__device__ __forceinline__ R apply_threshold(const R &x, double h) {
  const double v = val(x);
  if (v > h) return x - h;
  if (v < -h) return x + h;
  return RealTraits<R>::zero();
}

// =====================================================================================
// Main simulation kernel
// slot layout: [n_metric][NS][4+2NT] = pos, pos^2, neg, neg^2, d pos[NT], d neg[NT]
//              then [NS][4+2NT]      = pv, pv^2, cva, cva^2, d pv[NT], d cva[NT]
// Value slots hold sum(x - c) and sum((x - c)^2) with c = shift[slot], the value global
// path 0 takes (written by a one-path "pilot" launch of this same kernel).  Shifting by
// a sample of the distribution keeps the variance formula free of cancellation and makes
// degenerate dates (all paths equal, e.g. t = 0) give an exact zero Monte Carlo error.
//
// Layout choices that came out of the first ncu profile (profiles/r01_irc_main_v0_*):
//  * PP paths per thread, evaluated in lock-step: all plan loads, branches and index
//    arithmetic are shared by the PP paths and their Horner chains interleave;
//  * every per-step / per-date scalar sits in one packed record (mcre_irc_create packs
//    them), read with a handful of wide uniform loads instead of ~45 scalar loads;
//  * the "CVA only" case (one netting set, no threshold / collateral, no other metric, stochastic intensity)
//    has its own kernel: irc_cva.cu.
// =====================================================================================
constexpr int STEP_HDR = 4;   // dt, sqrt(dt), bits(date index), pad
constexpr int DATE_HDR = 6;   // bits(flags|(expo+1)<<32), bits((metric+1)|float_off<<32), bits(float_cnt), pad, shift, scale

__device__ __forceinline__ int lo32(double x) { return __double2loint(x); }
__device__ __forceinline__ int hi32(double x) { return __double2hiint(x); }

// Paths per thread / resident 128-thread blocks per SM of each build.  The FP64 pipe needs
// in-warp ILP (fastmath.cuh, MCRE_VP): the value-only builds carry per-set cashflow / exposure-history
// state for several paths per thread; tangent builds run one path.
#ifndef MCRE_IRC_PP2
#define MCRE_IRC_PP2 4     // paths per thread of the 2-set value-only build
#endif
#ifndef MCRE_IRC_MINB2
#define MCRE_IRC_MINB2 2
#endif
__host__ __device__ constexpr int irc_pp(int nt, int ns) { return nt > 0 ? 1 : (ns == 1 ? 4 : (ns == 2 ? MCRE_IRC_PP2 : 2)); }
__host__ __device__ constexpr int irc_minb(int nt, int ns) { return nt > 0 ? 1 : (ns == 1 ? 2 : (ns == 2 ? MCRE_IRC_MINB2 : 4)); }
template <int NT, int NS, bool CIR, int SCHEME, int PP, bool BERM>
__global__ void __launch_bounds__(128, irc_minb(NT, NS)) irc_main_kernel(IrcDev P, RngDev rng, ShardDev sh,
                                                                         double *partial, double *spill,
                                                                         double *shift, int pilot) {
  typedef typename RealOf<NT>::type R;
  typedef RealTraits<R> T;
  fm_tables_init();
  constexpr int W = NT + 1;
  constexpr int NV = 4 + 2 * NT;        // values per (set, date)
  constexpr int NVB = NS * NV;          // values per block_accumulate call
  constexpr int SR = STEP_HDR + 4 * W;  // packed step record stride
  extern __shared__ double smem[];
  const int nw = blockDim.x >> 5;
  const int n_slots = (P.n_metric + 1) * NVB;
  double *acc = smem;                   // [n_slots]
  double *stage = smem + n_slots;       // [2][nw][NVB]
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  const int DR = (DATE_HDR + 2 * W + 3 * W * P.n_sets + 1) & ~1;  // even: records are read as double2

  IrcParams<R, CIR> mp;
  irc_load_params<R, CIR>(P, mp);
  const int acc_flags = P.acc_flags;
  const bool vas_second = CIR && P.vas_noise == 1, cir_second = CIR && P.cir_noise == 1, cir_det = P.cir_det != 0;
  const bool y_positive = CIR && val(mp.y0) > 0.0;
  double thr[NS]; int sflags[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    thr[s] = s < P.n_sets ? __ldg(P.set_threshold + s) : 0.0;
    sflags[s] = s < P.n_sets ? __ldg(P.set_flags + s) : 0;
  }

  for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) acc[i] = 0.0;
    __syncthreads();
    int parity = 0;
    for (int it = 0; it < sh.chunk; it += blockDim.x * PP) {
      long long lpath[PP], gpath[PP];
      bool live[PP];
      NormalStream ns[PP];          // Vasicek only: one normal per step
      NormalStreamV<PP> nsv;        // Vasicek + CIR++: two normals per step, paths in lock-step
      IrcState<R> st[PP];
      R pv[PP][NS], cva[PP][NS], hist[PP][NS][MCRE_IRC_MAX_LAG];
      unsigned alive[PP];   // bit b: Bermudan unit b still holds its exercise right
#pragma unroll
      for (int p = 0; p < PP; ++p) {
        lpath[p] = chunk * sh.chunk + it + p * (int)blockDim.x + threadIdx.x;
        // (PP that does not divide chunk / blockDim: the tail lanes of the last pass idle)
        live[p] = lpath[p] < sh.n_paths && it + p * (int)blockDim.x + (int)threadIdx.x < sh.chunk;
        gpath[p] = P.path_list ? P.path_list[live[p] ? lpath[p] : 0] : sh.path_begin + (live[p] ? lpath[p] : 0);
        ns[p].init(rng, (unsigned long long)gpath[p]);
        st[p].r = mp.r0; st[p].logB = T::zero(); st[p].y = mp.y0; st[p].logBl = T::zero();
        alive[p] = BERM ? ((1u << P.n_berm) - 1u) : 0u;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          pv[p][s] = T::zero(); cva[p][s] = T::zero();
#pragma unroll
          for (int l = 0; l < MCRE_IRC_MAX_LAG; ++l) hist[p][s][l] = T::zero();
        }
      }
      nsv.init(rng, gpath);

      // ---- date evaluation (cashflows -> exposure -> metrics) ------------------------
      auto eval_date = [&](int di) {
        const double *dr = P.date_rec + (size_t)di * DR;
        const double2 h0 = __ldg((const double2 *)dr), h1 = __ldg((const double2 *)dr + 1),
                      h2 = __ldg((const double2 *)dr + 2);
        const int flags = lo32(h0.x), e = hi32(h0.x) - 1, m = lo32(h0.y) - 1;
        if (!(flags & (MCRE_DATE_HAS_CASHFLOW | MCRE_DATE_HAS_EXPOSURE | MCRE_DATE_HAS_METRIC | MCRE_DATE_HAS_EXERCISE)))
          return;
        const double bshift = h2.x, bscale = h2.y;
        const double *dc = dr + DATE_HDR;   // C[w], B[w], coef[set][3][w]
        R invN[PP];
#pragma unroll
        for (int p = 0; p < PP; ++p) invN[p] = r_exp(-st[p].logB);  // 1 / numeraire (vasicek.py:154-156)
        if ((flags & MCRE_DATE_HAS_CASHFLOW) && (acc_flags & MCRE_ACC_PV)) {
          R cf[PP][NS];
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const double fx = s < P.n_sets ? __ldg(P.set_fix + (size_t)s * P.n_dates + di) : 0.0;
#pragma unroll
            for (int p = 0; p < PP; ++p) cf[p][s] = T::lift(fx);
          }
          const int j0 = hi32(h0.y), j1 = j0 + lo32(h1.x);
          for (int j = j0; j < j1; ++j) {
            // LIBOR from the bond price at the payment date's own short rate (bond.py:55-66)
            const R alpha = T::load(P.float_coef, j * 2 + 0), B = T::load(P.float_coef, j * 2 + 1);
            const double inv_tau = __ldg(P.float_inv_tau + j);
#pragma unroll
            for (int p = 0; p < PP; ++p) {
              const R libor = (r_exp(B * st[p].r - alpha) - 1.0) * inv_tau;
#pragma unroll
              for (int s = 0; s < NS; ++s)
                if (s < P.n_sets) cf[p][s] = cf[p][s] + libor * __ldg(P.set_float + (size_t)s * P.n_float + j);
            }
          }
#pragma unroll
          for (int p = 0; p < PP; ++p)
#pragma unroll
            for (int s = 0; s < NS; ++s) pv[p][s] = pv[p][s] + cf[p][s] * invN[p];
        }
        if constexpr (BERM) {
          // exercise decisions come before the exposure of the same date (controller.py:417-430)
          const int x0 = __ldg(P.date_ex_off + di), x1 = __ldg(P.date_ex_off + di + 1);
          for (int x = x0; x < x1; ++x) {
            const int b = __ldg(P.ex_unit + x), bset = __ldg(P.berm_set + b);
            const double xs = __ldg(P.ex_basis + 2 * x), xc = __ldg(P.ex_basis + 2 * x + 1);
            const bool last = __ldg(P.ex_last + x) != 0;   // no continuation after the last date
            const double e0 = __ldg(P.ex_coef + (size_t)(3 * x) * W), e1 = __ldg(P.ex_coef + (size_t)(3 * x + 1) * W),
                         e2 = __ldg(P.ex_coef + (size_t)(3 * x + 2) * W);
#pragma unroll
            for (int p = 0; p < PP; ++p) {
              const R imm = irc_exercise_value<R>(P, x, st[p].r);
              const double u = (val(st[p].r) - xs) * xc;
              const double cont = last ? 0.0 : e0 + u * (e1 + u * e2);
              // hard indicator: immediate > continuation and a right left (bermudan_option.py:121)
              if (((alive[p] >> b) & 1u) && val(imm) > cont) {
                alive[p] &= ~(1u << b);
#pragma unroll
                for (int s = 0; s < NS; ++s) if (s == bset) pv[p][s] = pv[p][s] + imm * invN[p];
              }
            }
          }
        }
        if (flags & MCRE_DATE_HAS_EXPOSURE) {
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            R c0 = T::zero(), c1 = T::zero(), c2 = T::zero();
            if (s < P.n_sets) { c0 = T::load(dc, 2 + s * 3); c1 = T::load(dc, 3 + s * 3); c2 = T::load(dc, 4 + s * 3); }
#pragma unroll
            for (int p = 0; p < PP; ++p) {
#pragma unroll
              for (int l = MCRE_IRC_MAX_LAG - 1; l > 0; --l) hist[p][s][l] = hist[p][s][l - 1];
              const R u = (st[p].r - bshift) * bscale;
              R cont = c0 + u * (c1 + u * c2);
              if constexpr (BERM) {
                // state-dependent coefficients: exercised units (state 0) have none (controller.py:438-447)
                for (int b = 0; b < P.n_berm; ++b) {
                  if (__ldg(P.berm_set + b) != s || !((alive[p] >> b) & 1u)) continue;
                  const double *bc = P.berm_expo_coef + ((size_t)e * P.n_berm + b) * 3 * W;
                  cont = cont + (T::load(bc, 0) + u * (T::load(bc, 1) + u * T::load(bc, 2)));
                }
              }
              hist[p][s][0] = cont * invN[p];  // continuation / numeraire (controller.py:438-447)
            }
          }
        }
        if (flags & MCRE_DATE_HAS_METRIC) {
          double vals[NVB];
#pragma unroll
          for (int i = 0; i < NVB; ++i) vals[i] = 0.0;
          const bool cva_date = (acc_flags & MCRE_ACC_CVA) && m < P.n_metric - 1;
          R dflt[PP];
#pragma unroll
          for (int p = 0; p < PP; ++p) dflt[p] = T::zero();
          if (CIR && cva_date) {
            // S(0,t_k) = exp(-logB_lambda); S(t_k,t_k+1 | y) = C exp(-B y)   (cirpp.py:298-317)
            const R C = T::load(dc, 0), Bc = T::load(dc, 1);
#pragma unroll
            for (int p = 0; p < PP; ++p) dflt[p] = r_exp(-st[p].logBl) * (1.0 - C * r_exp(-(Bc * st[p].y)));
          }
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const int lag = ((sflags[s] & 1) && s < P.n_sets) ? __ldg(P.set_lag + (size_t)s * P.n_metric + m) : -1;
            const int sb = m * NVB + s * NV;
            double sh_pos = 0.0, sh_neg = 0.0;
            if (!pilot) { sh_pos = shift[sb + 0]; sh_neg = shift[sb + 2]; }
#pragma unroll
            for (int p = 0; p < PP; ++p) {
              R unsec;
              if (sflags[s] & 1) {
                R delayed = T::zero();
#pragma unroll
                for (int l = 0; l < MCRE_IRC_MAX_LAG; ++l) if (l == lag) delayed = hist[p][s][l];
                unsec = hist[p][s][0] - apply_threshold(delayed, thr[s]);
              } else {
                unsec = apply_threshold(hist[p][s][0], thr[s]);
              }
              const R pos = r_relu(unsec);
              const R neg = -r_relu(-unsec);
              if (cva_date && (sflags[s] & 2)) cva[p][s] = cva[p][s] + pos * dflt[p];
              if (pilot && p == 0 && threadIdx.x == 0) { shift[sb + 0] = val(pos); shift[sb + 2] = val(neg); }
              const double keep = live[p] ? 1.0 : 0.0;
              const double dp = val(pos) - sh_pos, dn = val(neg) - sh_neg;
              vals[s * NV + 0] += keep * dp; vals[s * NV + 1] += keep * dp * dp;
              vals[s * NV + 2] += keep * dn; vals[s * NV + 3] += keep * dn * dn;
#pragma unroll
              for (int k = 0; k < NT; ++k) {
                vals[s * NV + 4 + k] += keep * tan_of(pos, k);
                vals[s * NV + 4 + NT + k] += keep * tan_of(neg, k);
              }
              if ((acc_flags & MCRE_ACC_SPILL) && live[p] && s < P.n_sets && !P.tan_spill)
                spill[((size_t)s * P.n_metric + m) * sh.n_paths + lpath[p]] = val(unsec);
              if constexpr (NT > 0) {
                if (P.tan_spill && live[p] && s < P.n_sets && !pilot) {
#pragma unroll
                  for (int k = 0; k < NT; ++k)
                    P.tan_spill[(((size_t)lpath[p] * P.n_metric + m) * P.n_sets + s) * NT + k] = tan_of(unsec, k);
                }
              }
            }
          }
          if ((acc_flags & (MCRE_ACC_POS | MCRE_ACC_NEG)) && !pilot)
            {
              if constexpr (NT == 0 && NVB >= 4) block_accumulate_t128<NVB>(vals, acc, m * NVB, stage, parity);
              else block_accumulate<NVB>(vals, acc, m * NVB, stage, NVB, parity);
            }
        }
      };

      for (int di = 0; di < P.n_pre_dates; ++di) eval_date(di);
#pragma unroll 1
      for (int is = 0; is < P.n_sub; ++is) {
        const double *sr = P.step_rec + (size_t)is * SR;
        const double2 g0 = __ldg((const double2 *)sr), g1 = __ldg((const double2 *)sr + 1);
        const double dt = g0.x, sq = g0.y;
        const int di = lo32(g1.x);
        const R sv0 = T::load(sr + STEP_HDR, 0), sv1 = T::load(sr + STEP_HDR, 1);
        R sc0 = T::zero(), sc1 = T::zero();
        if (CIR) { sc0 = T::load(sr + STEP_HDR, 2); sc1 = T::load(sr + STEP_HDR, 3); }
        // ---- draws: PP paths in lock-step (Philox) or the reference's injected stream ----------
        double z0[PP], z1[PP];
        if (rng.mode == MCRE_RNG_INJECT) {
          MCRE_VP {
            const double *zp = rng.z + ((size_t)is * rng.n_total + gpath[p]) * (CIR ? 2 : 1);
            z0[p] = zp[0];
            z1[p] = CIR ? zp[1] : 0.0;
          }
        } else if constexpr (CIR) {
          nsv.next2(z0, z1);
        } else {
          MCRE_VP { z0[p] = ns[p].next(); z1[p] = 0.0; }
        }
        // ---- model step, lock-step over paths.  The correlated noise z @ L^T (model.py:46-48) is
        // folded into per-step coefficients: sigma sqrt(dt) (L z)_i = k_i0 z0 + k_i1 z1.
        R rate0[PP];
        MCRE_VP rate0[p] = st[p].r;
        if (SCHEME == MCRE_SCHEME_ANALYTICAL) {
          // exact OU transition; the 1x1 Cholesky factor of the step covariance is sv1 (vasicek.py:52-86)
          MCRE_VP st[p].r = mp.theta + (st[p].r - mp.theta) * sv0 + sv1 * z0[p];
        } else {
          // r + a (theta_t - r) dt + sigma sqrt(dt) w   (vasicek.py:88-112)
          const R adt = mp.a * dt, ssq = mp.sigma * sq;
          const R kv0 = ssq * (vas_second ? mp.L10 : mp.L00);
          MCRE_VP st[p].r = st[p].r + (sv0 - st[p].r) * adt + kv0 * z0[p];
          if (vas_second) {
            const R kv1 = ssq * mp.L11;
            MCRE_VP st[p].r = st[p].r + kv1 * z1[p];
          }
        }
        if (P.ext_num) {
          R e_num = T::lift(P.ext_rate);
          r_seed(e_num, P.ext_slot);
          MCRE_VP st[p].logB = st[p].logB + e_num * dt;
        } else
        MCRE_VP st[p].logB = st[p].logB + rate0[p] * dt;   // left Riemann sum with the pre-step rate (vasicek.py:80,107)
        if constexpr (CIR) {
          if (cir_det) {                      // cirpp.py:155-172
            MCRE_VP { st[p].logBl = st[p].logBl + sc0 * dt; st[p].y = sc1; }
          } else {                            // full-truncation Euler, cirpp.py:174-198
            // y >= 1e-12 after every step (clamp below); with y0 > 0 the relu is the identity
            R sy[PP], yn[PP], wn[PP];
            if constexpr (NT == 0) {
              if (y_positive) {
                double yv[PP];
                MCRE_VP yv[p] = st[p].y;
                fm_sqrt_posv<PP>(yv, sy);
              } else {
                MCRE_VP sy[p] = r_sqrt(r_relu(st[p].y));
              }
            } else {
              MCRE_VP sy[p] = y_positive ? r_sqrt_pos(st[p].y) : r_sqrt(r_relu(st[p].y));
            }
            const R kdt = mp.kappa * dt, csq = mp.csigma * sq;
            const R kc0 = csq * (cir_second ? mp.L10 : mp.L00);
            MCRE_VP wn[p] = kc0 * z0[p];
            if (cir_second) {
              const R kc1 = csq * mp.L11;
              MCRE_VP wn[p] = wn[p] + kc1 * z1[p];
            }
            MCRE_VP yn[p] = st[p].y + (mp.ctheta - st[p].y) * kdt + sy[p] * wn[p];
            MCRE_VP st[p].logBl = st[p].logBl + (st[p].y + sc0) * dt;
            MCRE_VP st[p].y = r_max(yn[p], 1e-12);
          }
        }
        if (di >= 0) eval_date(di);
      }
      // ---- per-path totals ------------------------------------------------------------
      {
        double vals[NVB];
#pragma unroll
        for (int i = 0; i < NVB; ++i) vals[i] = 0.0;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const int sb = P.n_metric * NVB + s * NV;
          double sh_pv = 0.0, sh_cva = 0.0;
          if (!pilot) { sh_pv = shift[sb + 0]; sh_cva = shift[sb + 2]; }
#pragma unroll
          for (int p = 0; p < PP; ++p) {
            const R c = cva[p][s] * P.lgd;
            if (pilot && p == 0 && threadIdx.x == 0) { shift[sb + 0] = val(pv[p][s]); shift[sb + 2] = val(c); }
            if (P.pv_spill && !pilot && live[p] && s < P.n_sets) P.pv_spill[(size_t)s * sh.n_paths + lpath[p]] = val(pv[p][s]);
            const double keep = live[p] ? 1.0 : 0.0;
            const double dp = val(pv[p][s]) - sh_pv, dcv = val(c) - sh_cva;
            vals[s * NV + 0] += keep * dp; vals[s * NV + 1] += keep * dp * dp;
            vals[s * NV + 2] += keep * dcv; vals[s * NV + 3] += keep * dcv * dcv;
#pragma unroll
            for (int k = 0; k < NT; ++k) {
              vals[s * NV + 4 + k] += keep * tan_of(pv[p][s], k);
              vals[s * NV + 4 + NT + k] += keep * tan_of(c, k);
            }
          }
        }
        if (!pilot) {
          if constexpr (NT == 0 && NVB >= 4) block_accumulate_t128<NVB>(vals, acc, P.n_metric * NVB, stage, parity);
          else block_accumulate<NVB>(vals, acc, P.n_metric * NVB, stage, NVB, parity);
        }
      }
      if (pilot) return;   // the pilot launch simulates global path 0 only: one pass is enough
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) partial[(size_t)chunk * n_slots + i] = acc[i];
    __syncthreads();
  }
}

}  // namespace mcre

// ---- host side shared by irc.cu and irc_berm.cu ----------------------------------------
using namespace mcre;

// Host copies of what the CVA-only kernel's event records are built from (irc_cva.cu)
constexpr int CVA_REC = 24;        // doubles per event record

// The CVA-only kernel evaluates the exposure polynomial in the raw basis [1, r, r^2]: c(u) with u = (r - shift) scale
// becomes c'(r).  Every product and sum is rounded on its own (no FMA contraction on either side), so that the host
// patch (mcre_irc_set_coefficients) and the device patch (irc_patch_coefficients_kernel) give the same bits.
#ifdef __CUDA_ARCH__
__device__ __forceinline__ double rn_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double rn_add(double a, double b) { return __dadd_rn(a, b); }
#else
inline double rn_mul(double a, double b) { volatile double r = a * b; return r; }
inline double rn_add(double a, double b) { volatile double r = a + b; return r; }
#endif
__host__ __device__ inline void irc_raw_basis(double c0, double c1, double c2, double sh, double sc, double out[3]) {
  const double c2s2 = rn_mul(rn_mul(c2, sc), sc), c1s = rn_mul(c1, sc);
  out[2] = c2s2;
  out[1] = rn_add(c1s, -rn_mul(rn_mul(2.0, c2s2), sh));
  out[0] = rn_add(rn_add(c0, -rn_mul(c1s, sh)), rn_mul(rn_mul(c2s2, sh), sh));
}
struct CvaHost {
  int n_sub = 0, n_pre_dates = 0, n_metric = 0, vas_noise = 0, cir_noise = 1;
  double vas[4] = {0, 0, 0, 0}, cir[3] = {0, 0, 0}, chol[4] = {1, 0, 0, 1}, y0 = 0.0, lgd = 0.0;
  std::vector<double> step_dt, step_theta, step_psi;
  std::vector<int> step_date, date_flags, date_metric;
};

struct mcre_irc_plan {
  IrcDev d;
  CvaHost cva;
  std::vector<double> cva_rec_host;
  double *cva_rec_dev = nullptr;
  unsigned *cva_sync_dev = nullptr;
  DevArray<double> cva_rec;
  DevArray<int> cva_sync;
  DevArena arena;   // all plan tables live in one device allocation
  DevArray<double> vas, cir, cir_init, chol, step_dt, step_vas, step_cir, float_coef, float_inv_tau, set_fix,
      set_float, set_threshold, expo_coef, expo_basis, cva_coef, unit_fix, unit_float, reg_basis;
  DevArray<int> step_date, date_flags, date_expo, date_metric, date_reg, date_float_off, set_flags, set_lag;
  DevArray<double> step_rec, date_rec;
  std::vector<double> h_date_rec;   // host copy: coefficients are patched in after the regression solve
  std::vector<int> h_date_expo;
  int date_stride = 0;
  size_t expo_coef_count = 0;
  bool cva_only = false;
  bool any_collateral = false;   // some netting set of the plan is MPoR-collateralised
  int max_lag = 0;               // largest MPoR look-back of the plan, in exposure dates
  DevArray<int> berm_set, date_ex_off, ex_unit, ex_last, ex_term_off;
  DevArray<double> berm_strike, berm_sign, ex_const, term_coef, term_w, ex_basis, ex_coef, berm_expo_coef;
  size_t ex_coef_count = 0, berm_expo_count = 0;
};


using namespace mcre;
template <int NT, int NS, bool BERM>
static int launch_main(mcre_irc_plan *p, const RngDev &rng, const ShardDev &sh, double *partial, double *spill,
                       double *shift, cudaStream_t st) {
  const IrcDev &d = p->d;

  const int threads = 128, nw = threads / 32;
  const int nvb = NS * (4 + 2 * NT);
  // accumulators + reduction stage: [2][nw][nvb] (shuffle trees) or [2][nvb][128] (transposed reduction, value-only)
  const size_t smem = ((size_t)(d.n_metric + 1) * nvb + 2 * (NT == 0 ? 128 : nw) * nvb) * sizeof(double);
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  // The pilot launch (global path 0 -> the common shift of the shifted sums) runs on every rank, also on one whose
  // shard is empty: all ranks must finish their all-reduced sums with the same shift.
#define LAUNCH(CIRV, SCH)                                                                              \
  do {                                                                                                 \
    auto k = irc_main_kernel<NT, NS, CIRV, SCH, irc_pp(NT, NS), BERM>;                                 \
    /* (static shared memory: 14 KB of function tables; static + dynamic beyond 48 KB needs the opt-in) */ \
    MCRE_SMEM(k, smem, "irc main kernel does not fit: too many metric dates x tangents (%s%lld bytes of shared memory)"); \
    int per_sm = 1;                                                                                    \
    MCRE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem));               \
    if (per_sm < 1) return fail(-3, "irc main kernel does not fit: too many metric dates x tangents%s", ""); \
    long long grid = (long long)sm_count() * per_sm;                                                   \
    if (grid > n_chunks) grid = n_chunks;                                                              \
    ShardDev pilot_sh{0, 1, sh.chunk};                                                                 \
    k<<<1, threads, smem, st>>>(d, rng, pilot_sh, partial, spill, shift, 1);                           \
    MCRE_LAUNCHED();                                                                                   \
    if (n_chunks > 0) {                                                                                \
      k<<<(unsigned)grid, threads, smem, st>>>(d, rng, sh, partial, spill, shift, 0);                  \
      MCRE_LAUNCHED();                                                                                 \
    }                                                                                                  \
  } while (0)
  if (d.has_cir) LAUNCH(true, MCRE_SCHEME_EULER);
  else if (d.scheme == MCRE_SCHEME_ANALYTICAL) LAUNCH(false, MCRE_SCHEME_ANALYTICAL);
  else LAUNCH(false, MCRE_SCHEME_EULER);
#undef LAUNCH
  return 0;
}


static inline int ns_template(int n_sets) { return n_sets <= 1 ? 1 : (n_sets <= 2 ? 2 : 4); }

// Picks the template instantiation for (tangents, netting sets).  Tangent builds exist for up
// to 2 netting sets per launch (register budget); the host splits larger books into groups
// and replays the same Philox streams.
template <bool BERM>
static int irc_dispatch_main(mcre_irc_plan *p, const RngDev &r, const ShardDev &sh, double *d_partial, double *d_spill,
                             double *d_shift, cudaStream_t st) {
  const int ns = ns_template(p->d.n_sets);
  if (p->d.nt == 0) {
    return ns == 1 ? launch_main<0, 1, BERM>(p, r, sh, d_partial, d_spill, d_shift, st)
         : ns == 2 ? launch_main<0, 2, BERM>(p, r, sh, d_partial, d_spill, d_shift, st)
                   : launch_main<0, 4, BERM>(p, r, sh, d_partial, d_spill, d_shift, st);
  }
  if (ns > 2) return fail(-3, "irc: at most 2 netting sets per launch when tangents are on%s", "");
  if (p->d.nt == 4) {
    return ns == 1 ? launch_main<4, 1, BERM>(p, r, sh, d_partial, d_spill, d_shift, st)
                   : launch_main<4, 2, BERM>(p, r, sh, d_partial, d_spill, d_shift, st);
  }
  return ns == 1 ? launch_main<8, 1, BERM>(p, r, sh, d_partial, d_spill, d_shift, st)
                 : launch_main<8, 2, BERM>(p, r, sh, d_partial, d_spill, d_shift, st);
}
// defined in irc_cva.cu (the CVA-only kernel)
void irc_cva_fill_static(mcre_irc_plan *p);
int irc_cva_apply_coefficients(mcre_irc_plan *p, cudaStream_t st);
long long irc_cva_units(long long n_paths);   // summation units (passes) of a shard
int irc_cva_launch(mcre_irc_plan *p, const mcre::RngDev &rng, const mcre::ShardDev &sh, double *partial, double *shift,
                   cudaStream_t st);
// defined in irc_berm.cu (books with Bermudan exercise units)
int irc_dispatch_main_berm(mcre_irc_plan *p, const mcre::RngDev &r, const mcre::ShardDev &sh, double *d_partial,
                           double *d_spill, double *d_shift, cudaStream_t st);
