// Value-only build of the fused interest-rate / credit main pass (no tangents, no exercise units): the same plan
// tables, slot layout, pilot scheme and semantics as irc_main_kernel (irc_main.cuh), written the way the CVA-only
// kernel is (irc_cva.cu) after the round-2 profile of the general template on BASELINE config 2
// (profiles/r02_other_kernels.md: 537 warp instructions per path-step, 100 of them FP64; 51 register moves, 41
// shuffles + 42 adds of per-date reductions, 34 branch instructions, 28 constant loads):
//  * PP = 4 paths per thread in lock-step, every operation interleaved over them;
//  * the SDE step in folded form  r' = r om + c + k z  (EULER: om = 1 - a dt, c = a theta_t dt; ANALYTICAL: om = decay,
//    c = theta (1 - decay)): the folding costs a few uniform operations per step and thread, not per path;
//  * the MPoR look-back ring lives in shared memory, indexed by the exposure date (no register shifting), and is
//    touched only when a set is collateralised;
//  * one transposed block reduction per metric date (block_accumulate_t128);
//  * relu pairs as (x + |x|) / 2, (x - |x|) / 2; the threshold dead-band as x - clamp(x, -h, h);
//  * plan scalars of a date come from the packed date record with a handful of 128-bit loads.
// Replaces, like irc_main_kernel: MonteCarloEngine.generate_paths (engine.py:27-123), request resolution
// (request_interface.py:115-130), Bond / IRS cashflows (bond.py:171-214), the regression-proxy exposure
// (controller.py:438-447), NettingSet threshold / MPoR collateral (netting_set.py:48-72, 136-184) and the metric
// integrands of PV / CE / EPE / ENE / CVA (metrics/*.py).
#pragma once
#include "irc_main.cuh"

namespace mcre {

constexpr int VAL_PP = 4;

// x - clamp(x, -h, h): the symmetric dead-band of netting_set.py:48-72 (x - h above h, x + h below -h, else 0)
__device__ __forceinline__ double val_threshold(double x, double h) { return x - fmin(fmax(x, -h), h); }

template <int NS, bool CIR>
__global__ void __launch_bounds__(128, NS == 1 ? 3 : 2) irc_value_kernel(IrcDev P, RngDev rng, ShardDev sh,
                                                                         double *__restrict__ partial,
                                                                         double *__restrict__ spill, double *shift,
                                                                         int pilot) {
  constexpr int PP = VAL_PP;
  constexpr int NV = 4, NVB = NS * NV;
  constexpr int W = 1, SR = STEP_HDR + 4 * W;
  constexpr int NVR = NVB < 4 ? 4 : NVB;       // the transposed reduction takes at least 4 values
  fm_tables_init();
  extern __shared__ double smem[];
  const int n_slots = (P.n_metric + 1) * NVB;
  double *acc = smem;                           // [n_slots]
  double *stage = acc + n_slots;                // [2][NVR][128]
  double *ring = stage + 2 * NVR * 128;         // [P.ring_depth][NS][128 * PP]: exposure look-back
  const int ring_mask = P.ring_depth - 1;       // (depth: a power of two above the largest MPoR lag of the plan)
  const int tid = threadIdx.x;
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  const int DR = (DATE_HDR + 2 * W + 3 * W * P.n_sets + 1) & ~1;
  const bool inject = rng.mode == MCRE_RNG_INJECT;
  const int acc_flags = P.acc_flags;
  const double a = __ldg(P.vas + 3), sigma = __ldg(P.vas + 1), theta = __ldg(P.vas + 2), r0 = __ldg(P.vas + 0);
  const bool analytical = P.scheme == MCRE_SCHEME_ANALYTICAL;
  // rows of the lower Cholesky factor (model.py:46-48): the noise of factor i is L[i][0] z0 + L[i][1] z1
  const double lv0 = CIR ? __ldg(P.chol + 2 * P.vas_noise) : __ldg(P.chol + 0);
  const double lv1 = CIR ? __ldg(P.chol + 2 * P.vas_noise + 1) : 0.0;
  double kappa = 0.0, ctheta = 0.0, csigma = 0.0, y0 = 0.0, lc0 = 0.0, lc1 = 0.0;
  if (CIR) {
    kappa = __ldg(P.cir + 0); ctheta = __ldg(P.cir + 1); csigma = __ldg(P.cir + 2); y0 = __ldg(P.cir_init);
    lc0 = __ldg(P.chol + 2 * P.cir_noise); lc1 = __ldg(P.chol + 2 * P.cir_noise + 1);
  }
  const bool cir_det = CIR && P.cir_det != 0;
  const bool y_positive = CIR && y0 > 0.0;
  double thr[NS];
  int sflags[NS];
  bool any_coll = false;
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    thr[s] = s < P.n_sets ? __ldg(P.set_threshold + s) : 0.0;
    sflags[s] = s < P.n_sets ? __ldg(P.set_flags + s) : 0;
    any_coll = any_coll || (sflags[s] & 1);
  }

  for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = tid; i < n_slots; i += 128) acc[i] = 0.0;
    __syncthreads();
    int parity = 0;
    for (int it = 0; it < sh.chunk; it += 128 * PP) {
      long long lpath[PP], gpath[PP];
      bool live[PP];
      MCRE_VP {
        const int in_chunk = it + p * 128 + tid;
        lpath[p] = chunk * sh.chunk + in_chunk;
        live[p] = lpath[p] < sh.n_paths && in_chunk < sh.chunk;
        gpath[p] = sh.path_begin + (live[p] ? lpath[p] : 0);
      }
      NormalStreamV<PP> nsv;
      nsv.init(rng, gpath);
      double r[PP], logB[PP], y[PP], logBl[PP], zb[PP], pv[PP][NS], cva[PP][NS], cur[PP][NS];
      MCRE_VP {
        r[p] = r0; logB[p] = 0.0; y[p] = y0; logBl[p] = 0.0; zb[p] = 0.0;
#pragma unroll
        for (int s = 0; s < NS; ++s) { pv[p][s] = 0.0; cva[p][s] = 0.0; cur[p][s] = 0.0; }
      }
      if (any_coll) {
        // exposures before the first exposure date count as zero (netting_set.py:139-146)
#pragma unroll
        for (int l = 0; l < P.ring_depth; ++l)
#pragma unroll
          for (int s = 0; s < NS; ++s)
            MCRE_VP ring[(l * NS + s) * (128 * PP) + p * 128 + tid] = 0.0;
      }

      // (h0, h1, h2: the header of the date record, loaded by the caller ahead of the draws of the step - with two
      // warps per scheduler a load used right away costs its whole latency: round-2 profile, long_scoreboard)
      auto eval_date = [&](int di, const double2 &h0, const double2 &h1, const double2 &h2) {
        const double *dr = P.date_rec + (size_t)di * DR;
        const int flags = lo32(h0.x), e = hi32(h0.x) - 1, m = lo32(h0.y) - 1;
        if (!(flags & (MCRE_DATE_HAS_CASHFLOW | MCRE_DATE_HAS_EXPOSURE | MCRE_DATE_HAS_METRIC))) return;
        const double bshift = h2.x, bscale = h2.y;
        const double *dc = dr + DATE_HDR;          // C, B, coef[set][3]
        // every plan scalar of the date is loaded here, ahead of the exponentials that need none of them
        double cc[NS][3], sh_pos[NS], sh_neg[NS];
        int lagv[NS];
        const double Cs = __ldg(dc + 0), Bs = __ldg(dc + 1);
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const bool on = s < P.n_sets;
          cc[s][0] = on ? __ldg(dc + 2 + s * 3) : 0.0; cc[s][1] = on ? __ldg(dc + 3 + s * 3) : 0.0;
          cc[s][2] = on ? __ldg(dc + 4 + s * 3) : 0.0;
          const bool mt = (flags & MCRE_DATE_HAS_METRIC) != 0;
          sh_pos[s] = (mt && !pilot) ? __ldg(shift + m * NVB + s * NV + 0) : 0.0;
          sh_neg[s] = (mt && !pilot) ? __ldg(shift + m * NVB + s * NV + 2) : 0.0;
          lagv[s] = (mt && on && (sflags[s] & 1)) ? __ldg(P.set_lag + (size_t)s * P.n_metric + m) : -1;
        }
        double nlb[PP], invN[PP];
        MCRE_VP nlb[p] = -logB[p];
        fm_exp_tv<PP>(nlb, invN);                    // 1 / numeraire (vasicek.py:154-156)
        if ((flags & MCRE_DATE_HAS_CASHFLOW) && (acc_flags & MCRE_ACC_PV)) {
          double cf[PP][NS];
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const double fx = s < P.n_sets ? __ldg(P.set_fix + (size_t)s * P.n_dates + di) : 0.0;
            MCRE_VP cf[p][s] = fx;
          }
          const int j0 = hi32(h0.y), j1 = j0 + lo32(h1.x);
          for (int j = j0; j < j1; ++j) {
            // LIBOR from the bond price at the payment date's own short rate (bond.py:55-66)
            const double alpha = __ldg(P.float_coef + j * 2), B = __ldg(P.float_coef + j * 2 + 1);
            const double inv_tau = __ldg(P.float_inv_tau + j);
            double xa[PP], ip[PP];
            MCRE_VP xa[p] = fma(B, r[p], -alpha);
            fm_exp_tv<PP>(xa, ip);
            MCRE_VP ip[p] = (ip[p] - 1.0) * inv_tau;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
              if (s < P.n_sets) {
                const double wgt = __ldg(P.set_float + (size_t)s * P.n_float + j);
                MCRE_VP cf[p][s] = fma(ip[p], wgt, cf[p][s]);
              }
            }
          }
#pragma unroll
          for (int s = 0; s < NS; ++s) { MCRE_VP pv[p][s] = fma(cf[p][s], invN[p], pv[p][s]); }
        }
        if (flags & MCRE_DATE_HAS_EXPOSURE) {
          double u[PP];
          MCRE_VP u[p] = (r[p] - bshift) * bscale;
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            // continuation / numeraire (controller.py:438-447)
            MCRE_VP cur[p][s] = fma(u[p], fma(u[p], cc[s][2], cc[s][1]), cc[s][0]) * invN[p];
            if (sflags[s] & 1) { MCRE_VP ring[((e & ring_mask) * NS + s) * (128 * PP) + p * 128 + tid] = cur[p][s]; }
          }
        }
        if (flags & MCRE_DATE_HAS_METRIC) {
          double vals[NVR];
#pragma unroll
          for (int i = 0; i < NVR; ++i) vals[i] = 0.0;
          const bool cva_date = (acc_flags & MCRE_ACC_CVA) && m < P.n_metric - 1;
          double dflt[PP];
          MCRE_VP dflt[p] = 0.0;
          if (CIR && cva_date) {
            // S(0,t_k) = exp(-logB_lambda); S(t_k,t_k+1 | y) = C exp(-B y)   (cirpp.py:298-317)
            const double C = Cs, Bc = Bs;
            double xs[PP], xh[PP], es[PP], eh[PP];
            MCRE_VP xs[p] = -logBl[p];
            MCRE_VP xh[p] = -(Bc * y[p]);
            fm_exp_tv<PP>(xs, es);
            fm_exp_tv<PP>(xh, eh);
            MCRE_VP dflt[p] = es[p] * fma(-C, eh[p], 1.0);
          }
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const int sb = m * NVB + s * NV;
            double unsec[PP];
            if (sflags[s] & 1) {
              const int lag = lagv[s];
              // collateral = thresholded exposure at t_k - MPoR, looked up by exposure index; none before t0
              // (netting_set.py:136-146, 175-176)
              if (lag >= 0) {
                const int slot = (e - lag) & ring_mask;
                MCRE_VP {
                  const double delayed = ring[(slot * NS + s) * (128 * PP) + p * 128 + tid];
                  unsec[p] = cur[p][s] - (thr[s] != 0.0 ? val_threshold(delayed, thr[s]) : delayed);
                }
              } else {
                MCRE_VP unsec[p] = cur[p][s];
              }
            } else {
              MCRE_VP unsec[p] = thr[s] != 0.0 ? val_threshold(cur[p][s], thr[s]) : cur[p][s];
            }
            double pos[PP], neg[PP];
            MCRE_VP pos[p] = 0.5 * (unsec[p] + fabs(unsec[p]));     // relu(E)
            MCRE_VP neg[p] = 0.5 * (unsec[p] - fabs(unsec[p]));     // -relu(-E)
            if (cva_date && (sflags[s] & 2)) { MCRE_VP cva[p][s] = fma(pos[p], dflt[p], cva[p][s]); }
            if (pilot && tid == 0) { shift[sb + 0] = pos[0]; shift[sb + 2] = neg[0]; }
            MCRE_VP {
              const double dp = live[p] ? pos[p] - sh_pos[s] : 0.0, dn = live[p] ? neg[p] - sh_neg[s] : 0.0;
              vals[s * NV + 0] += dp; vals[s * NV + 1] = fma(dp, dp, vals[s * NV + 1]);
              vals[s * NV + 2] += dn; vals[s * NV + 3] = fma(dn, dn, vals[s * NV + 3]);
            }
            if ((acc_flags & MCRE_ACC_SPILL) && s < P.n_sets && !pilot) {
              MCRE_VP { if (live[p]) spill[((size_t)s * P.n_metric + m) * sh.n_paths + lpath[p]] = unsec[p]; }
            }
          }
          if ((acc_flags & (MCRE_ACC_POS | MCRE_ACC_NEG)) && !pilot)
            block_accumulate_t128<NVR>(vals, acc, m * NVB, stage, parity);
        }
      };

      for (int di = 0; di < P.n_pre_dates; ++di) {
        const double2 *dh = (const double2 *)(P.date_rec + (size_t)di * DR);
        eval_date(di, __ldg(dh), __ldg(dh + 1), __ldg(dh + 2));
      }
      int di_next = P.n_sub > 0 ? __ldg(P.step_date) : -1;
#pragma unroll 1
      for (int is = 0; is < P.n_sub; ++is) {
        // loads first, uses after the draws: the step record, the index of the date after the NEXT step, and the
        // header of the date this step ends on
        const int di = di_next;
        if (is + 1 < P.n_sub) di_next = __ldg(P.step_date + is + 1);
        const double *sr = P.step_rec + (size_t)is * SR;
        const double2 g0 = __ldg((const double2 *)sr), g2 = __ldg((const double2 *)sr + 2),
                      g3 = __ldg((const double2 *)sr + 3);
        const double2 *dh = (const double2 *)(P.date_rec + (size_t)(di >= 0 ? di : 0) * DR);
        const double2 h0 = __ldg(dh), h1 = __ldg(dh + 1), h2 = __ldg(dh + 2);
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
          if ((is & 1) == 0) nsv.next2(z0, zb);        // one normal per step: a Box-Muller pair serves two steps
          else { MCRE_VP z0[p] = zb[p]; }
          MCRE_VP z1[p] = 0.0;
        }
        const double dt = g0.x, sq = g0.y, sv0 = g2.x, sv1 = g2.y, sc0 = g3.x, sc1 = g3.y;
        // folded step constants (uniform: once per step and thread)
        double om_v, c_v, kv0, kv1;
        if (analytical) {       // exact OU transition (vasicek.py:52-86): decay sv0, noise std sv1
          om_v = sv0; c_v = fma(-theta, sv0, theta); kv0 = sv1; kv1 = 0.0;
        } else {                // r + a (theta_t - r) dt + sigma sqrt(dt) w   (vasicek.py:88-112)
          const double adt = a * dt, ssq = sigma * sq;
          om_v = 1.0 - adt; c_v = sv0 * adt; kv0 = ssq * lv0; kv1 = ssq * lv1;
        }
        MCRE_VP logB[p] = fma(P.ext_num ? P.ext_rate : r[p], dt, logB[p]);      // left Riemann sum with the pre-step rate (vasicek.py:80,107)
        MCRE_VP r[p] = fma(kv0, z0[p], fma(r[p], om_v, c_v));
        if (kv1 != 0.0) { MCRE_VP r[p] = fma(kv1, z1[p], r[p]); }
        if (CIR) {
          if (cir_det) {                               // cirpp.py:155-172
            MCRE_VP { logBl[p] = fma(sc0, dt, logBl[p]); y[p] = sc1; }
          } else {                                     // full-truncation Euler, cirpp.py:174-198
            const double kdt = kappa * dt, csq = csigma * sq;
            const double om_c = 1.0 - kdt, c_c = ctheta * kdt, kc0 = csq * lc0, kc1 = csq * lc1;
            double yp[PP], sy[PP], wn[PP], yn[PP];
            // sqrt(max(y, 0)): y >= 1e-12 after every step (clamp below), so only y0 = 0 needs the guard
            if (y_positive) {
              fm_sqrt_posv<PP>(y, sy);
            } else {
              MCRE_VP yp[p] = fmax(y[p], 1e-300);
              fm_sqrt_posv<PP>(yp, sy);
              MCRE_VP sy[p] = y[p] > 0.0 ? sy[p] : 0.0;
            }
            MCRE_VP wn[p] = kc0 * z0[p];
            if (kc1 != 0.0) { MCRE_VP wn[p] = fma(kc1, z1[p], wn[p]); }
            MCRE_VP yn[p] = fma(sy[p], wn[p], fma(y[p], om_c, c_c));
            MCRE_VP logBl[p] = fma(y[p] + sc0, dt, logBl[p]);
            MCRE_VP y[p] = fmax(yn[p], 1e-12);
          }
        }
        if (di >= 0) eval_date(di, h0, h1, h2);
      }
      // ---- per-path totals ------------------------------------------------------------------------
      {
        double vals[NVR];
#pragma unroll
        for (int i = 0; i < NVR; ++i) vals[i] = 0.0;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const int sb = P.n_metric * NVB + s * NV;
          double sh_pv = 0.0, sh_cva = 0.0;
          if (!pilot) { sh_pv = shift[sb + 0]; sh_cva = shift[sb + 2]; }
          if (pilot && tid == 0) { shift[sb + 0] = pv[0][s]; shift[sb + 2] = cva[0][s] * P.lgd; }
          if (P.pv_spill && !pilot && s < P.n_sets) {
            MCRE_VP { if (live[p]) P.pv_spill[(size_t)s * sh.n_paths + lpath[p]] = pv[p][s]; }
          }
          MCRE_VP {
            const double dp = live[p] ? pv[p][s] - sh_pv : 0.0, dcv = live[p] ? cva[p][s] * P.lgd - sh_cva : 0.0;
            vals[s * NV + 0] += dp; vals[s * NV + 1] = fma(dp, dp, vals[s * NV + 1]);
            vals[s * NV + 2] += dcv; vals[s * NV + 3] = fma(dcv, dcv, vals[s * NV + 3]);
          }
        }
        if (!pilot) block_accumulate_t128<NVR>(vals, acc, P.n_metric * NVB, stage, parity);
      }
      if (pilot) return;   // the pilot launch simulates global path 0 only: one pass is enough
    }
    __syncthreads();
    for (int i = tid; i < n_slots; i += 128) partial[(size_t)chunk * n_slots + i] = acc[i];
    __syncthreads();
  }
}

// Launch (pilot + main) of the value-only kernel; same contract as launch_main in irc_main.cuh.
template <int NS>
static int launch_value(mcre_irc_plan *p, const RngDev &rng, const ShardDev &sh, double *partial, double *spill,
                        double *shift, cudaStream_t st) {
  const IrcDev &d = p->d;
  constexpr int NVB = NS * 4, NVR = NVB < 4 ? 4 : NVB;
  // (the look-back ring is only there when a set is collateralised)
  const size_t smem = ((size_t)(d.n_metric + 1) * NVB + 2 * NVR * 128 +
                       (p->any_collateral ? (size_t)d.ring_depth * NS * 128 * VAL_PP : 0)) * sizeof(double);
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
#define LAUNCHV(CIRV)                                                                                     \
  do {                                                                                                    \
    auto k = irc_value_kernel<NS, CIRV>;                                                                  \
    MCRE_SMEM(k, smem, "irc value kernel does not fit: too many metric dates / too long an MPoR look-back (%s%lld bytes of shared memory)"); \
    int per_sm = 1;                                                                                       \
    MCRE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, 128, smem));                      \
    if (per_sm < 1) return fail(-3, "irc value kernel does not fit: too many metric dates / too long an MPoR look-back%s", "");        \
    long long grid = (long long)sm_count() * per_sm;                                                      \
    if (grid > n_chunks) grid = n_chunks;                                                                 \
    ShardDev pilot_sh{0, 1, sh.chunk};                                                                    \
    k<<<1, 128, smem, st>>>(d, rng, pilot_sh, partial, spill, shift, 1);                                  \
    MCRE_LAUNCHED();                                                                                      \
    if (n_chunks > 0) {                                                                                   \
      k<<<(unsigned)grid, 128, smem, st>>>(d, rng, sh, partial, spill, shift, 0);                         \
      MCRE_LAUNCHED();                                                                                    \
    }                                                                                                     \
  } while (0)
  if (d.has_cir) LAUNCHV(true); else LAUNCHV(false);
#undef LAUNCHV
  return 0;
}

}  // namespace mcre
