// Equity family: fused path generation + payoff + PV / pathwise-Greek reduction for
// Black-Scholes (single, multi-asset, ModelConfig of BS models), Heston (Euler, Andersen
// QE with fuzzy branching; also several correlated Heston assets) and Schwartz two-factor,
// with European / binary / basket / Asian / barrier payoffs.
//
// SIMT mapping: one LANE per (path, asset).  A warp holds floor(32 / A) paths; the A lanes
// of a path exchange their independent normals with warp shuffles to form the correlated
// noise (z @ L^T, src/models/model.py:46-48) and reduce weighted spots to basket values the
// same way.  Every lane carries the tangents of its own asset's state with respect to its
// own asset's parameters only (3 for Black-Scholes, 7 for Heston, 6 for Schwartz): an
// asset's path never depends on another asset's parameters, so the full gradient over all
// model parameters costs (1 + local parameters) x, not (1 + all parameters) x.  The payoff
// is a function of group-reduced values, so each lane's tangent of it is the part flowing
// through its own asset; the host scatters the lane-local sums to the global parameter
// order (and adds the deterministic-numeraire term).
//
// Nothing but block-reduced sums reaches HBM.  See include/mcre.h for what this replaces.
#define MCRE_FAST_MATH 2
#include "common.cuh"
#include "philox.cuh"
#include "dual2.cuh"
#include "heston.cuh"
#include "reduce.cuh"
#include "launch.cuh"

namespace mcre {

constexpr int EQ_PR = 16;     // doubles per product record
// path-dependent / exercise trackers per launch.  Value-only builds keep 64 of them in dynamically indexed
// per-thread arrays (local memory, touched only at product events): large mixed books need few launches.
// Tangent builds keep 2 in registers (compile-time selects; the trackers carry the tangents).
__host__ __device__ constexpr int eq_ntrk(int nt) { return nt == 0 ? 64 : 2; }
// visits tracker `slot` (none if slot < 0): one dynamic access (NT = 0) or an unrolled compare-select
#define MCRE_TRK_FOR(k, slot)                                                                         \
  for (int k = (NT == 0 ? ((slot) > 0 ? (slot) : 0) : 0), k##_end = (NT == 0 ? (slot) + 1 : NTRK); k < k##_end; ++k) \
    if (k == (slot))
constexpr int EQ_PAR = 8;     // doubles per asset parameter row

struct EqDev {
  int kind, scheme, smoothing, n_assets, noise_dim, n_uniform;
  const double *asset_par; const int *asset_noise, *asset_uniform, *col_asset, *col_elem;
  int n_sub, n_dates, n_pre_dates;
  const double *step_dt, *step_sq; const int *step_date, *step_chol;
  const double *step_aux, *init_aux;
  int corr_mode; const double *chol, *chol_dual;
  const int *date_ev_off, *ev_prod, *ev_flags;
  int n_prod; const double *prod, *prod_w;
  int n_sets;
  const double *ev_data, *prod_x;   // exercise products (Bermudan / American)
  // exposure profiles (analytic Black-Scholes exposure of European options, european_option.py:123-145)
  int n_expo, n_metric, acc_flags;
  const int *date_expo, *date_metric;
  const double *xp;                  // [n_expo][n_prod][4]: type (0 none, 1 analytic BS), time to maturity, 1/numeraire(t), pad
  const double *set_threshold; const int *set_flags, *set_lag;
  // sparse form of a single joint Cholesky factor (built by mcre_eq_create): per asset the non-zeros of
  // the row of its first noise column as (coefficient, source asset << 1 | element); its second column's
  // row is the identity (Heston QE variance draws are independent).  sp_n = 0: use the dense factor.
  int sp_n, n_sub_total;
  const double *sp_coef; const int *sp_src;
  // pre-simulation spill (mcre_eq_presim): spot of every asset per exposure date, date-major, and the
  // discounted cashflow of every product rounded to float32 (the reference's float32 accumulators)
  double *ps_x;   // [n_expo][A][n_paths]
  float *ps_cf;   // [n_prod][n_paths]
  // book splitting (mcre_eq_set_pv_accumulator): per-path discounted cashflow totals of the launch are ADDED
  // to pv_accum [n_sets][n_paths], so a netting set with more path-dependent products than one launch can
  // track is evaluated in several launches over the same Philox streams and finished by mcre_sum_stats
  double *pv_accum;
  // Brownian-bridge barrier monitoring in RNG compatibility mode: the reference's numpy uniforms,
  // [tracker slot][barrier 0/1][n_paths_total][bridge_stride] (NULL: Philox kind 2)
  const double *bridge_u;
  int bridge_stride;
  // book splitting with exposure profiles (mcre_eq_set_exposure_accumulator): the netted exposure of the
  // launch's products is ADDED to expo_accum [n_sets][n_expo][n_paths]; netting terms / metrics are applied
  // afterwards by mcre_eq_unsecured_exposures + mcre_sum_stats
  double *expo_accum;
  // ... and the lane-local tangents of those exposures to expo_accum_tan [n_sets][n_expo][A][nt][n_paths]
  // (mcre_eq_set_exposure_tangent_accumulator; hybrid books, mcre/hybrid.py)
  double *expo_accum_tan;
  // tangent builds (Black-Scholes): tangents of the regression-proxy coefficients with respect to the lane-local
  // parameters of the product's asset, [n_expo][n_prod][3 coefficients][nt] (mcre_eq_set_exposure_coef_tangents),
  // and the tangent spill of the pre-simulation pass (mcre_eq_presim_tangents): ps_dx [n_expo][A][nt][n_paths],
  // ps_dcf [n_prod][nt][n_paths] (f64: the reference's float32 rounding touches values only under autograd's chain)
  const double *xp_tan;
  // ... and of the continuation values of exercise products (exposure type 3), per state s = rights left at row s - 1:
  // [n_expo][n_prod][EQ_MAX_RIGHTS][3 coefficients][nt] (mcre_eq_set_exercise_exposure_coef_tangents)
  const double *xp_ex_tan;
  // per exposure date the products whose record carries an exposure (type != 0), ascending: xact[xact_off[e] .. xact_off[e+1])
  // (built by mcre_eq_create from xp; matured products and the other launches' products are never visited)
  const int *xact_off, *xact;
  double *ps_dx, *ps_dcf;
  // credit factor of a hybrid ModelConfig (mcre_eq_set_credit): CIR++ intensity of the counterparty stepped next to
  // the equity assets (cirpp.py:155-198), its normal = noise column cir_col correlated through cir_row [noise_dim]
  // (the credit row of the joint Cholesky factor); CVA weights per metric date cva_coef [n_metric][2] = (C_k, B_k)
  // of S(t_k, t_k+1 | y) = C exp(-B y) (cirpp.py:246-285); set_cva [n_sets]: the metric's counterparty faces the set
  int has_cir, cir_det, cir_col;
  double cir_kappa, cir_theta, cir_sigma, cir_y0, lgd;
  const double *step_cir, *cir_row, *cva_coef;
  const int *set_cva;
  // book splitting with CVA (mcre_eq_set_cva_weight_spill): the default weights S(0, t_k) (1 - S(t_k, t_k+1 | y_k)) of
  // every path per metric date, [n_metric][n_paths]; mcre_eq_cva_paths combines them with the unsecured exposures
  double *cva_w;
};
constexpr int EQ_XP = 32;      // doubles per exposure record: [0..7] type, state-1 coefficients, basis, numeraire; [16 + 3 (st - 2)] states 2..6
constexpr int EQ_PF = 8;     // exposure records prefetched ahead of the walk (measured: 8 ahead -7 % on the 5k-product CVA book, 32 ahead no gain)
__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
constexpr int EQ_EVD = 32;  // doubles per event record ([16 + 3 (st - 2)]: continuation coefficients of states 2..6) (exercise events: see mcre_eq_desc.ev_data)
constexpr int EQ_MAX_LAG = 4;
constexpr int EQ_MAX_RIGHTS = MCRE_LSM_MAX_RIGHTS;
constexpr int EQ_SPNZ = 8;   // non-zeros kept per sparse correlation row

enum { EQ_EUROPEAN = MCRE_EQ_EUROPEAN, EQ_BINARY = MCRE_EQ_BINARY, EQ_BASKET = MCRE_EQ_BASKET, EQ_ASIAN = MCRE_EQ_ASIAN,
       EQ_BARRIER = MCRE_EQ_BARRIER, EQ_EXERCISE = MCRE_EQ_EXERCISE };
enum { EQ_EV_OBSERVE = MCRE_EQ_EV_OBSERVE, EQ_EV_PAY = MCRE_EQ_EV_PAY, EQ_EV_FIRST = MCRE_EQ_EV_FIRST,
       EQ_EV_EXERCISE = MCRE_EQ_EV_EXERCISE };

template <int KIND> struct EqParCount;
template <> struct EqParCount<MCRE_EQ_BS> { static const int n = 3; };
template <> struct EqParCount<MCRE_EQ_HESTON> { static const int n = 7; };
template <> struct EqParCount<MCRE_EQ_SCHWARTZ> { static const int n = 6; };

// sum of x over the A lanes of this lane's path group
__device__ __forceinline__ double group_sum(double x, int base, int A) {
  double tot = 0.0;
  for (int j = 0; j < A; ++j) tot += __shfl_sync(0xffffffffu, x, (base + j) & 31);
  return tot;
}

template <typename R>
__device__ __forceinline__ R option_payoff(const R &u, double strike, double sign) {
  return r_relu((u - strike) * sign);
}

// barrier survival factor with the always-fuzzy indicator, eps = 0.05 in spot units
// (src/products/barrier_option.py:66-125, src/maths/maths.py:8-9)
template <typename R>
__device__ __forceinline__ R barrier_factor(const R &mx, const R &mn, double barrier, int btype) {
  const R below = r_fuzzy(barrier - mx, true, 0.05);
  const R above = r_fuzzy(mn - barrier, true, 0.05);
  switch (btype) {
    case 1: return below;            // up-and-out
    case 2: return above;            // down-and-out
    case 3: return 1.0 - below;      // up-and-in
    default: return 1.0 - above;     // down-and-in
  }
}

// coef = -2 / (sigma^2 maturity / n_obs) of the Brownian-bridge crossing probability as a function of the volatility
// (c0 = its value): d coef / d sigma = -2 coef / sigma
template <int N> __device__ __forceinline__ Dual<N> bridge_coef(double c0, const Dual<N> &sigma) {
  Dual<N> r = dual_zero<N>(); r.v = c0; r.d[1] = -2.0 * c0 / sigma.v;
  return r;
}
template <int N> __device__ __forceinline__ Dual2<N> bridge_coef(double c0, const Dual2<N> &sigma) {
  return (c0 * sigma.v * sigma.v) / (sigma * sigma);
}

// standard normal CDF of a dual number (tangent = density)
template <int N>
__device__ __forceinline__ Dual<N> dual_ncdf(const Dual<N> &x) {
  Dual<N> r;
  r.v = 0.5 * erfc(-x.v * 0.70710678118654752440);
  const double pdf = 0.39894228040143267794 * exp(-0.5 * x.v * x.v);
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = pdf * x.d[i];
  return r;
}

// Sensitivities of exposure profiles (controller.py:609-627 on EPE / ENE / CE / EEPE): Black-Scholes builds with
// tangents carry the exposures as duals (lane-local tangents like the cashflows); other models keep doubles.
// (NT = 9: the second-order build, Dual2<3> - present values only)
// Heston builds with XH (plans with exposure dates: every exposure a regression proxy on the spot; the analytic branch is
// Black-Scholes only).  Heston plans without exposure dates keep the lean build: exposures as duals cost the 35-Greek
// run of BASELINE config 5 45 % when they rode along unused.
template <int KIND, int NT, bool XH> struct EqExpoTan {
  static const bool on = (KIND == MCRE_EQ_BS && NT > 0 && NT != 9) || (KIND == MCRE_EQ_HESTON && NT > 0 && XH);
};
static inline bool eq_kind_has_exposure_tangents(int kind) { return kind == MCRE_EQ_BS || kind == MCRE_EQ_HESTON; }
template <bool ON, typename R> struct EqExpoReal { typedef double type; };
template <typename R> struct EqExpoReal<true, R> { typedef R type; };

// slot layout: [NS][3] = sum(cf - c), sum((cf - c)^2), sum(payoff * d invN / d r)   then
//              [A][NS][NT] lane-local tangents of sum_p payoff_p * invN_p             then
//              [n_metric][NS][4] exposure sums                                          then (exposure tangents on)
//              [n_metric][A][NS][2][NT] lane-local tangents of sum relu(E), sum -relu(-E)
template <int KIND, int ALT, int NT, int NS, bool XH = false>
__global__ void __launch_bounds__(128, (NT == 0 ? 4 : 2)) eq_main_kernel(EqDev P, RngDev rng, ShardDev sh, double *partial,
                                                      double *shift, double *spill, int pilot) {
  typedef typename RealOf<NT>::type R;
  typedef RealTraits<R> T;
  typedef RealVar<R> V;
  fm_tables_init();
  constexpr int NP = EqParCount<KIND>::n;
  constexpr int NVH = NS * 3;
  constexpr int NVT = NS * (NT > 0 ? NT : 1);
  constexpr int NVX = NS * 4;                 // exposure values per metric date
  constexpr bool XT = EqExpoTan<KIND, NT, XH>::on;
  typedef typename EqExpoReal<XT, R>::type XR;
  constexpr int NVXT = XT ? NS * 2 * NT : 1;  // exposure tangents per (metric date, asset)
  constexpr int NVMAX0 = (NVH > NVT ? NVH : NVT) > NVX ? (NVH > NVT ? NVH : NVT) : NVX;
  constexpr int NVMAX = NVMAX0 > NVXT ? NVMAX0 : NVXT;
  extern __shared__ double smem[];
  const int nw = blockDim.x >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int A = P.n_assets, ppw = 32 / A;
  const int expo_base = NS * 3 + A * NS * NT;
  const int xt_base = expo_base + P.n_metric * NVX;
  const int cva_base = xt_base + (XT ? P.n_metric * A * NVXT : 0);      // [NS][2] sum(cva - c), sum((cva - c)^2)
  const int n_slots = cva_base + ((KIND == MCRE_EQ_BS && P.has_cir) ? NS * 2 : 0);
  double *acc = smem;                 // [n_slots]
  double *stage = smem + n_slots;     // [2][nw][NVMAX]
  const int g = lane / A, a = lane - g * A, base = g * A;
  const bool lane_ok = g < ppw;
  const int aa = lane_ok ? a : 0;     // ghost lanes replay asset 0 and are masked out
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  const int paths_per_iter = nw * ppw;

  // ---- this lane's asset -----------------------------------------------------------
  R par[NP];
#pragma unroll
  for (int k = 0; k < NP; ++k) par[k] = V::make(__ldg(P.asset_par + aa * EQ_PAR + k), k);
  const int c0 = __ldg(P.asset_noise + aa * 2), c1 = __ldg(P.asset_noise + aa * 2 + 1);
  const int uidx = __ldg(P.asset_uniform + aa);
  const int d = P.noise_dim;
  const bool smooth = P.smoothing != 0;
  double spc[EQ_SPNZ];
  int sps[EQ_SPNZ];
#pragma unroll
  for (int k = 0; k < EQ_SPNZ; ++k) {
    spc[k] = k < P.sp_n ? __ldg(P.sp_coef + aa * EQ_SPNZ + k) : 0.0;
    sps[k] = k < P.sp_n ? __ldg(P.sp_src + aa * EQ_SPNZ + k) : 0;
  }

  for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) acc[i] = 0.0;
    __syncthreads();
    int parity = 0;
    for (int it = 0; it < sh.chunk; it += paths_per_iter) {
      const int in_chunk = it + warp * ppw + g;
      const long long lpath = chunk * sh.chunk + in_chunk;
      const bool live = lane_ok && in_chunk < sh.chunk && lpath < sh.n_paths;
      const unsigned long long gpath = (unsigned long long)(sh.path_begin + (live ? lpath : 0));
      NormalStream ns; ns.init(rng, gpath);
      QeStepConst<R> qe;
      qe.dt = -1.0;
      double u_even = 0.5, u_odd = 0.5;

      R s0, s1;
      if constexpr (KIND == MCRE_EQ_BS) { s0 = par[0]; s1 = T::zero(); }
      else if constexpr (KIND == MCRE_EQ_HESTON) { s0 = r_log(par[0]); s1 = par[6]; }
      else { s0 = T::zero(); s1 = T::zero(); }
      double logF = KIND == MCRE_EQ_SCHWARTZ ? __ldg(P.init_aux + aa) : 0.0;
      double cy = P.cir_y0, clogB = 0.0, cva_path[NS];     // credit factor: every lane of the group carries a copy
#pragma unroll
      for (int s = 0; s < NS; ++s) cva_path[s] = 0.0;
      constexpr int NTRK = eq_ntrk(NT);
      R cf[NS], trk_a[NTRK], trk_b[NTRK];
      // Brownian-bridge barriers (value-only builds): previous monitored spot, running no-hit products
      double trk_c[NT == 0 ? NTRK : 1], trk_d[NT == 0 ? NTRK : 1], trk_e[NT == 0 ? NTRK : 1];
      // ... tangent builds (Black-Scholes): the same three as duals, dynamically indexed - they live in local memory and are
      // touched at the observation events of bridge-monitored barriers only
      R brg_c[NT > 0 ? NTRK : 1], brg_d[NT > 0 ? NTRK : 1], brg_e[NT > 0 ? NTRK : 1];
      double numtan[NS];
      XR hist[NS][EQ_MAX_LAG];
#pragma unroll
      for (int s = 0; s < NS; ++s)
#pragma unroll
        for (int l = 0; l < EQ_MAX_LAG; ++l) hist[s][l] = RealTraits<XR>::zero();
#pragma unroll
      for (int s = 0; s < NS; ++s) { cf[s] = T::zero(); numtan[s] = 0.0; }
      if constexpr (NT > 0) {   // (value-only builds: every tracker is set by its FIRST event / the loop below)
#pragma unroll
        for (int k = 0; k < NTRK; ++k) { trk_a[k] = T::zero(); trk_b[k] = T::zero(); }
      }
      // exercise products start with all their rights (state = rights left): exposure dates before the
      // first exercise date already look the state up
      for (int pi = 0; pi < P.n_prod; ++pi) {
        const double *pr = P.prod + (size_t)pi * EQ_PR;
        if ((int)__ldg(pr + 0) != EQ_EXERCISE) continue;
        const int slot = (int)__ldg(pr + 14);
#pragma unroll
        MCRE_TRK_FOR(k, slot) trk_a[k] = T::lift(__ldg(pr + 13));
      }

      auto spot_now = [&]() -> R {
        if (KIND == MCRE_EQ_BS) return s0;
        if (KIND == MCRE_EQ_HESTON) return r_exp(s0);
        return r_exp(logF + s0 + s1);
      };

      // ---- product events of one simulation date --------------------------------------
      // exposure of the date (after its cashflows, controller.py:417-447), netting, collateral, metrics
      auto eval_exposure = [&](int di) {
        if (P.n_expo == 0) return;
        const int xe = __ldg(P.date_expo + di), m = P.ps_x ? -1 : __ldg(P.date_metric + di);
        if (KIND == MCRE_EQ_BS && P.has_cir && P.cva_w && m >= 0 && live && a == 0 && !pilot) {
          const double Ck = __ldg(P.cva_coef + 2 * m), Bk = __ldg(P.cva_coef + 2 * m + 1);
          P.cva_w[(size_t)m * sh.n_paths + lpath] = m < P.n_metric - 1 ? exp(-clogB) * (1.0 - Ck * exp(-Bk * cy)) : 0.0;
        }
        if (xe >= 0 && P.ps_x) {
          if (live) {
            const R Sp = spot_now();
            P.ps_x[((size_t)xe * A + a) * sh.n_paths + lpath] = val(Sp);
            if constexpr (NT > 0) {
              if (P.ps_dx) {
#pragma unroll
                for (int k = 0; k < NT; ++k) P.ps_dx[(((size_t)xe * A + a) * NT + k) * sh.n_paths + lpath] = tan_of(Sp, k);
              }
            }
          }
          return;     // pre-simulation pass: no exposures, no metrics
        }
        if (xe >= 0) {
          const double Sv = val(spot_now());
          XR expo[NS];
#pragma unroll
          for (int s = 0; s < NS; ++s) expo[s] = RealTraits<XR>::zero();
          // the records of a date are walked one after the other and each decides a branch: on books of hundreds of
          // products per launch and ~1000 paths (one warp per scheduler) the walk was a chain of L2 round trips
          // (ncu: long_scoreboard 9 of 14 cycles per issue, half of all stall samples on the record's first load).
          // One 128-byte record = one line: prefetch EQ_PF records ahead into L1.
          const double *xrow = P.xp + (size_t)xe * P.n_prod * EQ_XP;
          const int q0 = __ldg(P.xact_off + xe), q1 = __ldg(P.xact_off + xe + 1);
          for (int q = q0; q < q0 + EQ_PF && q < q1; ++q) prefetch_l1(xrow + (size_t)__ldg(P.xact + q) * EQ_XP);
          for (int q = q0; q < q1; ++q) {
            const int pi = __ldg(P.xact + q);
            const double *op = xrow + (size_t)pi * EQ_XP;
            if (q + EQ_PF < q1) prefetch_l1(xrow + (size_t)__ldg(P.xact + q + EQ_PF) * EQ_XP);
            const int xtype = (int)__ldg(op);
            if (xtype == 0) continue;
            const double *pr = P.prod + (size_t)pi * EQ_PR;
            double v = 0.0;
            if (xtype == 2 || xtype == 3) {
              // regression proxy: continuation(x) / numeraire with x the spot of the product's asset
              // (controller.py:438-447), evaluated on the lane that owns that asset; type 3 (exercise
              // products): the coefficients of the product's current state = rights left, none in state 0
              const double xw = __ldg(P.prod_x + (size_t)pi * A + aa);
              int st = 1;
              if (xtype == 3) {
                const int slot = (int)__ldg(pr + 14);
#pragma unroll
                MCRE_TRK_FOR(k, slot) st = (int)val(trk_a[k]);
              }
              if constexpr (XT) {
                if (xtype == 2 && P.xp_tan) {
                  // the same quadratic on duals: tangents through the spot, the fitted coefficients (differentiated
                  // normal equations of the pre-simulation, mcre/lsm.py:regression_tangents) and the numeraire
                  XR vq = RealTraits<XR>::zero();
                  if (xw != 0.0) {
                    const R uq = (spot_now() - __ldg(op + 5)) * __ldg(op + 6);
                    R q0 = T::lift(__ldg(op + 1)), q1 = T::lift(__ldg(op + 3)), q2 = T::lift(__ldg(op + 4));
                    const double *ct = P.xp_tan + ((size_t)xe * P.n_prod + pi) * 3 * NT;
#pragma unroll
                    for (int k = 0; k < NT; ++k) {
                      q0.d[k] = __ldg(ct + k); q1.d[k] = __ldg(ct + NT + k); q2.d[k] = __ldg(ct + 2 * NT + k);
                    }
                    const R poly = q0 + uq * (q1 + uq * q2);
                    vq = poly * __ldg(op + 2);
                    vq.d[2] += val(poly) * __ldg(op + 7);
                  }
                  const XR totq = r_with_value(vq, group_sum(val(vq), base, A));
                  const int setq = (int)__ldg(pr + 1);
#pragma unroll
                  for (int s = 0; s < NS; ++s) if (s == setq) expo[s] = expo[s] + totq;
                  continue;
                }
                if (xtype == 3 && P.xp_ex_tan) {
                  // exercise products: the quadratic of the current state on duals (coefficients and their tangents
                  // selected by the state, which itself carries none: the reference gathers coefficients by state)
                  XR ve = RealTraits<XR>::zero();
                  if (xw != 0.0 && st > 0) {
                    const R ue = (spot_now() - __ldg(op + 5)) * __ldg(op + 6);
                    const double *cv = st == 1 ? op + 1 : op + 16 + 3 * (st - 2);
                    const int o1 = st == 1 ? 2 : 1;     // state 1 keeps 1 / N(t) between c0 and c1
                    R e0 = T::lift(__ldg(cv)), e1 = T::lift(__ldg(cv + o1)), e2 = T::lift(__ldg(cv + o1 + 1));
                    const double *ct = P.xp_ex_tan + (((size_t)xe * P.n_prod + pi) * EQ_MAX_RIGHTS + (st - 1)) * 3 * NT;
#pragma unroll
                    for (int k = 0; k < NT; ++k) {
                      e0.d[k] = __ldg(ct + k); e1.d[k] = __ldg(ct + NT + k); e2.d[k] = __ldg(ct + 2 * NT + k);
                    }
                    const R poly = e0 + ue * (e1 + ue * e2);
                    ve = poly * __ldg(op + 2);
                    ve.d[2] += val(poly) * __ldg(op + 7);
                  }
                  const XR tote = r_with_value(ve, group_sum(val(ve), base, A));
                  const int sete = (int)__ldg(pr + 1);
#pragma unroll
                  for (int s = 0; s < NS; ++s) if (s == sete) expo[s] = expo[s] + tote;
                  continue;
                }
              }
              if (xw != 0.0 && st > 0) {
                const double u = (Sv - __ldg(op + 5)) * __ldg(op + 6);
                const double c0 = st == 1 ? __ldg(op + 1) : __ldg(op + 16 + 3 * (st - 2));
                const double c1 = st == 1 ? __ldg(op + 3) : __ldg(op + 17 + 3 * (st - 2));
                const double c2 = st == 1 ? __ldg(op + 4) : __ldg(op + 18 + 3 * (st - 2));
                v = (c0 + u * (c1 + u * c2)) * __ldg(op + 2);
              }
              const double tot2 = group_sum(v, base, A);
              const int set2 = (int)__ldg(pr + 1);
#pragma unroll
              for (int s = 0; s < NS; ++s) if (s == set2) expo[s] += tot2;
              continue;
            }
            const double wgt = __ldg(P.prod_w + (size_t)pi * A + aa);
            XR vx = RealTraits<XR>::zero();
            if (wgt != 0.0) {
              // Black-Scholes value of the remaining option at (S_t, T - t), over the numeraire
              // (european_option.py:70-100, 123-145); evaluated on the lane that owns the asset
              const double ttm = __ldg(op + 1), K = __ldg(pr + 2), sign = __ldg(pr + 3);
              if constexpr (XT) {
                // the same closed form on duals: tangents through the spot, the volatility and the rate (drift,
                // discounting inside the formula, and the numeraire 1 / N(t): d invN / d r in op[7])
                const R Sr = spot_now();
                const R &sg = par[1], &rt = par[2];
                const R vol_t = sg * sqrt(ttm);
                const R d1 = (r_log(Sr / K) + (rt + 0.5 * sg * sg) * ttm) / vol_t, d2 = d1 - vol_t;
                const R disc = r_exp(-(rt * ttm)) * K;
                const R price = sign > 0.0 ? Sr * dual_ncdf(d1) - disc * dual_ncdf(d2)
                                           : disc * dual_ncdf(-d2) - Sr * dual_ncdf(-d1);
                vx = price * (wgt * __ldg(op + 2));
                vx.d[2] += wgt * val(price) * __ldg(op + 7);
              } else {
                const double sigma = val(par[1]), rate = val(par[2]);
                const double vol_t = sigma * sqrt(ttm);
                const double d1 = (log(Sv / K) + (rate + 0.5 * sigma * sigma) * ttm) / vol_t, d2 = d1 - vol_t;
                const double disc = K * exp(-rate * ttm);
                const double price = sign > 0.0 ? Sv * 0.5 * erfc(-d1 * 0.70710678118654752440) - disc * 0.5 * erfc(-d2 * 0.70710678118654752440)
                                                : disc * 0.5 * erfc(d2 * 0.70710678118654752440) - Sv * 0.5 * erfc(d1 * 0.70710678118654752440);
                vx = RealTraits<XR>::lift(wgt * price * __ldg(op + 2));
              }
            }
            // value: the group's total; tangents: the part flowing through this lane's asset
            const XR tot = r_with_value(vx, group_sum(val(vx), base, A));
            const int set = (int)__ldg(pr + 1);
#pragma unroll
            for (int s = 0; s < NS; ++s) if (s == set) expo[s] = expo[s] + tot;
          }
          if (P.expo_accum) {
            if (live && a == 0 && !pilot) {
#pragma unroll
              for (int s = 0; s < NS; ++s)
                if (s < P.n_sets) P.expo_accum[((size_t)s * P.n_expo + xe) * sh.n_paths + lpath] += val(expo[s]);
            }
            if constexpr (XT) {
              if (P.expo_accum_tan && live && !pilot) {
#pragma unroll
                for (int s = 0; s < NS; ++s)
                  if (s < P.n_sets) {
#pragma unroll
                    for (int k = 0; k < NT; ++k)
                      P.expo_accum_tan[((((size_t)s * P.n_expo + xe) * A + a) * NT + k) * sh.n_paths + lpath] += tan_of(expo[s], k);
                  }
              }
            }
            return;   // netting terms and metrics are applied once all launches of the book have added up
          }
#pragma unroll
          for (int s = 0; s < NS; ++s) {
#pragma unroll
            for (int l = EQ_MAX_LAG - 1; l > 0; --l) hist[s][l] = hist[s][l - 1];
            hist[s][0] = expo[s];
          }
        }
        if (P.expo_accum) return;
        if (m >= 0) {
          double vals[NVX];
          XR xpos[NS], xneg[NS];
#pragma unroll
          for (int s = 0; s < NS; ++s) {
            const bool coll = s < P.n_sets && (__ldg(P.set_flags + s) & 1);
            const double h = s < P.n_sets ? __ldg(P.set_threshold + s) : 0.0;
            const int lag = coll ? __ldg(P.set_lag + (size_t)s * P.n_metric + m) : -1;
            auto thr = [h](const XR &x) -> XR {    // netting_set.py:48-72
              return val(x) > h ? x - h : (val(x) < -h ? x + h : RealTraits<XR>::zero());
            };
            XR unsec;
            if (coll) {
              XR delayed = RealTraits<XR>::zero();
#pragma unroll
              for (int l = 0; l < EQ_MAX_LAG; ++l) if (l == lag) delayed = hist[s][l];
              unsec = hist[s][0] - thr(delayed);
            } else {
              unsec = thr(hist[s][0]);
            }
            xpos[s] = r_relu(unsec); xneg[s] = -r_relu(-unsec);
            const double pos = val(xpos[s]), neg = val(xneg[s]);
            if (KIND == MCRE_EQ_BS && P.has_cir && m < P.n_metric - 1 && s < P.n_sets && __ldg(P.set_cva + s)) {
              // cva_metric.py:62-100: relu(E_k) S(0, t_k) (1 - S(t_k, t_k+1 | y_k)), S(0, t) = exp(-logB_lambda)
              const double Ck = __ldg(P.cva_coef + 2 * m), Bk = __ldg(P.cva_coef + 2 * m + 1);
              cva_path[s] = fma(pos, exp(-clogB) * (1.0 - Ck * exp(-Bk * cy)), cva_path[s]);
            }
            const int sb = expo_base + m * NVX + s * 4;
            if (pilot) { if (threadIdx.x == 0) { shift[sb + 0] = pos; shift[sb + 2] = neg; } }
            const double dp = pos - (pilot ? 0.0 : shift[sb + 0]), dn = neg - (pilot ? 0.0 : shift[sb + 2]);
            const double keep = (live && a == 0) ? 1.0 : 0.0;
            vals[s * 4 + 0] = keep * dp; vals[s * 4 + 1] = keep * dp * dp;
            vals[s * 4 + 2] = keep * dn; vals[s * 4 + 3] = keep * dn * dn;
            if ((P.acc_flags & MCRE_ACC_SPILL) && live && a == 0 && s < P.n_sets && !pilot)
              spill[((size_t)s * P.n_metric + m) * sh.n_paths + lpath] = val(unsec);
          }
          if (!pilot) block_accumulate<NVX>(vals, acc, expo_base + m * NVX, stage, NVMAX, parity);
          if constexpr (XT) {
            if (!pilot) {
              for (int ap = 0; ap < A; ++ap) {
                const double keep = (live && a == ap) ? 1.0 : 0.0;
                double tv[NVXT];
#pragma unroll
                for (int s = 0; s < NS; ++s)
#pragma unroll
                  for (int k = 0; k < NT; ++k) {
                    tv[(s * 2 + 0) * NT + k] = keep * tan_of(xpos[s], k);
                    tv[(s * 2 + 1) * NT + k] = keep * tan_of(xneg[s], k);
                  }
                block_accumulate<NVXT>(tv, acc, xt_base + (m * A + ap) * NVXT, stage, NVMAX, parity);
              }
            }
          }
        }
      };

      auto eval_date = [&](int di) {
        const int e0 = __ldg(P.date_ev_off + di), e1 = __ldg(P.date_ev_off + di + 1);
        if (e0 == e1) return;
        const R S = spot_now();
        for (int e = e0; e < e1; ++e) {
          const int pi = __ldg(P.ev_prod + e), ef = __ldg(P.ev_flags + e);
          const double *pr = P.prod + (size_t)pi * EQ_PR;
          const int kind = (int)__ldg(pr + 0), set = (int)__ldg(pr + 1), pflags = (int)__ldg(pr + 6);
          const double strike = __ldg(pr + 2), sign = __ldg(pr + 3);
          const double wgt = __ldg(P.prod_w + (size_t)pi * A + aa);
          // composite underlying: arithmetic and / or geometric weighted basket of the group's spots
          const bool need_geo = (kind == EQ_BASKET) && (pflags & 3);
          const bool need_ari = !(kind == EQ_BASKET && (pflags & 1));
          R U = T::zero(), G = T::zero();
          if (need_ari) {
            const R term = S * wgt;
            U = r_with_value(term, group_sum(val(term), base, A));
          }
          if (need_geo) {
            const R term = r_log(S + 1e-10) * wgt;      // basket_option.py:62-66
            G = r_exp(r_with_value(term, group_sum(val(term), base, A)));
          }
          const int slot = (int)__ldg(pr + 14);
          if (ef & EQ_EV_EXERCISE) {
            // Bermudan / American exercise date (bermudan_option.py:93-131): exercise iff the
            // immediate value beats the regressed continuation value (hard indicator) and the right
            // is still alive; tracker a of the product's slot is the alive flag.
            // FlexiCall (flexicall.py:56-160): tracker a holds the number of rights left (state s); a path in
            // state s > 0 exercises iff immediate + continuation(s - 1) > continuation(s), strike per date.
            const double *ed = P.ev_data + (size_t)e * EQ_EVD;
            const double xw = __ldg(P.prod_x + (size_t)pi * A + aa);
            const double X = group_sum(val(S) * xw, base, A);          // explanatory spot
            const double u = (X - __ldg(ed + 3)) * __ldg(ed + 4);
            const bool lastd = __ldg(ed + 7) != 0.0;                   // no continuation after the last date
            auto cont_of = [&](int st) -> double {
              if (lastd || st <= 0) return 0.0;
              const double *c = st == 1 ? ed : ed + 16 + 3 * (st - 2);
              return __ldg(c + 0) + u * (__ldg(c + 1) + u * __ldg(c + 2));
            };
            const R imm = option_payoff(U, __ldg(ed + 14), sign);
#pragma unroll
            MCRE_TRK_FOR(k, slot) {
              const int st = (int)val(trk_a[k]);
              if (st > 0 && val(imm) + cont_of(st - 1) > cont_of(st)) {
                trk_a[k] = T::lift((double)(st - 1));
#pragma unroll
                for (int s = 0; s < NS; ++s)
                  if (s == set) { cf[s] = cf[s] + imm * __ldg(ed + 5); numtan[s] += val(imm) * __ldg(ed + 6); }
              }
            }
            continue;
          }
          if (ef & EQ_EV_OBSERVE) {
#pragma unroll
            MCRE_TRK_FOR(k, slot) {
              if (kind == EQ_ASIAN) {
                const R x = (pflags & 1) ? r_log(U + 1e-10) : U;     // asian_option.py:51-69
                trk_a[k] = (ef & EQ_EV_FIRST) ? x : trk_a[k] + x;
              } else {                                                // running max / min
                if ((ef & EQ_EV_FIRST) || val(U) > val(trk_a[k])) trk_a[k] = U;
                if ((ef & EQ_EV_FIRST) || val(U) < val(trk_b[k])) trk_b[k] = U;
                if constexpr (NT == 0) {
                  if (pflags & 4) {
                    // Brownian bridge between monitoring dates (barrier_option.py:138-222): crossing probability
                    // exp(coef ln(S_prev / B) ln(S / B)), coef = -2 / (sigma^2 maturity / n_obs), against one
                    // uniform per (path, interval); fuzzy indicator eps 0.05 like the rest of the product
                    const double *ed = P.ev_data + (size_t)e * EQ_EVD;   // [0] Philox block, [1] coef, [2] interval
                    const double Uv = val(U);
                    if (ef & EQ_EV_FIRST) { trk_d[k] = 1.0; trk_e[k] = 1.0; }
                    else {
                      double ua, ub;
                      if (P.bridge_u) {
                        const size_t per = (size_t)rng.n_total * P.bridge_stride;
                        const double *bu = P.bridge_u + (size_t)slot * 2 * per + (size_t)gpath * P.bridge_stride + (int)__ldg(ed + 2);
                        ua = bu[0]; ub = bu[per];
                      } else {
                        ns.uniform_pair_kind((uint32_t)__ldg(ed + 0), 2u, ua, ub);
                      }
                      const double coef = __ldg(ed + 1), prev = trk_c[k];
                      const double b1 = __ldg(pr + 9);
                      const double p1 = exp(coef * log(prev / b1) * log(Uv / b1));
                      trk_d[k] *= 1.0 - r_fuzzy(p1 - ua, true, 0.05);
                      if ((int)__ldg(pr + 12) > 0) {
                        const double b2 = __ldg(pr + 11);
                        const double p2 = exp(coef * log(prev / b2) * log(Uv / b2));
                        trk_e[k] *= 1.0 - r_fuzzy(p2 - ub, true, 0.05);
                      }
                    }
                    trk_c[k] = Uv;
                  }
                }
              }
            }
            if constexpr (NT > 0 && KIND == MCRE_EQ_BS) {
              if (kind == EQ_BARRIER && (pflags & 4) && slot >= 0 && slot < NTRK) {
                // the same crossing probabilities on duals: through both monitored spots and, in coef = -2 / (sigma^2
                // maturity / n_obs), through the volatility (lane parameter 1): d coef / d sigma = -2 coef / sigma
                const double *ed = P.ev_data + (size_t)e * EQ_EVD;
                if (ef & EQ_EV_FIRST) { brg_d[slot] = T::lift(1.0); brg_e[slot] = T::lift(1.0); }
                else {
                  double ua, ub;
                  if (P.bridge_u) {
                    const size_t per = (size_t)rng.n_total * P.bridge_stride;
                    const double *bu = P.bridge_u + (size_t)slot * 2 * per + (size_t)gpath * P.bridge_stride + (int)__ldg(ed + 2);
                    ua = bu[0]; ub = bu[per];
                  } else {
                    ns.uniform_pair_kind((uint32_t)__ldg(ed + 0), 2u, ua, ub);
                  }
                  const R coef = bridge_coef(__ldg(ed + 1), par[1]);
                  const R prev = brg_c[slot];
                  const double b1 = __ldg(pr + 9);
                  const R p1 = r_exp(coef * r_log(prev / b1) * r_log(U / b1));
                  brg_d[slot] = brg_d[slot] * (1.0 - r_fuzzy(p1 - ua, true, 0.05));
                  if ((int)__ldg(pr + 12) > 0) {
                    const double b2 = __ldg(pr + 11);
                    const R p2 = r_exp(coef * r_log(prev / b2) * r_log(U / b2));
                    brg_e[slot] = brg_e[slot] * (1.0 - r_fuzzy(p2 - ub, true, 0.05));
                  }
                }
                brg_c[slot] = U;
              }
            }
          }
          if (!(ef & EQ_EV_PAY)) continue;
          R pay;
          if (kind == EQ_EUROPEAN) {
            pay = option_payoff(U, strike, sign);                     // european_option.py:45-68
          } else if (kind == EQ_BINARY) {
            const R ind = r_fuzzy(U - strike, true, 1.0);             // binary_option.py:37-42
            pay = (sign > 0.0 ? ind : 1.0 - ind) * __ldg(pr + 8);
          } else if (kind == EQ_BASKET) {
            // control variate (basket_option.py:72-78): classical - geometric (+ closed form, added by the host)
            pay = option_payoff((pflags & 1) ? G : U, strike, sign);
            if (pflags & 2) pay = pay - option_payoff(G, strike, sign) + __ldg(pr + 7);
          } else if (kind == EQ_ASIAN) {
            const double inv_n = 1.0 / __ldg(pr + 13);
            R avg = T::zero();
#pragma unroll
            MCRE_TRK_FOR(k, slot) avg = trk_a[k] * inv_n;
            if (pflags & 1) avg = r_exp(avg);
            pay = option_payoff(avg, strike, sign);
          } else {
            R mx = T::zero(), mn = T::zero();
#pragma unroll
            MCRE_TRK_FOR(k, slot) { mx = trk_a[k]; mn = trk_b[k]; }
            pay = option_payoff(U, strike, sign) * barrier_factor(mx, mn, __ldg(pr + 9), (int)__ldg(pr + 10));
            const int bt2 = (int)__ldg(pr + 12);
            if (bt2 > 0) pay = pay * barrier_factor(mx, mn, __ldg(pr + 11), bt2);
            if constexpr (NT == 0) {
              if (pflags & 4) {
                // knock-out: also no crossing between the dates; knock-in: (1 - indicator)(1 - no-hit)
                double nh1 = 1.0, nh2 = 1.0;
                MCRE_TRK_FOR(k, slot) { nh1 = trk_d[k]; nh2 = trk_e[k]; }
                auto bridged = [&](double barrier, int bt, double nh) -> double {
                  const double out = val(barrier_factor(mx, mn, barrier, bt <= 2 ? bt : bt - 2));   // the "out" indicator
                  return bt <= 2 ? out * nh : (1.0 - out) * (1.0 - nh);
                };
                double f = bridged(__ldg(pr + 9), (int)__ldg(pr + 10), nh1);
                if (bt2 > 0) f *= bridged(__ldg(pr + 11), bt2, nh2);
                pay = option_payoff(U, strike, sign) * f;
              }
            }
            if constexpr (NT > 0 && KIND == MCRE_EQ_BS) {
              if ((pflags & 4) && slot >= 0 && slot < NTRK) {
                auto bridged = [&](double barrier, int bt, const R &nh) -> R {
                  const R out = barrier_factor(mx, mn, barrier, bt <= 2 ? bt : bt - 2);
                  return bt <= 2 ? out * nh : (1.0 - out) * (1.0 - nh);
                };
                R f = bridged(__ldg(pr + 9), (int)__ldg(pr + 10), brg_d[slot]);
                if (bt2 > 0) f = f * bridged(__ldg(pr + 11), bt2, brg_e[slot]);
                pay = option_payoff(U, strike, sign) * f;
              }
            }
          }
          const double invN = __ldg(pr + 4), dinvN = __ldg(pr + 5);
          if (P.ps_cf && live && a == 0) P.ps_cf[(size_t)pi * sh.n_paths + lpath] = (float)(val(pay) * invN);
          if constexpr (NT > 0) {
            // tangents of the deflated cashflow with respect to the parameters of the product's asset, written by
            // the lane that owns it (single-asset products; index 2 = the rate also carries the numeraire term)
            if (P.ps_dcf && live && __ldg(P.prod_x + (size_t)pi * A + aa) != 0.0) {
#pragma unroll
              for (int k = 0; k < NT; ++k)
                P.ps_dcf[((size_t)pi * NT + k) * sh.n_paths + lpath] = tan_of(pay, k) * invN + (k == 2 ? val(pay) * dinvN : 0.0);
            }
          }
#pragma unroll
          for (int s = 0; s < NS; ++s)
            if (s == set) {
              if constexpr (NT == 9) {
                // second-order build: the numeraire 1 / N(T) = exp(-r T) as a function of the lane's rate (the host admits
                // books whose assets share the numeraire's rate parameter), so the header's separate rate term stays 0
                // (every lane of the group holds the payoff's value, the product's own lane its derivatives: the
                // numeraire's derivatives ride with that lane alone)
                R nrm = T::lift(invN);
                if (wgt != 0.0) { nrm.d[2] = dinvN; nrm.h[5] = dinvN * dinvN / invN; }
                cf[s] = cf[s] + pay * nrm;
              } else {
                cf[s] = cf[s] + pay * invN; numtan[s] += val(pay) * dinvN;
              }
            }
        }
      };

      for (int di = 0; di < P.n_pre_dates; ++di) { eval_date(di); eval_exposure(di); }
      for (int is = 0; is < P.n_sub; ++is) {
        const double dt = __ldg(P.step_dt + is), sq = __ldg(P.step_sq + is);
        // ---- independent draws of this lane's noise columns -----------------------------
        double z0 = 0.0, z1 = 0.0, u = 0.5;
        if (rng.mode == MCRE_RNG_INJECT) {
          const double *zp = rng.z + ((size_t)is * rng.n_total + gpath) * d;
          z0 = zp[c0];
          if (c1 >= 0) z1 = zp[c1];
          if (KIND == MCRE_EQ_HESTON && ALT == 1) u = rng.u[((size_t)is * rng.n_total + gpath) * P.n_uniform + uidx];
        } else {
          const uint32_t n0 = (uint32_t)(is * d + c0);
          double p0, p1;
          ns.pair(n0 >> 1, p0, p1);
          z0 = (n0 & 1u) ? p1 : p0;
          if (c1 >= 0) {
            const uint32_t n1 = (uint32_t)(is * d + c1);
            if ((n1 >> 1) == (n0 >> 1)) z1 = (n1 & 1u) ? p1 : p0;
            else { ns.pair(n1 >> 1, p0, p1); z1 = (n1 & 1u) ? p1 : p0; }
          }
          if (KIND == MCRE_EQ_HESTON && ALT == 1) {
            // uniform #(asset * n_sub + step): consecutive steps of an asset share a Philox block
            const uint32_t m = (uint32_t)(uidx * P.n_sub_total + is);
            if (is == 0 || (m & 1u) == 0u) ns.uniform_pair(m >> 1, u_even, u_odd);
            u = (m & 1u) ? u_odd : u_even;
          }
        }
        // ---- correlate: w = z @ L^T -----------------------------------------------------
        R w0 = T::lift(z0), w1 = T::lift(z1);
        if (P.corr_mode == 2 && P.sp_n > 0) {
          double a0 = 0.0;
#pragma unroll
          for (int k = 0; k < EQ_SPNZ; ++k) {
            if (k < P.sp_n) {
              const double zj = __shfl_sync(0xffffffffu, (sps[k] & 1) ? z1 : z0, (base + (sps[k] >> 1)) & 31);
              a0 = fma(spc[k], zj, a0);
            }
          }
          w0 = T::lift(a0);      // w1 = z1: identity row
        } else if (P.corr_mode == 2) {
          const double *L = P.chol + (size_t)__ldg(P.step_chol + is) * d * d;
          double a0 = 0.0, a1 = 0.0;
          for (int j = 0; j < d; ++j) {
            const int src = (base + __ldg(P.col_asset + j)) & 31;
            const double zj = __shfl_sync(0xffffffffu, __ldg(P.col_elem + j) ? z1 : z0, src);
            a0 += __ldg(L + c0 * d + j) * zj;
            if (c1 >= 0) a1 += __ldg(L + c1 * d + j) * zj;
          }
          w0 = T::lift(a0); w1 = T::lift(a1);
        } else if (P.corr_mode == 1) {
          const double *L = P.chol_dual + (size_t)__ldg(P.step_chol + is) * 4 * (NT + 1);
          w0 = T::load(L, 0) * z0;
          w1 = T::load(L, 2) * z0 + T::load(L, 3) * z1;
        }
        // ---- model step ------------------------------------------------------------------
        if constexpr (KIND == MCRE_EQ_BS) {
          const R &sigma = par[1], &rate = par[2];
          if (ALT == 1) s0 = s0 * r_exp(rate * dt + (sigma * (sq * w0) - 0.5 * dt * sigma * sigma));  // black_scholes.py:44-67
          else s0 = s0 + (rate * s0 * dt + sigma * s0 * sq * w0);                                     // :69-85
        } else if constexpr (KIND == MCRE_EQ_HESTON) {
          if (ALT == 1) {
            if (dt != qe.dt) heston_qe_prepare<R>(par[1], par[2], par[3], par[4], par[5], dt, qe);   // uniform: dt is a plan scalar
            heston_qe_step_c<R>(qe, par[5], smooth, val(w0), val(w1), u, s0, s1);
          }
          else heston_euler_step<R>(par[1], par[2], par[4], par[5], dt, sq, w0, w1, s0, s1);
        } else {
          const R &kappa = par[1], &ss = par[2], &mu = par[3], &sl = par[4];
          if (ALT == 1) {            // schwartz_two_factor.py:147-171 (w = covariance-scaled)
            const R xm = fabs(val(kappa)) <= 1e-12 ? s0 : s0 * r_exp(-(kappa * dt));
            s0 = xm + w0;
            s1 = s1 + mu * dt + w1;
          } else {                   // :173-196
            s0 = s0 - kappa * s0 * dt + ss * sq * w0;
            s1 = s1 + mu * dt + sl * sq * w1;
          }
          logF = __ldg(P.step_aux + (size_t)is * A + aa);
        }
        if (KIND == MCRE_EQ_BS && P.has_cir) {
          // correlated credit normal: its own draw plus the equity draws of the group (row of the joint factor)
          double zc;
          if (rng.mode == MCRE_RNG_INJECT) zc = rng.z[((size_t)is * rng.n_total + gpath) * d + P.cir_col];
          else {
            const uint32_t nc = (uint32_t)(is * d + P.cir_col);
            double p0, p1;
            ns.pair(nc >> 1, p0, p1);
            zc = (nc & 1u) ? p1 : p0;
          }
          double wc = __ldg(P.cir_row + P.cir_col) * zc;
          for (int j = 0; j < d; ++j) {
            if (j == P.cir_col) continue;
            const double zj = __shfl_sync(0xffffffffu, __ldg(P.col_elem + j) ? z1 : z0, (base + __ldg(P.col_asset + j)) & 31);
            wc = fma(__ldg(P.cir_row + j), zj, wc);
          }
          if (P.cir_det) {
            clogB += __ldg(P.step_cir + 2 * is) * dt;
            cy = __ldg(P.step_cir + 2 * is + 1);
          } else {      // Euler with full truncation (cirpp.py:174-198)
            const double yn = cy + P.cir_kappa * (P.cir_theta - cy) * dt + P.cir_sigma * sqrt(fmax(cy, 0.0)) * sq * wc;
            clogB += (cy + __ldg(P.step_cir + 2 * is)) * dt;
            cy = fmax(yn, 1e-12);
          }
        }
        const int di = __ldg(P.step_date + is);
        if (di >= 0) { eval_date(di); eval_exposure(di); }
      }

      // ---- per-path totals -> block accumulators -------------------------------------------
      const double keep1 = (live && a == 0) ? 1.0 : 0.0;
      {
        double vals[NVH];
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          if (pilot) { if (threadIdx.x == 0) shift[s] = val(cf[s]); }
          if (P.pv_accum && !pilot && live && a == 0 && s < P.n_sets) P.pv_accum[(size_t)s * sh.n_paths + lpath] += val(cf[s]);
          const double x = val(cf[s]) - (pilot ? 0.0 : shift[s]);
          vals[s * 3 + 0] = keep1 * x; vals[s * 3 + 1] = keep1 * x * x; vals[s * 3 + 2] = keep1 * numtan[s];
        }
        if (!pilot) block_accumulate<NVH>(vals, acc, 0, stage, NVMAX, parity);
      }
      if (KIND == MCRE_EQ_BS && P.has_cir) {
        double cv[NS * 2];
#pragma unroll
        for (int s = 0; s < NS; ++s) {
          const double c = cva_path[s] * P.lgd;
          if (pilot) { if (threadIdx.x == 0) shift[cva_base + 2 * s] = c; }
          const double x = c - (pilot ? 0.0 : shift[cva_base + 2 * s]);
          cv[2 * s] = keep1 * x; cv[2 * s + 1] = keep1 * x * x;
        }
        if (!pilot) block_accumulate<NS * 2>(cv, acc, cva_base, stage, NVMAX, parity);
      }
      if (NT > 0 && !pilot) {
        for (int ap = 0; ap < A; ++ap) {
          const double keep = (live && a == ap) ? 1.0 : 0.0;
          double tv[NVT];
#pragma unroll
          for (int s = 0; s < NS; ++s)
#pragma unroll
            for (int k = 0; k < NT; ++k) tv[s * NT + k] = keep * tan_of(cf[s], k);
          block_accumulate<NVT>(tv, acc, NS * 3 + ap * NS * NT, stage, NVMAX, parity);
        }
      }
      if (pilot) return;
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

struct mcre_eq_plan {
  EqDev d;
  int nt = 0;
  DevArena arena;   // all plan tables live in one device allocation
  DevArray<double> asset_par, step_dt, step_sq, step_aux, init_aux, chol, chol_dual, prod, prod_w, ev_data, prod_x;
  DevArray<int> asset_noise, asset_uniform, col_asset, col_elem, step_date, step_chol, date_ev_off, ev_prod, ev_flags;
  DevArray<int> date_expo, date_metric, set_flags, set_lag, sp_src, xact_off, xact;
  DevArray<double> xp, set_threshold, sp_coef;
  double *xp_tan = nullptr;   // own allocation (set after mcre_eq_create)
  double *xp_ex_tan = nullptr;   // own allocation (mcre_eq_set_exercise_exposure_coef_tangents)
  double *credit = nullptr;   // own allocation (mcre_eq_set_credit): step_cir, cir_row, cva_coef, set_cva
  bool has_proxy = false;     // some exposure is a regression proxy (type 2)
  bool has_exercise_expo = false;   // some exposure is an exercise product's continuation value (type 3)
};

extern "C" int mcre_eq_create(const mcre_eq_desc *c, mcre_eq_plan **out) {
  if (!c || !out) return fail(-1, "null argument%s", "");
  if (c->n_assets < 1 || c->n_assets > 32) return fail(-1, "eq: 1..32 assets per path group%s", "");
  if (c->n_sets < 1 || c->n_sets > MCRE_EQ_MAX_SETS) return fail(-1, "eq: n_sets out of range%s", "");
  const int np = c->kind == MCRE_EQ_BS ? 3 : c->kind == MCRE_EQ_HESTON ? 7 : c->kind == MCRE_EQ_SCHWARTZ ? 6 : -1;
  if (np < 0) return fail(-1, "eq: unknown model kind%s", "");
  const bool second = c->kind == MCRE_EQ_BS && c->nt == 9;   // value + 3 first + 6 second derivatives per lane (Dual2<3>)
  if (c->nt != 0 && c->nt != np && !second)
    return fail(-1, "eq: nt must be 0, the model's parameter count, or 9 (second order, Black-Scholes)%s", "");
  if (second && c->n_expo > 0)
    return fail(-4, "eq: the second-order build carries present values only%s", "");
  if (c->nt != 0 && c->n_sets > 2) return fail(-3, "eq: at most 2 netting sets per launch when tangents are on%s", "");
  if (c->nt != 0 && c->n_expo > 0) {
    if (!eq_kind_has_exposure_tangents(c->kind))
      return fail(-4, "eq: sensitivities of exposure profiles need a Black-Scholes or Heston model%s", "");
    for (size_t i = 0; i < (size_t)c->n_expo * c->n_prod; ++i)
      if (c->xp[i * EQ_XP] > 3.0)
        return fail(-4, "eq: unknown exposure type%s", "");
  }
  if (c->corr_mode == 1 && (c->n_assets != 1 || c->noise_dim != 2))
    return fail(-1, "eq: dual Cholesky needs one asset with two noise sources%s", "");
  const bool scheme_ok = (c->kind == MCRE_EQ_HESTON) ? (c->scheme == MCRE_SCHEME_EULER || c->scheme == MCRE_SCHEME_QE)
                                                     : (c->scheme == MCRE_SCHEME_EULER || c->scheme == MCRE_SCHEME_ANALYTICAL);
  if (!scheme_ok) return fail(-1, "eq: scheme not defined for this model%s", "");
  for (int p = 0; p < c->n_prod; ++p) {
    const int slot = (int)c->prod[(size_t)p * EQ_PR + 14], kind = (int)c->prod[(size_t)p * EQ_PR];
    if ((kind == EQ_ASIAN || kind == EQ_BARRIER || kind == EQ_EXERCISE) && (slot < 0 || slot >= eq_ntrk(c->nt)))
      return fail(-3, "eq: too many path-dependent / exercise products per launch (64, or 2 with tangents)%s", "");
    if (kind == EQ_EXERCISE && (!c->ev_data || !c->prod_x)) return fail(-1, "eq: exercise product without event data%s", "");
    const int set = (int)c->prod[(size_t)p * EQ_PR + 1];
    if (set < 0 || set >= c->n_sets) return fail(-1, "eq: product set index out of range%s", "");
  }
  mcre_eq_plan *p = new mcre_eq_plan();
  ArenaScope arena_scope(&p->arena);
  p->nt = c->nt;
  for (size_t i = 0; c->n_expo > 0 && i < (size_t)c->n_expo * c->n_prod; ++i) {
    p->has_proxy = p->has_proxy || c->xp[i * EQ_XP] == 2.0;
    p->has_exercise_expo = p->has_exercise_expo || c->xp[i * EQ_XP] == 3.0;
  }
  const int A = c->n_assets, d = c->noise_dim, n_ev = c->date_ev_off[c->n_dates];
  int rc = 0;
#define UP(field, host, count) if (!rc) rc = p->field.upload(host, (size_t)(count))
  UP(asset_par, c->asset_par, A * EQ_PAR); UP(asset_noise, c->asset_noise, A * 2); UP(asset_uniform, c->asset_uniform, A);
  UP(col_asset, c->col_asset, d); UP(col_elem, c->col_elem, d);
  UP(step_dt, c->step_dt, c->n_sub); UP(step_sq, c->step_sq, c->n_sub);
  UP(step_date, c->step_date, c->n_sub); UP(step_chol, c->step_chol, c->n_sub);
  UP(step_aux, c->step_aux, (size_t)c->n_sub * A); UP(init_aux, c->init_aux, A);
  UP(chol, c->chol, c->corr_mode == 2 ? (size_t)c->n_chol * d * d : 0);
  UP(chol_dual, c->chol_dual, c->corr_mode == 1 ? (size_t)c->n_chol * 4 * (c->nt + 1) : 0);
  UP(date_ev_off, c->date_ev_off, c->n_dates + 1); UP(ev_prod, c->ev_prod, n_ev); UP(ev_flags, c->ev_flags, n_ev);
  UP(prod, c->prod, (size_t)c->n_prod * EQ_PR); UP(prod_w, c->prod_w, (size_t)c->n_prod * A);
  UP(ev_data, c->ev_data, c->ev_data ? (size_t)n_ev * EQ_EVD : 0); UP(prod_x, c->prod_x, c->prod_x ? (size_t)c->n_prod * A : 0);
  if (c->n_expo > 0) {
    UP(date_expo, c->date_expo, c->n_dates); UP(date_metric, c->date_metric, c->n_dates);
    UP(xp, c->xp, (size_t)c->n_expo * c->n_prod * EQ_XP);
    UP(set_threshold, c->set_threshold, c->n_sets); UP(set_flags, c->set_flags, c->n_sets);
    UP(set_lag, c->set_lag, (size_t)c->n_sets * c->n_metric);
    // products with an exposure per date (see EqDev)
    std::vector<int> off(c->n_expo + 1, 0), act;
    for (int e = 0; e < c->n_expo; ++e) {
      for (int pi = 0; pi < c->n_prod; ++pi)
        if (c->xp[((size_t)e * c->n_prod + pi) * EQ_XP] != 0.0) act.push_back(pi);
      off[e + 1] = (int)act.size();
    }
    if (act.empty()) act.push_back(0);
    UP(xact_off, off.data(), off.size()); UP(xact, act.data(), act.size());
  }
  // sparse rows of the joint Cholesky factor (see EqDev)
  int sp_n = 0;
  if (c->corr_mode == 2 && c->n_chol == 1 && c->chol) {
    std::vector<double> coef((size_t)A * EQ_SPNZ, 0.0);
    std::vector<int> src((size_t)A * EQ_SPNZ, 0);
    bool ok = true;
    for (int a = 0; a < A && ok; ++a) {
      const int r0 = c->asset_noise[a * 2], r1 = c->asset_noise[a * 2 + 1];
      if (r1 >= 0)
        for (int j = 0; j < d; ++j) ok = ok && c->chol[(size_t)r1 * d + j] == (j == r1 ? 1.0 : 0.0);
      int n = 0;
      for (int j = 0; j < d && ok; ++j) {
        const double v = c->chol[(size_t)r0 * d + j];
        if (v == 0.0) continue;
        if (n == EQ_SPNZ) { ok = false; break; }
        coef[(size_t)a * EQ_SPNZ + n] = v;
        src[(size_t)a * EQ_SPNZ + n] = (c->col_asset[j] << 1) | (c->col_elem[j] & 1);
        ++n;
      }
      if (n > sp_n) sp_n = n;
    }
    if (!ok) sp_n = 0;
    if (sp_n > 0) { UP(sp_coef, coef.data(), coef.size()); UP(sp_src, src.data(), src.size()); }
  }
#undef UP
  if (!rc) rc = p->arena.commit();
  if (rc) { mcre_eq_destroy(p); return rc; }
  EqDev &D = p->d;
  D.sp_n = sp_n; D.sp_coef = p->sp_coef.p; D.sp_src = p->sp_src.p; D.n_sub_total = c->n_sub;
  D.xp_tan = nullptr; D.xp_ex_tan = nullptr; D.ps_dx = nullptr; D.ps_dcf = nullptr;
  D.has_cir = 0; D.cir_det = 0; D.cir_col = 0; D.cir_kappa = D.cir_theta = D.cir_sigma = D.cir_y0 = D.lgd = 0.0;
  D.step_cir = D.cir_row = D.cva_coef = nullptr; D.set_cva = nullptr; D.cva_w = nullptr;
  D.ps_x = nullptr; D.ps_cf = nullptr; D.pv_accum = nullptr; D.bridge_u = nullptr; D.bridge_stride = 0; D.expo_accum = nullptr; D.expo_accum_tan = nullptr;
  D.kind = c->kind; D.scheme = c->scheme; D.smoothing = c->smoothing; D.n_assets = A; D.noise_dim = d;
  D.n_uniform = c->n_uniform > 0 ? c->n_uniform : 1;
  D.asset_par = p->asset_par.p; D.asset_noise = p->asset_noise.p; D.asset_uniform = p->asset_uniform.p;
  D.col_asset = p->col_asset.p; D.col_elem = p->col_elem.p;
  D.n_sub = c->n_sub; D.n_dates = c->n_dates; D.n_pre_dates = c->n_pre_dates;
  D.step_dt = p->step_dt.p; D.step_sq = p->step_sq.p; D.step_date = p->step_date.p; D.step_chol = p->step_chol.p;
  D.step_aux = p->step_aux.p; D.init_aux = p->init_aux.p;
  D.corr_mode = c->corr_mode; D.chol = p->chol.p; D.chol_dual = p->chol_dual.p;
  D.date_ev_off = p->date_ev_off.p; D.ev_prod = p->ev_prod.p; D.ev_flags = p->ev_flags.p;
  D.n_prod = c->n_prod; D.prod = p->prod.p; D.prod_w = p->prod_w.p; D.n_sets = c->n_sets;
  D.ev_data = p->ev_data.p; D.prod_x = p->prod_x.p;
  D.n_expo = c->n_expo; D.n_metric = c->n_expo > 0 ? c->n_metric : 0; D.acc_flags = c->acc_flags;
  D.date_expo = p->date_expo.p; D.date_metric = p->date_metric.p; D.xp = p->xp.p;
  D.set_threshold = p->set_threshold.p; D.set_flags = p->set_flags.p; D.set_lag = p->set_lag.p;
  D.xact_off = p->xact_off.p; D.xact = p->xact.p;
  *out = p;
  return 0;
}

extern "C" void mcre_eq_destroy(mcre_eq_plan *p) {
  if (!p) return;
  p->asset_par.release(); p->step_dt.release(); p->step_sq.release(); p->step_aux.release(); p->init_aux.release();
  p->chol.release(); p->chol_dual.release(); p->prod.release(); p->prod_w.release(); p->asset_noise.release();
  p->asset_uniform.release(); p->col_asset.release(); p->col_elem.release(); p->step_date.release();
  p->step_chol.release(); p->date_ev_off.release(); p->ev_prod.release(); p->ev_flags.release();
  p->ev_data.release(); p->prod_x.release();
  p->date_expo.release(); p->date_metric.release(); p->set_flags.release(); p->set_lag.release();
  p->xp.release(); p->set_threshold.release(); p->sp_coef.release(); p->sp_src.release();
  p->xact_off.release(); p->xact.release();
  p->arena.release();
  if (p->xp_tan) cudaFree(p->xp_tan);
  if (p->xp_ex_tan) cudaFree(p->xp_ex_tan);
  if (p->credit) cudaFree(p->credit);
  delete p;
}

extern "C" int mcre_eq_set_exposure_coef_tangents(mcre_eq_plan *p, const double *xp_tan) {
  if (!p || !xp_tan) return fail(-1, "null argument%s", "");
  if (p->nt <= 0 || !eq_kind_has_exposure_tangents(p->d.kind) || p->d.n_expo <= 0)
    return fail(-4, "eq: coefficient tangents need a Black-Scholes / Heston plan with tangents and exposure dates%s", "");
  const size_t n = (size_t)p->d.n_expo * p->d.n_prod * 3 * p->nt;
  if (!p->xp_tan) MCRE_CUDA(cudaMalloc((void **)&p->xp_tan, n * sizeof(double)));
  MCRE_CUDA(cudaMemcpy(p->xp_tan, xp_tan, n * sizeof(double), cudaMemcpyHostToDevice));
  p->d.xp_tan = p->xp_tan;
  return 0;
}

extern "C" int mcre_eq_set_exercise_exposure_coef_tangents(mcre_eq_plan *p, const double *tan) {
  if (!p || !tan) return fail(-1, "null argument%s", "");
  if (p->nt <= 0 || !eq_kind_has_exposure_tangents(p->d.kind) || p->d.n_expo <= 0)
    return fail(-4, "eq: coefficient tangents need a Black-Scholes / Heston plan with tangents and exposure dates%s", "");
  const size_t n = (size_t)p->d.n_expo * p->d.n_prod * EQ_MAX_RIGHTS * 3 * p->nt;
  if (!p->xp_ex_tan) MCRE_CUDA(cudaMalloc((void **)&p->xp_ex_tan, n * sizeof(double)));
  MCRE_CUDA(cudaMemcpy(p->xp_ex_tan, tan, n * sizeof(double), cudaMemcpyHostToDevice));
  p->d.xp_ex_tan = p->xp_ex_tan;
  return 0;
}

extern "C" int mcre_eq_set_credit(mcre_eq_plan *p, const mcre_eq_credit *c) {
  if (!p || !c || !c->step_cir || !c->chol_row || !c->set_cva) return fail(-1, "null argument%s", "");
  if (p->nt != 0) return fail(-4, "eq: sensitivities of hybrid equity + credit runs are not implemented%s", "");
  if (p->d.kind != MCRE_EQ_BS) return fail(-4, "eq: the credit factor rides with Black-Scholes market models%s", "");
  if (c->noise_col < 0 || c->noise_col >= p->d.noise_dim) return fail(-1, "eq: credit noise column out of range%s", "");
  if (p->d.n_metric > 0 && !c->cva_coef) return fail(-1, "eq: credit factor without CVA coefficients%s", "");
  const EqDev &D0 = p->d;
  const size_t n_step = (size_t)2 * (D0.n_sub > 0 ? D0.n_sub : 1), n_row = (size_t)D0.noise_dim,
               n_cva = (size_t)2 * (D0.n_metric > 0 ? D0.n_metric : 1), n_set = (size_t)D0.n_sets;
  std::vector<double> host(n_step + n_row + n_cva + n_set, 0.0);   // set flags ride as doubles' storage (ints behind)
  for (size_t i = 0; i < (size_t)2 * D0.n_sub; ++i) host[i] = c->step_cir[i];
  for (size_t i = 0; i < n_row; ++i) host[n_step + i] = c->chol_row[i];
  for (size_t i = 0; i < (size_t)2 * D0.n_metric; ++i) host[n_step + n_row + i] = c->cva_coef[i];
  int *flags = reinterpret_cast<int *>(host.data() + n_step + n_row + n_cva);
  for (size_t i = 0; i < n_set; ++i) flags[i] = c->set_cva[i];
  if (p->credit) { cudaFree(p->credit); p->credit = nullptr; }
  MCRE_CUDA(cudaMalloc((void **)&p->credit, host.size() * sizeof(double)));
  MCRE_CUDA(cudaMemcpy(p->credit, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice));
  EqDev &D = p->d;
  D.has_cir = 1; D.cir_det = c->deterministic; D.cir_col = c->noise_col;
  D.cir_kappa = c->kappa; D.cir_theta = c->theta; D.cir_sigma = c->sigma; D.cir_y0 = c->y0; D.lgd = c->lgd;
  D.step_cir = p->credit; D.cir_row = p->credit + n_step; D.cva_coef = p->credit + n_step + n_row;
  D.set_cva = reinterpret_cast<const int *>(p->credit + n_step + n_row + n_cva);
  return 0;
}

static int eq_ns_template(int n_sets) { return n_sets <= 1 ? 1 : (n_sets <= 2 ? 2 : 4); }

extern "C" int64_t mcre_eq_slots(const mcre_eq_plan *p) {
  const int ns = eq_ns_template(p->d.n_sets);
  const bool xt = p->nt > 0 && ((p->d.kind == MCRE_EQ_BS && p->nt != 9) || (p->d.kind == MCRE_EQ_HESTON && p->d.n_expo > 0));
  return (int64_t)ns * 3 + (int64_t)p->d.n_assets * ns * p->nt + (int64_t)p->d.n_metric * ns * 4 +
         (xt ? (int64_t)p->d.n_metric * p->d.n_assets * ns * 2 * p->nt : 0) + (p->d.has_cir ? ns * 2 : 0);
}

template <int KIND, int ALT, int NT, int NS, bool XH = false>
static int eq_launch(mcre_eq_plan *p, const RngDev &rng, const ShardDev &sh, double *partial, double *shift,
                     double *spill, cudaStream_t st) {
  const EqDev &d = p->d;
  const bool presim = d.ps_x != nullptr;
  const int threads = 128, nw = threads / 32;
  constexpr int NVH = NS * 3, NVT = NS * (NT > 0 ? NT : 1), NVX = NS * 4;
  constexpr bool XT = EqExpoTan<KIND, NT, XH>::on;
  constexpr int NVXT = XT ? NS * 2 * NT : 1;
  constexpr int NVMAX0 = (NVH > NVT ? NVH : NVT) > NVX ? (NVH > NVT ? NVH : NVT) : NVX;
  constexpr int NVMAX = NVMAX0 > NVXT ? NVMAX0 : NVXT;
  const int n_slots = NS * 3 + d.n_assets * NS * NT + d.n_metric * NVX + (XT ? d.n_metric * d.n_assets * NVXT : 0) +
                      (d.has_cir ? NS * 2 : 0);
  const size_t smem = ((size_t)n_slots + 2 * nw * NVMAX) * sizeof(double);
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  if (n_chunks == 0 && presim) return 0;
  auto k = eq_main_kernel<KIND, ALT, NT, NS, XH>;
  // (14 KB of static function tables: static + dynamic shared memory beyond 48 KB needs the opt-in, before the query)
  MCRE_SMEM(k, smem, "eq main kernel does not fit (%s%lld bytes of shared memory)");
  int per_sm = 1;
  MCRE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem));
  if (per_sm < 1) return fail(-3, "eq main kernel does not fit%s", "");
  long long grid = (long long)sm_count() * per_sm;
  if (grid > n_chunks) grid = n_chunks;
  // The pilot launch (global path 0 -> the common shift of the shifted sums) runs on every rank, also on one whose
  // shard is empty (fewer chunks than ranks): all ranks finish the all-reduced sums with the same shift.
  ShardDev pilot_sh{0, 1, sh.chunk};
  if (!presim) {   // the pre-simulation pass only spills; it needs no pilot shifts
    k<<<1, threads, smem, st>>>(d, rng, pilot_sh, partial, shift, spill, 1);
    MCRE_LAUNCHED();
  }
  if (n_chunks == 0) return 0;
  k<<<(unsigned)grid, threads, smem, st>>>(d, rng, sh, partial, shift, spill, 0);
  MCRE_LAUNCHED();
  return 0;
}

template <int KIND, int ALT, int NTK>
static int eq_dispatch(mcre_eq_plan *p, const RngDev &rng, const ShardDev &sh, double *partial, double *shift,
                       double *spill, cudaStream_t st) {
  const int ns = eq_ns_template(p->d.n_sets);
  if (p->nt == 0) {
    return ns == 1 ? eq_launch<KIND, ALT, 0, 1>(p, rng, sh, partial, shift, spill, st)
         : ns == 2 ? eq_launch<KIND, ALT, 0, 2>(p, rng, sh, partial, shift, spill, st)
                   : eq_launch<KIND, ALT, 0, 4>(p, rng, sh, partial, shift, spill, st);
  }
  if constexpr (KIND == MCRE_EQ_BS) {
    if (p->nt == 9)
      return ns == 1 ? eq_launch<KIND, ALT, 9, 1>(p, rng, sh, partial, shift, spill, st)
                     : eq_launch<KIND, ALT, 9, 2>(p, rng, sh, partial, shift, spill, st);
  }
  if constexpr (KIND == MCRE_EQ_HESTON) {
    if (p->d.n_expo > 0)     // exposures as duals (sensitivities of exposure metrics through the regression proxy)
      return ns == 1 ? eq_launch<KIND, ALT, NTK, 1, true>(p, rng, sh, partial, shift, spill, st)
                     : eq_launch<KIND, ALT, NTK, 2, true>(p, rng, sh, partial, shift, spill, st);
  }
  return ns == 1 ? eq_launch<KIND, ALT, NTK, 1>(p, rng, sh, partial, shift, spill, st)
                 : eq_launch<KIND, ALT, NTK, 2>(p, rng, sh, partial, shift, spill, st);
}

extern "C" int mcre_eq_mainsim(mcre_eq_plan *p, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                               double *d_acc, double *d_shift, double *d_spill, void *stream) {
  if (!p || !rng || !d_partial || !d_acc || !d_shift) return fail(-1, "null argument%s", "");
  // the equity kernel takes any chunk that is a multiple of a warp (small runs use small chunks)
  if (!shard || shard->n_paths < 0 || shard->chunk_paths <= 0 || shard->chunk_paths % 32 != 0)
    return fail(-2, "invalid shard: chunk_paths must be a positive multiple of 32%s", "");
  if (shard->path_begin % shard->chunk_paths != 0) return fail(-2, "invalid shard: path_begin not chunk aligned%s", "");
  int rc = 0;
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  if (p->d.n_expo > 0 && (p->d.acc_flags & MCRE_ACC_SPILL) && !d_spill && !p->d.ps_x && !p->d.expo_accum)
    return fail(-1, "spill requested but d_spill is null%s", "");
  if (p->nt > 0 && p->has_proxy && !p->d.xp_tan && !p->d.ps_x)
    return fail(-1, "eq: plan with tangents and regression-proxy exposures: call mcre_eq_set_exposure_coef_tangents first%s", "");
  if (p->nt > 0 && p->has_exercise_expo && !p->d.xp_ex_tan && !p->d.ps_x)
    return fail(-1, "eq: plan with tangents and exposures of exercise products: call "
                    "mcre_eq_set_exercise_exposure_coef_tangents first%s", "");
  if (rng->mode == MCRE_RNG_INJECT && p->d.kind == MCRE_EQ_HESTON && p->d.scheme == MCRE_SCHEME_QE && !rng->d_u)
    return fail(-1, "inject mode: QE needs uniforms%s", "");
  RngDev r = make_rng(rng);
  ShardDev sh{shard->path_begin, shard->n_paths, shard->chunk_paths};
  cudaStream_t st = (cudaStream_t)stream;
  const int alt = (p->d.scheme == MCRE_SCHEME_EULER) ? 0 : 1;
  switch (p->d.kind) {
    case MCRE_EQ_BS:
      rc = alt ? eq_dispatch<MCRE_EQ_BS, 1, 3>(p, r, sh, d_partial, d_shift, d_spill, st)
               : eq_dispatch<MCRE_EQ_BS, 0, 3>(p, r, sh, d_partial, d_shift, d_spill, st);
      break;
    case MCRE_EQ_HESTON:
      rc = alt ? eq_dispatch<MCRE_EQ_HESTON, 1, 7>(p, r, sh, d_partial, d_shift, d_spill, st)
               : eq_dispatch<MCRE_EQ_HESTON, 0, 7>(p, r, sh, d_partial, d_shift, d_spill, st);
      break;
    default:
      rc = alt ? eq_dispatch<MCRE_EQ_SCHWARTZ, 1, 6>(p, r, sh, d_partial, d_shift, d_spill, st)
               : eq_dispatch<MCRE_EQ_SCHWARTZ, 0, 6>(p, r, sh, d_partial, d_shift, d_spill, st);
  }
  if (rc) return rc;
  const long long n_chunks = (sh.n_paths + sh.chunk - 1) / sh.chunk;
  return mcre_tree_reduce(d_partial, n_chunks, mcre_eq_slots(p), d_acc, stream);
}

extern "C" int mcre_eq_set_exposure_accumulator(mcre_eq_plan *p, double *d_accum) {
  if (!p) return fail(-1, "null argument%s", "");
  p->d.expo_accum = d_accum;
  return 0;
}

extern "C" int mcre_eq_set_exposure_tangent_accumulator(mcre_eq_plan *p, double *d_accum_tan) {
  if (!p) return fail(-1, "null argument%s", "");
  if (d_accum_tan && (p->d.kind != MCRE_EQ_BS || p->nt <= 0))
    return fail(-3, "eq: exposure tangents exist in Black-Scholes plans with tangents%s", "");
  p->d.expo_accum_tan = d_accum_tan;
  return 0;
}

namespace mcre {
// Tangent sums of the exposure metrics of one netting set from per-path exposures and tangents: one block per
// (chunk of paths, parameter, metric date); fixed summation order inside the block.
// CVA weights: w [n_metric] shared by all paths, or per path wp [n_metric][n] (stochastic intensity) scaled by lgd; with
// wt [n_metric][n_wtan][n] = tangents of the per-path weights w.r.t. the credit model's own parameters the grid's
// y-dimension runs over n_par + n_wtan "parameters": for g >= n_par slot 2 = lgd * sum relu(U) d w / d credit_g.
__global__ void __launch_bounds__(128) exposure_tangent_sums_kernel(const double *__restrict__ expo, const double *__restrict__ tan,
                                                                    long long n, int n_expo, int n_par, int n_metric,
                                                                    const int *__restrict__ metric_expo,
                                                                    const int *__restrict__ lag, int collateralised, double h,
                                                                    const double *__restrict__ w, const double *__restrict__ wp,
                                                                    double lgd, const double *__restrict__ wt, int n_wtan,
                                                                    int chunk, double *__restrict__ partial) {
  __shared__ double stage[4][3];
  const int g = blockIdx.y, m = blockIdx.z;
  const int xe = metric_expo[m];
  const int l = collateralised ? lag[m] : -1;
  const bool credit = g >= n_par;
  const double *tg = tan + (size_t)(credit ? 0 : g) * n_expo * n;
  const double *wtg = credit ? wt + ((size_t)m * n_wtan + (g - n_par)) * n : nullptr;
  double s_pos = 0.0, s_neg = 0.0, s_cva = 0.0;
  const long long base = (long long)blockIdx.x * chunk;
  for (int it = threadIdx.x; it < chunk; it += blockDim.x) {
    const long long p = base + it;
    if (p >= n) break;
    const double now = expo[(size_t)xe * n + p], dnow = credit ? 0.0 : tg[(size_t)xe * n + p];
    auto thr = [h](double x) { return x > h ? x - h : (x < -h ? x + h : 0.0); };
    auto dthr = [h](double x) { return (x > h || x < -h) ? 1.0 : 0.0; };
    double u, du;
    if (collateralised) {
      const double delayed = l >= 0 ? expo[(size_t)(xe - l) * n + p] : 0.0;
      const double ddel = (l >= 0 && !credit) ? tg[(size_t)(xe - l) * n + p] : 0.0;
      u = now - thr(delayed); du = dnow - dthr(delayed) * ddel;
    } else {
      u = thr(now); du = dthr(now) * dnow;
    }
    if (credit) {
      if (u > 0.0) s_cva += u * wtg[p];
    } else {
      if (u > 0.0) { s_pos += du; if (wp) s_cva += du * wp[(size_t)m * n + p]; }
      if (u < 0.0) s_neg += du;
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 16; off > 0; off >>= 1) {
    s_pos += __shfl_xor_sync(0xffffffffu, s_pos, off);
    s_neg += __shfl_xor_sync(0xffffffffu, s_neg, off);
    s_cva += __shfl_xor_sync(0xffffffffu, s_cva, off);
  }
  if (lane == 0) { stage[warp][0] = s_pos; stage[warp][1] = s_neg; stage[warp][2] = s_cva; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0, c = 0.0;
    for (int k = 0; k < 4; ++k) { a += stage[k][0]; b += stage[k][1]; c += stage[k][2]; }
    const int np_tot = n_par + n_wtan;
    double *o = partial + ((size_t)blockIdx.x * n_metric * np_tot + (size_t)m * np_tot + g) * 3;
    o[0] = a; o[1] = b; o[2] = (wp || credit) ? lgd * c : w[m] * a;
  }
}

// Tangents of the per-path default weights w_k = exp(-int lambda) (1 - C_k exp(-B_k y_k)) of a stochastic CIR++ credit
// factor w.r.t. its own parameters (kappa, theta, sigma, y0): the factor is replayed from the same draws as in
// eq_main_kernel (column cir_col of the joint draw, correlated through the credit row of the Cholesky factor) with the
// Euler recursion differentiated by hand (cirpp.py:174-198, clamps pass the derivative like torch.clamp), one path per
// thread.  psi [n_sub], dpsi [n_sub][4], coef [n_metric][2] = (C_k, B_k), dcoef [n_metric][2][4].
struct CreditTanDev {
  double kappa, theta, sigma, y0;
  int cir_col;
  const double *row, *psi, *dpsi, *coef, *dcoef;
};
__global__ void __launch_bounds__(128) credit_weight_tangents_kernel(EqDev P, RngDev rng, ShardDev sh, CreditTanDev ct,
                                                                      double *__restrict__ w_tan) {
  fm_tables_init();      // (the Philox normals go through the table-driven elementary functions, like eq_main_kernel's)
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= sh.n_paths) return;
  const unsigned long long gpath = (unsigned long long)(sh.path_begin + p);
  NormalStream ns; ns.init(rng, gpath);
  const int d = P.noise_dim;
  double cy = ct.y0, lb = 0.0, cyd[4] = {0.0, 0.0, 0.0, 1.0}, lbd[4] = {0.0, 0.0, 0.0, 0.0};
  auto emit = [&](int di) {
    const int m = __ldg(P.date_metric + di);
    if (m < 0) return;
    const double Ck = __ldg(ct.coef + 2 * m), Bk = __ldg(ct.coef + 2 * m + 1);
    const double e1 = exp(-lb), e2 = exp(-Bk * cy), w = e1 * (1.0 - Ck * e2);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const double dC = __ldg(ct.dcoef + (size_t)m * 8 + j), dB = __ldg(ct.dcoef + (size_t)m * 8 + 4 + j);
      const double dw = -w * lbd[j] + e1 * e2 * (Ck * (dB * cy + Bk * cyd[j]) - dC);
      w_tan[((size_t)m * 4 + j) * sh.n_paths + p] = m < P.n_metric - 1 ? dw : 0.0;
    }
  };
  for (int di = 0; di < P.n_pre_dates; ++di) emit(di);
  for (int is = 0; is < P.n_sub; ++is) {
    const double dt = __ldg(P.step_dt + is), sq = __ldg(P.step_sq + is);
    double wc = 0.0;
    for (int j = 0; j < d; ++j) {
      double zj;
      if (rng.mode == MCRE_RNG_INJECT) zj = rng.z[((size_t)is * rng.n_total + gpath) * d + j];
      else {
        const uint32_t nc = (uint32_t)(is * d + j);
        double p0, p1;
        ns.pair(nc >> 1, p0, p1);
        zj = (nc & 1u) ? p1 : p0;
      }
      wc = fma(__ldg(ct.row + j), zj, wc);
    }
    const double sp = sqrt(fmax(cy, 0.0)), gsp = cy > 0.0 ? 0.5 / sp : 0.0;
    const double yn = cy + ct.kappa * (ct.theta - cy) * dt + ct.sigma * sp * sq * wc;
    const double carry = 1.0 - ct.kappa * dt + ct.sigma * sq * wc * gsp;
    double dyn[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) dyn[j] = carry * cyd[j];
    dyn[0] += (ct.theta - cy) * dt; dyn[1] += ct.kappa * dt; dyn[2] += sp * sq * wc;
    lb += (cy + __ldg(ct.psi + is)) * dt;
#pragma unroll
    for (int j = 0; j < 4; ++j) lbd[j] += (cyd[j] + __ldg(ct.dpsi + (size_t)is * 4 + j)) * dt;
    const bool pass = yn >= 1e-12;
    cy = fmax(yn, 1e-12);
#pragma unroll
    for (int j = 0; j < 4; ++j) cyd[j] = pass ? dyn[j] : 0.0;
    const int di = __ldg(P.step_date + is);
    if (di >= 0) emit(di);
  }
}
}  // namespace mcre

extern "C" int mcre_eq_credit_weight_tangents(mcre_eq_plan *p, const mcre_eq_credit *c, const double *dpsi, const double *dcoef,
                                              const mcre_rng *rng, const mcre_shard *shard, double *d_w_tan, void *stream) {
  if (!p || !c || !dpsi || !dcoef || !rng || !shard || !d_w_tan || !c->step_cir || !c->chol_row || !c->cva_coef)
    return fail(-1, "null argument%s", "");
  if (c->deterministic) return fail(-4, "credit weight tangents: the deterministic intensity has no parameters%s", "");
  if (p->d.n_metric <= 0 || !p->d.date_metric) return fail(-4, "credit weight tangents: the plan has no metric dates%s", "");
  if (c->noise_col < 0 || c->noise_col >= p->d.noise_dim) return fail(-1, "eq: credit noise column out of range%s", "");
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  const EqDev &D = p->d;
  const size_t ns_ = (size_t)(D.n_sub > 0 ? D.n_sub : 1), nm = (size_t)D.n_metric, nd = (size_t)D.noise_dim;
  std::vector<double> host(nd + ns_ + ns_ * 4 + nm * 2 + nm * 8, 0.0);
  double *row = host.data(), *psi = row + nd, *dps = psi + ns_, *cf = dps + ns_ * 4, *dcf = cf + nm * 2;
  for (size_t i = 0; i < nd; ++i) row[i] = c->chol_row[i];
  for (size_t i = 0; i < (size_t)D.n_sub; ++i) psi[i] = c->step_cir[2 * i];
  for (size_t i = 0; i < (size_t)D.n_sub * 4; ++i) dps[i] = dpsi[i];
  for (size_t i = 0; i < nm * 2; ++i) cf[i] = c->cva_coef[i];
  for (size_t i = 0; i < nm * 8; ++i) dcf[i] = dcoef[i];
  double *dev = nullptr;
  MCRE_CUDA(cudaMalloc((void **)&dev, host.size() * sizeof(double)));
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemcpyAsync(dev, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice, st);
  int rc = e == cudaSuccess ? 0 : cuda_fail(e, "copy");
  if (!rc && shard->n_paths > 0) {
    CreditTanDev ct{c->kappa, c->theta, c->sigma, c->y0, c->noise_col, dev, dev + nd, dev + nd + ns_, dev + nd + ns_ * 5,
                    dev + nd + ns_ * 5 + nm * 2};
    RngDev r = make_rng(rng);
    ShardDev sh{shard->path_begin, shard->n_paths, shard->chunk_paths};
    credit_weight_tangents_kernel<<<(unsigned)((shard->n_paths + 127) / 128), 128, 0, st>>>(D, r, sh, ct, d_w_tan);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "kernel launch");
  }
  cudaStreamSynchronize(st);   // the tables are freed below (pageable host source: the copy has completed too)
  cudaFree(dev);
  return rc;
}

static int exposure_tangent_sums_impl(const double *d_expo, const double *d_tan, int64_t n_paths, int32_t n_expo,
                                      int32_t n_par, int32_t n_metric, const int32_t *metric_expo, const int32_t *lag,
                                      int32_t collateralised, double threshold, const double *weights,
                                      const double *d_w_paths, double lgd, const double *d_w_tan, int32_t n_wtan,
                                      int32_t chunk_paths, double *d_partial, double *d_out, void *stream) {
  if (!d_expo || !d_tan || !metric_expo || !lag || (!weights && !d_w_paths) || !d_partial || !d_out)
    return fail(-1, "null argument%s", "");
  if (n_par <= 0 || n_metric <= 0 || n_expo <= 0 || chunk_paths <= 0 || n_wtan < 0 || (n_wtan > 0 && !d_w_tan))
    return fail(-2, "tangent sums: bad shape%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t slots = (int64_t)n_metric * (n_par + n_wtan) * 3;
  const long long n_chunks = n_paths > 0 ? (n_paths + chunk_paths - 1) / chunk_paths : 0;
  std::vector<double> zero_w((size_t)n_metric, 0.0);
  DevArray<int> me, lg;
  DevArray<double> wd;
  DevArena arena;
  int rc = 0;
  {
    ArenaScope scope(&arena);
    rc = me.upload(metric_expo, n_metric);
    if (!rc) rc = lg.upload(lag, n_metric);
    if (!rc) rc = wd.upload(weights ? weights : zero_w.data(), n_metric);
    if (!rc) rc = arena.commit();
  }
  if (!rc && n_chunks > 0) {
    dim3 grid((unsigned)n_chunks, (unsigned)(n_par + n_wtan), (unsigned)n_metric);
    exposure_tangent_sums_kernel<<<grid, 128, 0, st>>>(d_expo, d_tan, n_paths, n_expo, n_par, n_metric, me.p, lg.p,
                                                       collateralised, threshold, wd.p, d_w_paths, lgd, d_w_tan, n_wtan,
                                                       chunk_paths, d_partial);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "kernel launch");
  }
  if (!rc) rc = mcre_tree_reduce(d_partial, n_chunks, slots, d_out, stream);
  if (!rc) cudaStreamSynchronize(st);   // the index tables are freed below
  arena.release();
  return rc;
}

extern "C" int mcre_exposure_tangent_sums(const double *d_expo, const double *d_tan, int64_t n_paths, int32_t n_expo,
                                          int32_t n_par, int32_t n_metric, const int32_t *metric_expo, const int32_t *lag,
                                          int32_t collateralised, double threshold, const double *weights,
                                          int32_t chunk_paths, double *d_partial, double *d_out, void *stream) {
  if (!weights) return fail(-1, "null argument%s", "");
  return exposure_tangent_sums_impl(d_expo, d_tan, n_paths, n_expo, n_par, n_metric, metric_expo, lag, collateralised,
                                    threshold, weights, nullptr, 0.0, nullptr, 0, chunk_paths, d_partial, d_out, stream);
}

extern "C" int mcre_exposure_tangent_sums_paths(const double *d_expo, const double *d_tan, int64_t n_paths, int32_t n_expo,
                                                int32_t n_par, int32_t n_metric, const int32_t *metric_expo,
                                                const int32_t *lag, int32_t collateralised, double threshold,
                                                const double *d_w_paths, double lgd, const double *d_w_tan, int32_t n_wtan,
                                                int32_t chunk_paths, double *d_partial, double *d_out, void *stream) {
  if (!d_w_paths) return fail(-1, "null argument%s", "");
  return exposure_tangent_sums_impl(d_expo, d_tan, n_paths, n_expo, n_par, n_metric, metric_expo, lag, collateralised,
                                    threshold, nullptr, d_w_paths, lgd, d_w_tan, n_wtan, chunk_paths, d_partial, d_out, stream);
}

namespace mcre {
// Netting-set terms on accumulated exposures (netting_set.py:48-72, 136-184): one thread per (path, metric date).
// expo [n_expo][n], metric_expo [n_metric] = exposure index of the metric date, lag [n_metric] = exposure indices
// back to the collateral date (-1: none), out [n_metric][n] unsecured exposure.
__global__ void __launch_bounds__(256) eq_unsecured_kernel(const double *__restrict__ expo, long long n, int n_metric,
                                                           const int *__restrict__ metric_expo, const int *__restrict__ lag,
                                                           int collateralised, double h, double *__restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  if (p >= n || m >= n_metric) return;
  auto thr = [h](double x) { return x > h ? x - h : (x < -h ? x + h : 0.0); };
  const int xe = metric_expo[m];
  const double now = expo[(size_t)xe * n + p];
  double unsec;
  if (collateralised) {
    const int l = lag[m];
    const double delayed = l >= 0 ? expo[(size_t)(xe - l) * n + p] : 0.0;
    unsec = now - thr(delayed);
  } else {
    unsec = thr(now);
  }
  out[(size_t)m * n + p] = unsec;
}
}  // namespace mcre

extern "C" int mcre_eq_unsecured_exposures(const double *d_expo, int64_t n_paths, int32_t n_metric, const int32_t *metric_expo,
                                           const int32_t *lag, int32_t collateralised, double threshold, double *d_out,
                                           void *stream) {
  if (!d_expo || !metric_expo || !lag || !d_out) return fail(-1, "null argument%s", "");
  if (n_paths <= 0 || n_metric <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  DevArray<int> me, lg;
  DevArena arena;
  int rc = 0;
  {
    ArenaScope scope(&arena);
    rc = me.upload(metric_expo, n_metric);
    if (!rc) rc = lg.upload(lag, n_metric);
    if (!rc) rc = arena.commit();
  }
  if (!rc) {
    dim3 grid((unsigned)((n_paths + 255) / 256), (unsigned)n_metric);
    eq_unsecured_kernel<<<grid, 256, 0, st>>>(d_expo, n_paths, n_metric, me.p, lg.p, collateralised, threshold, d_out);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = cuda_fail(e, "kernel launch");
    else cudaStreamSynchronize(st);   // the index tables are freed below
  }
  arena.release();
  return rc;
}

extern "C" int mcre_eq_set_cva_weight_spill(mcre_eq_plan *p, double *d_w) {
  if (!p) return fail(-1, "null argument%s", "");
  if (d_w && !p->d.has_cir) return fail(-1, "eq: CVA weight spill without a credit factor (mcre_eq_set_credit)%s", "");
  p->d.cva_w = d_w;
  return 0;
}

namespace mcre {
// per-path CVA of a netting set from its unsecured exposures and the default weights, both [n_metric][n]
// (cva_metric.py:62-100): out[p] = lgd * sum_m relu(unsec[m][p]) * w[m][p]
__global__ void __launch_bounds__(256) eq_cva_paths_kernel(const double *__restrict__ unsec, const double *__restrict__ w,
                                                           long long n, int n_metric, double lgd, double *__restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  double tot = 0.0;
  for (int m = 0; m < n_metric - 1; ++m) tot = fma(fmax(unsec[(size_t)m * n + p], 0.0), w[(size_t)m * n + p], tot);
  out[p] = tot * lgd;
}
}  // namespace mcre

extern "C" int mcre_eq_cva_paths(const double *d_unsec, const double *d_w, int64_t n_paths, int32_t n_metric, double lgd,
                                 double *d_out, void *stream) {
  if (!d_unsec || !d_w || !d_out) return fail(-1, "null argument%s", "");
  if (n_paths <= 0) return 0;
  eq_cva_paths_kernel<<<(unsigned)((n_paths + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_unsec, d_w, n_paths, n_metric, lgd, d_out);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_eq_set_bridge_uniforms(mcre_eq_plan *p, const double *d_u, int32_t stride) {
  if (!p) return fail(-1, "null argument%s", "");
  p->d.bridge_u = d_u; p->d.bridge_stride = stride;
  return 0;
}

extern "C" int mcre_eq_set_pv_accumulator(mcre_eq_plan *p, double *d_accum) {
  if (!p) return fail(-1, "null argument%s", "");
  p->d.pv_accum = d_accum;
  return 0;
}

extern "C" int mcre_eq_presim_tangents(mcre_eq_plan *p, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                                       double *d_shift, double *d_x, float *d_cf, double *d_dx, double *d_dcf, void *stream) {
  if (!p || !rng || !d_partial || !d_shift || !d_x || !d_cf || !d_dx || !d_dcf) return fail(-1, "null argument%s", "");
  if (p->nt <= 0 || !eq_kind_has_exposure_tangents(p->d.kind))
    return fail(-4, "eq presim tangents: Black-Scholes / Heston plans with tangents only%s", "");
  if (p->d.n_expo <= 0) return fail(-1, "eq presim: the plan has no exposure dates%s", "");
  p->d.ps_x = d_x; p->d.ps_cf = d_cf; p->d.ps_dx = d_dx; p->d.ps_dcf = d_dcf;
  const int rc = mcre_eq_mainsim(p, rng, shard, d_partial, d_partial /* scratch: sums are not used */, d_shift, nullptr, stream);
  p->d.ps_x = nullptr; p->d.ps_cf = nullptr; p->d.ps_dx = nullptr; p->d.ps_dcf = nullptr;
  return rc;
}

extern "C" int mcre_eq_presim(mcre_eq_plan *p, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                              double *d_shift, double *d_x, float *d_cf, void *stream) {
  if (!p || !rng || !d_partial || !d_shift || !d_x || !d_cf) return fail(-1, "null argument%s", "");
  if (p->nt != 0) return fail(-4, "eq presim: tangents through the regression are not implemented%s", "");
  if (p->d.n_expo <= 0) return fail(-1, "eq presim: the plan has no exposure dates%s", "");
  p->d.ps_x = d_x; p->d.ps_cf = d_cf;
  const int rc = mcre_eq_mainsim(p, rng, shard, d_partial, d_partial /* scratch: sums are not used */, d_shift, nullptr, stream);
  p->d.ps_x = nullptr; p->d.ps_cf = nullptr;
  return rc;
}
