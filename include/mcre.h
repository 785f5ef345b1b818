/*
 * mcre.h - C ABI of the B200-native Monte Carlo risk engine (libmcre_b200.so).
 *
 * The reference (konstantineder/montecarlo-risk-engine) is pure Python on PyTorch
 * CPU and has no FFI.  The seam this library sits behind is its Python API
 * (SimulationController.run_simulation, src/controller/controller.py:663-709); the
 * entry points below are what that API's hot loops are replaced by.  Each one cites
 * the reference code whose work it takes over.  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / C++ types.  All `const double*` /
 *     `const int32_t*` inputs of *_create are HOST pointers (copied to the device);
 *     all `d_*` pointers are DEVICE pointers owned by the caller
 *     (torch.Tensor.data_ptr()).  `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, <0 for an invalid argument / plan,
 *     >0 for a cudaError_t.  mcre_last_error() gives the message (thread local).
 *   - launches are asynchronous on `stream`; nothing synchronises unless stated.
 *   - "dual" tables: a model-parameter-dependent scalar is stored as (1+NT) doubles,
 *     value first, then its tangents w.r.t. the NT model parameters.  NT = 0 when
 *     sensitivities are off.
 */
#ifndef MCRE_H
#define MCRE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCRE_ABI_VERSION 1

/* ---- enums -------------------------------------------------------------------- */
enum { MCRE_SCHEME_EULER = 0, MCRE_SCHEME_ANALYTICAL = 2, MCRE_SCHEME_QE = 3 }; /* src/common/enums.py:4-8 */
enum {
  MCRE_MODEL_BS = 0,        /* src/models/black_scholes.py       */
  MCRE_MODEL_BSM = 1,       /* src/models/black_scholes_multi.py */
  MCRE_MODEL_HESTON = 2,    /* src/models/heston.py              */
  MCRE_MODEL_VASICEK = 3,   /* src/models/vasicek.py             */
  MCRE_MODEL_CIRPP = 4,     /* src/models/cirpp.py               */
  MCRE_MODEL_SCHWARTZ2F = 5 /* src/models/schwartz_two_factor.py */
};

/* Normal-draw source.  PHILOX: counter-based Philox4x32-10, key=(seed, stream),
 * counter=(global path id, sub-step, draw block) + Box-Muller in registers.
 * INJECT: read the reference's own draws (torch.manual_seed(42|43); torch.randn(N,d)
 * per sub-step, src/engine/engine.py:25, src/models/model.py:47) from device memory:
 * z[n_sub][n_paths][noise_dim] (and u[n_sub][n_paths] for Heston-QE). */
enum { MCRE_RNG_PHILOX = 0, MCRE_RNG_INJECT = 1 };

typedef struct {
  int32_t mode;          /* MCRE_RNG_* */
  uint64_t seed;         /* Philox key low 64 bits: 42 pre-simulation, 43 main (engine.py:25) */
  uint64_t stream;       /* Philox key high bits: scenario / sweep index */
  const double *d_z;     /* INJECT: device, [n_sub][n_paths_total][noise_dim] */
  const double *d_u;     /* INJECT: device, [n_sub][n_paths_total] (QE uniforms) or NULL */
  int64_t n_paths_total; /* leading stride of d_z / d_u */
} mcre_rng;

/* Which slice of the global path range this process simulates (multi-GPU sharding,
 * SURVEY §8e): global path ids [path_begin, path_begin + n_paths).  Partial sums are
 * formed per fixed-size chunk of `chunk_paths` global ids and combined in a fixed
 * binary tree, so results do not depend on the number of GPUs. */
typedef struct {
  int64_t path_begin;
  int64_t n_paths;
  int32_t chunk_paths; /* multiple of 256; path_begin % chunk_paths == 0 */
} mcre_shard;

/* ================================================================================
 * Generic path generator (compatibility / debugging seam)
 * replaces MonteCarloEngine.generate_paths(), src/engine/engine.py:27-123, and
 * Model.simulate_time_step_*; materialises paths [n_paths][n_dates][state_dim].
 * NOT used by the fused hot path.
 * ============================================================================== */
typedef struct {
  int32_t n_models;
  const int32_t *model_kind;    /* [n_models] MCRE_MODEL_*                                   */
  const int32_t *model_nassets; /* [n_models] (BSM: number of assets, else 1)                */
  const double *model_params;   /* concatenated parameters in the reference's order          */
  const int32_t *model_flags;   /* [n_models] bit0: CIR++ deterministic, bit1: fuzzy smoothing*/
  int32_t scheme;               /* MCRE_SCHEME_*                                             */
  int32_t noise_dim, state_dim;
  int32_t n_sub, n_dates;
  int32_t n_pre_dates;          /* number of leading dates with dt<=0 (initial state copied) */
  const double *step_dt;        /* [n_sub] time2 - time1 as the models see it                */
  const double *step_t1;        /* [n_sub] accumulated start time (engine.py:60)             */
  const int32_t *step_date;     /* [n_sub] simulation-date index completed by the step or -1 */
  const double *chol;           /* [n_chol][noise_dim][noise_dim] lower Cholesky factors:
                                   of the correlation (EULER/QE) or of the step covariance
                                   (ANALYTICAL, one per distinct dt; model.py:50-73)         */
  const int32_t *step_chol;     /* [n_sub] index into chol                                   */
  const double *step_aux;       /* [n_sub][n_models][4] per-step model scalars:
                                   [0] CIR++ psi(t1) | Schwartz log F0(t2)
                                   [1],[2] deterministic CIR++ lambda_mkt(t1), lambda_mkt(t2)
                                   [3] Vasicek / Hull-White mean level theta(t1)             */
  const double *init_state;     /* [state_dim]                                               */
} mcre_paths_desc;

int mcre_generate_paths(const mcre_paths_desc *desc, const mcre_rng *rng, const mcre_shard *shard,
                        double *d_paths /* [n_paths][n_dates][state_dim] */, void *stream);

/* ================================================================================
 * Interest-rate / credit family (IRC): Vasicek short rate (+ optional CIR++ intensity)
 * with bonds, swaps and (later) options on them; PV / CE / EPE / ENE / EEPE / PFE / CVA
 * with thresholds and MPoR-delayed collateral.
 * Replaces, fused into one pass per path with no path tensor:
 *   engine.generate_paths           src/engine/engine.py:27-123
 *   RequestInterface.resolve_requests   src/request_interface/request_interface.py:115-130
 *   Bond / InterestRateSwap cashflows   src/products/bond.py:165-214, swap.py:142-172
 *   SimulationController._evaluate_product  src/controller/controller.py:385-471
 *   NettingSet.compute_unsecured_exposure_profiles  src/products/netting_set.py:156-184
 *   Metric.evaluate (PV/CE/EPE/ENE/CVA)  src/metrics/*.py
 * ============================================================================== */
#define MCRE_IRC_MAX_SETS 4   /* netting sets per launch (host splits larger books)    */
#define MCRE_IRC_MAX_UNITS 4  /* regression units (products) per pre-simulation launch  */
#define MCRE_IRC_MAX_LAG 4    /* max exposure-date lag of the MPoR look-back            */
#define MCRE_IRC_MAX_BERM 8   /* Bermudan exercise units per launch                     */

/* per-date flags */
#define MCRE_DATE_HAS_CASHFLOW 1
#define MCRE_DATE_HAS_EXPOSURE 2
#define MCRE_DATE_HAS_METRIC 4
#define MCRE_DATE_HAS_REGRESSION 8
#define MCRE_DATE_HAS_EXERCISE 16

/* what the main simulation accumulates */
#define MCRE_ACC_PV 1
#define MCRE_ACC_POS 2    /* sum relu(E), sum relu(E)^2 per metric date (CE / EPE / EEPE) */
#define MCRE_ACC_NEG 4    /* sum -relu(-E) and squares per metric date (ENE)               */
#define MCRE_ACC_CVA 8
#define MCRE_ACC_SPILL 16 /* write unsecured exposures [set][metric date][path] (PFE)      */

typedef struct {
  /* ---- models ---- */
  int32_t nt;            /* number of tangent directions (0, 4 or 8)                         */
  int32_t scheme;        /* EULER, or ANALYTICAL (Vasicek only)                              */
  int32_t has_cir;       /* 0: Vasicek only (noise_dim 1); 1: Vasicek + CIR++ (noise_dim 2)  */
  int32_t cir_deterministic;
  int32_t vas_noise, cir_noise; /* column of the correlated noise each model consumes       */
  const double *vas;     /* dual[4]: r0, sigma, theta, a            (vasicek.py:24-27)       */
  const double *cir;     /* dual[4]: kappa, theta, sigma, y0        (cirpp.py:42-47)         */
  const double *cir_init;/* dual[1]: initial y (y0, or lambda_mkt(0) when deterministic)     */
  const double *chol;    /* dual[4]: L00, L01(=0), L10, L11 of the correlation (model.py:66-73) */
  /* ---- time grid ---- */
  int32_t n_sub, n_dates, n_pre_dates;
  const double *step_dt;       /* [n_sub]                                                    */
  const int32_t *step_date;    /* [n_sub] date index completed by this sub-step or -1        */
  const double *step_vas;      /* dual[n_sub][2]: ANALYTICAL decay e^{-a dt}, noise std;
                                  EULER: theta(t1) (Hull-White extension), unused            */
  const double *step_cir;      /* dual[n_sub][2]: psi(t1), unused | lambda(t1), lambda(t2)   */
  /* ---- per simulation date ---- */
  const int32_t *date_flags;   /* [n_dates]                                                  */
  const int32_t *date_expo;    /* [n_dates] internal exposure index or -1                    */
  const int32_t *date_metric;  /* [n_dates] metric-date index or -1                          */
  const int32_t *date_reg;     /* [n_dates] regression-date index or -1 (pre-simulation)     */
  const int32_t *date_float_off; /* [n_dates+1] CSR offsets into the float-period pool       */
  const double *float_coef;    /* dual[n_float][2]: alpha, B of P(t1,t2;r)=exp(alpha-B r)    */
  const double *float_inv_tau; /* [n_float] 1/(t2-t1) of the LIBOR period (vasicek.py:147-151)*/
  /* ---- netting sets (main simulation) ---- */
  int32_t n_sets;
  int32_t n_expo, n_metric;
  int32_t acc_flags;           /* MCRE_ACC_*                                                 */
  const double *set_fix;       /* [n_sets][n_dates] fixed cashflow amount paid at the date   */
  const double *set_float;     /* [n_sets][n_float] weight on LIBOR_j * 1 (already * dt)     */
  const double *set_threshold; /* [n_sets]                                                   */
  const int32_t *set_flags;    /* [n_sets] bit0 collateralised, bit1 CVA applies             */
  const int32_t *set_lag;      /* [n_sets][n_metric] exposure-index lag of the collateral date, -1: none */
  const double *expo_coef;     /* dual[n_expo][n_sets][3] netted regression coefficients     */
  const double *expo_basis;    /* [n_expo][2] shift, scale of the explanatory variable       */
  const double *cva_coef;      /* dual[n_metric][2]: C_k, B_k of S(t_k,t_k+1|y)=C exp(-B y) (cirpp.py:246-285) */
  double lgd;                  /* 1 - recovery (cva_metric.py:97)                            */
  /* ---- regression units (pre-simulation) ---- */
  int32_t n_units, n_reg;
  const double *unit_fix;      /* [n_units][n_dates]                                         */
  const double *unit_float;    /* [n_units][n_float]                                         */
  const int32_t *unit_last_reg;/* [n_units] number of regression dates that see cashflows    */
  const double *reg_basis;     /* [n_reg][2] shift, scale                                    */
  /* ---- Bermudan exercise units (bermudan_option.py:93-188); n_berm = 0: none ---- */
  int32_t n_berm;              /* <= MCRE_IRC_MAX_BERM                                       */
  const int32_t *berm_set;     /* [n_berm] netting-set row the unit's cashflows / exposure go to */
  const double *berm_strike;   /* [n_berm]                                                   */
  const double *berm_sign;     /* [n_berm] +1 call, -1 put                                   */
  const int32_t *date_ex_off;  /* [n_dates+1] CSR offsets of the exercise records per date   */
  const int32_t *ex_unit;      /* [n_ex] unit of the record                                  */
  const int32_t *ex_last;      /* [n_ex] 1: last exercise date of the unit (continuation 0)  */
  const int32_t *ex_term_off;  /* [n_ex+1] CSR offsets into the zero-bond term pool          */
  const double *ex_const;      /* [n_ex] constant part of the underlying's value             */
  const double *term_coef;     /* dual[n_term][2] alpha, B of P(t_ex, T_j; r) = exp(alpha - B r) */
  const double *term_w;        /* [n_term] weight of the zero bond in the underlying's value */
  const double *ex_basis;      /* [n_ex][2] shift, scale of the explanatory variable         */
  /* ---- hybrid books: numeraire of another model (model_config.py:44-47, numeraire_model_idx) ---- */
  int32_t ext_numeraire;       /* 1: numeraire = exp(ext_rate (t - t0)) instead of the short rate's own account */
  double ext_rate;
  int32_t ext_slot;            /* plans with tangents: the tangent slot that stands for ext_rate, -1: a constant   */
} mcre_irc_desc;

typedef struct mcre_irc_plan mcre_irc_plan;

int mcre_irc_create(const mcre_irc_desc *desc, mcre_irc_plan **out);
void mcre_irc_destroy(mcre_irc_plan *plan);
/* Per-path discounted cashflow totals of the main simulation: d_pv [n_sets][shard->n_paths] is WRITTEN by the next
 * mcre_irc_mainsim (plans of linear products with MCRE_ACC_PV).  With MCRE_ACC_SPILL on a plan whose
 * metric dates are all its exposure dates this gives per-path cashflows and exposures of the rate products of a book
 * that also holds products of another model family (mcre/hybrid.py; the reference nets them in one loop over
 * products, controller.py:506-563).  NULL: off. */
int mcre_irc_set_pv_spill(mcre_irc_plan *plan, double *d_pv);

/* Number of accumulator slots of the main simulation / pre-simulation moments. */
int64_t mcre_irc_main_slots(const mcre_irc_plan *plan);
int64_t mcre_irc_presim_slots(const mcre_irc_plan *plan);
/* Bytes of device scratch the pre-simulation needs for `n_paths` local paths. */
int64_t mcre_irc_presim_scratch_bytes(const mcre_irc_plan *plan, int64_t n_paths);
int64_t mcre_irc_partial_bytes(const mcre_irc_plan *plan, int64_t n_paths, int32_t chunk_paths, int presim);

/* Pre-simulation (replaces controller._perform_regression, controller.py:272-383, up to
 * the least-squares solve): accumulates for every regression date k the Gram moments
 * sum u^0..u^4 and, per unit, sum u^j * Y_k with Y_k = N(t_k) * fp32 suffix sum of the
 * discounted future cashflows (the FP32 accumulation of controller.py:312-351 is
 * reproduced bit for bit).  d_moments: [n_reg][5 + 3*n_units].
 * Plans with tangents (nt > 0, differentiate=True): the reference's regression coefficients stay
 * inside the autograd graph (controller.py:118-119, 368-383), so sensitivities of exposure metrics
 * contain d(coefficients)/d(parameters).  The forward pass then propagates the pathwise tangents of
 * x, N and the windowed cashflows and d_tmoments receives [n_units][nt][n_reg][9] =
 * sum u^m du (m = 0..3), sum u^i dY (i = 0..2), sum du Y, sum 2 u du Y, from which the host
 * differentiates the normal equations.  d_tmoments may be NULL for nt = 0.
 * d_scratch / d_partial sized by the helpers above.
 * A shard without paths (a rank that holds none of the pre-simulation's chunks) writes zeros to its
 * mcre_irc_presim_slots moments and, with tangents, its mcre_irc_presim_tangent_slots tangent moments, so
 * that callers need not pre-zero them before the all-reduce.  A plan whose regression dates do not fit the
 * moment kernels' shared memory returns -3 before any kernel is launched. */
int64_t mcre_irc_presim_tangent_slots(const mcre_irc_plan *plan);
int mcre_irc_presim(mcre_irc_plan *plan, const mcre_rng *rng, const mcre_shard *shard,
                    void *d_scratch, double *d_partial, double *d_moments, double *d_tmoments, void *stream);

/* Device side of the exposure regression of value-only plans of linear products (takes the place of
 * torch.linalg.lstsq, controller.py:368-374, with the minimum-norm convention of its gelsy driver): solves the 3x3
 * normal equations of every regression date from d_moments (mcre_irc_presim, all-reduced over the ranks) without
 * leaving the device.  unit_set[u] (host): netting-set row of unit u in the main plan, or -1.
 * d_coef_unit: [n_units][n_reg][3], d_coef_sum: [n_reg][n_sets][3] (standardised basis), both device. */
int mcre_irc_solve_coefficients(const mcre_irc_plan *presim_plan, const double *d_moments, const int32_t *unit_set,
                                int32_t n_sets, double *d_coef_unit, double *d_coef_sum, void *stream);
/* Same as mcre_irc_set_coefficients for value-only plans, from DEVICE coefficients [n_expo][n_sets][3]
 * (mcre_irc_solve_coefficients): pre-simulation -> solve -> main simulation then is one stream of kernels. */
int mcre_irc_set_coefficients_device(mcre_irc_plan *plan, const double *d_expo_coef, void *stream);

/* Upload regression coefficients (after the host solved the normal equations). */
int mcre_irc_set_coefficients(mcre_irc_plan *plan, const double *expo_coef /* host, dual[n_expo][n_sets][3] */,
                              void *stream);

/* Upload the exercise-boundary coefficients of the Bermudan units: ex_coef host dual[n_ex][3]
 * (continuation value after each exercise date) and expo_coef host dual[n_expo][n_berm][3]
 * (exposure of a still-alive unit per internal exposure date). */
int mcre_irc_set_exercise_coefficients(mcre_irc_plan *plan, const double *ex_coef, const double *expo_coef,
                                       void *stream);

/* Pre-simulation of a Bermudan unit, forward pass (replaces the path generation + request
 * resolution feeding controller._perform_regression_for_product, controller.py:294-383):
 * spills x [n_reg][n], numeraire [n_reg][n] and the immediate exercise values imm [n_ex][n]
 * (all f64, date-major) for the backward induction of mcre_lsm_step.
 * Plans with tangents (nt > 0): dx [n_reg][nt][n], dN [n_reg][nt][n] and dimm [n_ex][nt][n] follow, for the
 * sensitivities of exposure metrics of exercise products (mcre_lsm_step_tangents). */
int64_t mcre_irc_lsm_scratch_bytes(const mcre_irc_plan *plan, int64_t n_paths);
int mcre_irc_lsm_forward(mcre_irc_plan *plan, const mcre_rng *rng, const mcre_shard *shard, void *d_scratch,
                         void *stream);

/* Path replay for the sensitivities of PFE: under autograd the gradient of the reference's order statistic
 * (pfe_metric.py:59-71) is the pathwise gradient of the selected path.  With a path list set, the next
 * mcre_irc_mainsim on a plan with tangents simulates the listed global path ids (shard: path_begin 0, n_paths =
 * list length) and writes d_tan_spill [path][n_metric][n_sets][nt], the tangents of every unsecured exposure.
 * NULL, NULL switches it off.  mcre_select_locate finds the paths: per row the smallest local index whose value
 * equals d_targets[row] bit for bit (an index >= n_local: not on this rank). */
int mcre_irc_set_path_replay(mcre_irc_plan *plan, const int64_t *d_paths, double *d_tan_spill);
int mcre_select_locate(const double *d_values, int64_t row_stride, int64_t n_local, int32_t n_rows,
                       const double *d_targets, int64_t *d_index, void *stream);

/* Main simulation.  d_acc, d_shift: [mcre_irc_main_slots]; d_spill [n_sets][n_metric][n_paths]
 * or NULL.  Slot layout (NS = n_sets rounded up to 1, 2 or 4; w = 4 + 2*nt):
 *   [n_metric][NS][w] : sum(pos-c), sum((pos-c)^2), sum(neg-c'), sum((neg-c')^2), d pos[nt], d neg[nt]
 *   [NS][w]           : same for (pv, cva) per path totals
 * with c = d_shift[slot] = the value on global path 0 (written by a one-path pilot launch), so
 * mean = c + sum/N and the unbiased variance (metric.py:26-35) has no cancellation. */
int mcre_irc_mainsim(mcre_irc_plan *plan, const mcre_rng *rng, const mcre_shard *shard,
                     double *d_partial, double *d_acc, double *d_shift, double *d_spill, void *stream);

/* ================================================================================
 * Equity family: Black-Scholes (single / multi asset / ModelConfig of BS models), Heston
 * (Euler, Andersen QE with fuzzy branching; several correlated Heston assets as an
 * extension) and Schwartz two-factor, with European / binary / basket / Asian / barrier
 * payoffs; PV and first-order pathwise sensitivities in one fused pass.
 * Replaces:
 *   engine.generate_paths                 src/engine/engine.py:27-123
 *   BlackScholesModel / BlackScholesMulti  src/models/black_scholes.py:44-85, black_scholes_multi.py:63-96
 *   HestonModel (Euler, QE)               src/models/heston.py:99-121, 161-253
 *   SchwartzTwoFactorModel                src/models/schwartz_two_factor.py:147-196
 *   correlated draws z @ L^T              src/models/model.py:38-73, model_config.py:101-221
 *   payoffs                               src/products/european_option.py:45-68, binary_option.py:37-42,
 *                                         basket_option.py:55-78, asian_option.py:51-95, barrier_option.py:65-125
 *   PVMetric + torch.autograd.grad        src/metrics/pv_metric.py:3-18, src/controller/controller.py:609-627
 * One lane per (path, asset); lanes of a path exchange normals / spots by warp shuffle.
 * ============================================================================== */
enum { MCRE_EQ_BS = 0, MCRE_EQ_HESTON = 1, MCRE_EQ_SCHWARTZ = 2 };
#define MCRE_EQ_MAX_SETS 4
/* product kinds / event flags of the tables below */
enum { MCRE_EQ_EUROPEAN = 0, MCRE_EQ_BINARY = 1, MCRE_EQ_BASKET = 2, MCRE_EQ_ASIAN = 3, MCRE_EQ_BARRIER = 4,
       MCRE_EQ_EXERCISE = 5 /* Bermudan / American, src/products/bermudan_option.py:93-188 */ };
#define MCRE_EQ_EV_OBSERVE 1
#define MCRE_EQ_EV_PAY 2
#define MCRE_EQ_EV_FIRST 4
#define MCRE_EQ_EV_EXERCISE 8

typedef struct {
  int32_t kind;          /* MCRE_EQ_*: every asset of a launch is of this kind                       */
  int32_t scheme;        /* MCRE_SCHEME_*                                                            */
  int32_t nt;            /* tangents per lane: 0, or the kind's parameter count (BS 3, Heston 7, Schwartz 6), or 9 =
                            second order on Black-Scholes lanes: 3 first + 6 second derivatives (upper triangle,
                            row-major), present values only; the tangent slots of the result hold all 9          */
  int32_t smoothing;     /* Heston fuzzy indicators on (the reference ties this to differentiate)    */
  int32_t n_assets, noise_dim, n_uniform;
  const double *asset_par;      /* [n_assets][8] lane parameters: BS spot, sigma, rate | Heston spot, sigma, rate,
                                   rho, kappa, theta, v0 | Schwartz rate, kappa_s, sigma_s, mu_l, sigma_l, rho   */
  const int32_t *asset_noise;   /* [n_assets][2] noise columns the asset consumes (second: -1 if none)  */
  const int32_t *asset_uniform; /* [n_assets] index of the asset's QE uniform within a sub-step          */
  const int32_t *col_asset;     /* [noise_dim] asset owning noise column j                               */
  const int32_t *col_elem;      /* [noise_dim] 0 / 1: first or second normal of that asset               */
  int32_t n_sub, n_dates, n_pre_dates, n_chol;
  const double *step_dt;        /* [n_sub] time2 - time1                                                 */
  const double *step_sq;        /* [n_sub] sqrt(dt) (EULER / QE) or sqrt(nominal dt) (ANALYTICAL)        */
  const int32_t *step_date;     /* [n_sub] simulation date completed by the sub-step or -1               */
  const int32_t *step_chol;     /* [n_sub] index into chol / chol_dual                                   */
  const double *step_aux;       /* [n_sub][n_assets] Schwartz: log F0(time2)                             */
  const double *init_aux;       /* [n_assets] Schwartz: log F0(calibration date)                         */
  int32_t corr_mode;            /* 0 identity, 1 chol_dual (one asset, two noise sources), 2 chol        */
  const double *chol;           /* [n_chol][noise_dim][noise_dim] lower factor of the joint correlation  */
  const double *chol_dual;      /* dual[n_chol][4]: L00, L01, L10, L11 with lane-local tangents          */
  const int32_t *date_ev_off;   /* [n_dates+1] CSR offsets of the product events per simulation date     */
  const int32_t *ev_prod;       /* [n_ev] product index                                                  */
  const int32_t *ev_flags;      /* [n_ev] MCRE_EQ_EV_*                                                   */
  int32_t n_prod;
  const double *prod;           /* [n_prod][16]: kind, set, strike, sign(+1 call / -1 put), 1/numeraire,
                                   d(1/numeraire)/d rate, flags(bit0 geometric, bit1 control variate, bit2 Brownian-bridge barrier),
                                   control-variate constant, payment amount, barrier1, type1 (1 UO, 2 DO, 3 UI,
                                   4 DI), barrier2, type2 (0: none), n observations, tracker slot, reserved  */
  const double *prod_w;         /* [n_prod][n_assets] weights of the composite underlying                 */
  int32_t n_sets;
  /* exercise products (Bermudan / American: 1 right, bermudan_option.py:93-188; FlexiCall: up to 3 rights,
   * flexicall.py:56-160; prod[13] = number of rights, the tracker holds the rights left): per event (same
   * indexing as ev_prod) 16 doubles: [0..2] c0, c1, c2 of the continuation value of state 1 in
   * u = (x - shift) * scale, [3] shift, [4] scale, [5] 1/numeraire(t), [6] d(1/numeraire)/d rate, [7] last-date
   * flag, [14] strike of this exercise date, [16 + 3 (s - 2) ..] coefficients of states s = 2 .. 6 (32 doubles per event);
   * prod_x [n_prod][n_assets]: weights picking the explanatory variable x (spot of the option's asset). */
  const double *ev_data;
  const double *prod_x;
  /* exposure profiles (n_expo = 0: PV only).  Per internal exposure date and product an exposure op, 32 doubles:
   * type 1 = analytic Black-Scholes value of a European option (european_option.py:123-145): [1, time to maturity,
   * 1/numeraire(t), ...]; type 2 = regression proxy c(u) / numeraire (controller.py:438-447), u = (x - shift) scale,
   * x = spot picked by prod_x: [2, c0, 1/numeraire(t), c1, c2, shift, scale, pad]; type 3 = the same for an exercise
   * product, with the coefficients of its current state (rights left; [16 + 3 (s - 2) ..] for states s = 2 .. 6; no
   * exposure in state 0); type 0 = none.
   * Netting-set terms as in mcre_irc_desc.  acc_flags: MCRE_ACC_POS /
   * NEG / SPILL.  Adds [n_metric][NS][4] = sum(pos-c), sum((pos-c)^2), sum(neg-c'), sum((neg-c')^2) to the slots. */
  int32_t n_expo, n_metric, acc_flags;
  const int32_t *date_expo;     /* [n_dates] internal exposure index or -1 */
  const int32_t *date_metric;   /* [n_dates] metric-date index or -1       */
  const double *xp;             /* [n_expo][n_prod][32]                    */
  const double *set_threshold;  /* [n_sets]                                */
  const int32_t *set_flags;     /* [n_sets] bit0 collateralised            */
  const int32_t *set_lag;       /* [n_sets][n_metric] exposure-index lag of the collateral date, -1: none */
} mcre_eq_desc;

typedef struct mcre_eq_plan mcre_eq_plan;
int mcre_eq_create(const mcre_eq_desc *desc, mcre_eq_plan **out);
void mcre_eq_destroy(mcre_eq_plan *plan);
/* Accumulator slots (NS = n_sets rounded up to 1, 2 or 4):
 *   [NS][3]              : sum(cf - c), sum((cf - c)^2), sum_p payoff_p * d(1/N_p)/d rate
 *   [n_assets][NS][nt]   : lane-local tangents of sum_p payoff_p / N_p
 * with c = d_shift[set] = the value on global path 0 (pilot launch). */
int64_t mcre_eq_slots(const mcre_eq_plan *plan);
int mcre_eq_mainsim(mcre_eq_plan *plan, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                    double *d_acc, double *d_shift, double *d_spill /* [n_sets][n_metric][n_paths] or NULL */,
                    void *stream);
/* Book splitting: a netting set with more path-dependent / exercise products than one launch can track
 * (4 value-only, 2 with tangents) is evaluated in several launches over the same Philox streams; each launch
 * ADDS its per-path discounted cashflow totals to d_accum [n_sets][n_paths] (NULL: off) and mcre_sum_stats
 * turns the accumulated per-path PVs into the sums of metric.py:26-35.  Replaces the reference's loop over
 * the products of a netting set (controller.py:506-563) for books of thousands of products
 * (tests/pv_tests/pv_performance_large_netting_set.py). */
int mcre_eq_set_pv_accumulator(mcre_eq_plan *plan, double *d_accum);
/* Brownian-bridge barrier monitoring (barrier_option.py:138-222; product flag bit 2, value-only plans): the
 * observation events of such a product carry in their ev_data row [0] the Philox block of their (product,
 * interval) uniforms (stream kind 2; element 0 / 1 = first / second barrier), [1] -2 / (sigma^2 maturity / n_obs),
 * [2] the interval index.  In RNG compatibility mode the reference's numpy uniforms replace Philox:
 * d_u [tracker slot][barrier][n_paths_total][stride] (NULL: Philox). */
int mcre_eq_set_bridge_uniforms(mcre_eq_plan *plan, const double *d_u, int32_t stride);
/* The same for exposure profiles: each launch ADDS the netted exposure of its products to
 * d_accum [n_sets][n_expo][n_paths] (and evaluates no netting terms or metrics); mcre_eq_unsecured_exposures then
 * applies threshold / MPoR collateral (netting_set.py:48-72, 136-184) to one set's accumulated exposures:
 * d_expo [n_expo][n_paths] -> d_out [n_metric][n_paths], metric_expo[m] = exposure index of metric date m,
 * lag[m] = exposure indices back to its collateral date (-1: none).  Host index arrays. */
int mcre_eq_set_exposure_accumulator(mcre_eq_plan *plan, double *d_accum);
/* Black-Scholes plans with tangents in accumulating mode: the lane-local tangents of the netted exposures are ADDED to
 * d_accum_tan [n_sets][n_expo][n_assets][nt][n_paths] (nt = 3: spot, volatility, rate of the lane's asset).  With the
 * per-path tangents of the other product family of a hybrid book (mcre_irc_set_path_replay) they feed
 * mcre_exposure_tangent_sums.  NULL: off. */
int mcre_eq_set_exposure_tangent_accumulator(mcre_eq_plan *plan, double *d_accum_tan);
/* Pathwise sensitivities of exposure metrics from per-path exposures and their tangents (what torch.autograd gives
 * through netting_set.py:48-72, 136-184, epe_metric.py / ene_metric.py / cva_metric.py:62-100 for weights that do not
 * depend on the parameters): d_expo [n_expo][n], d_tan [n_par][n_expo][n]; per metric date m and parameter g
 *   U = unsecured exposure (threshold / collateral like mcre_eq_unsecured_exposures), dU its tangent,
 *   d_out [n_metric][n_par][3] = sum 1{U > 0} dU, sum 1{U < 0} dU, sum w_m 1{U > 0} dU   (w: host [n_metric]).
 * Fixed-order chunk partials d_partial [ceil(n / chunk_paths)][n_metric * n_par * 3] + tree. */
int mcre_exposure_tangent_sums(const double *d_expo, const double *d_tan, int64_t n_paths, int32_t n_expo, int32_t n_par,
                               int32_t n_metric, const int32_t *metric_expo, const int32_t *lag, int32_t collateralised,
                               double threshold, const double *weights, int32_t chunk_paths, double *d_partial,
                               double *d_out, void *stream);
/* The same with default weights that differ per path (stochastic intensity, cva_metric.py:62-100 under autograd):
 * d_w_paths [n_metric][n] replaces `weights`, slot 2 = lgd * sum w_m(path) 1{U > 0} dU.  With d_w_tan
 * [n_metric][n_wtan][n] (mcre_eq_credit_weight_tangents) the output has n_par + n_wtan rows per metric date,
 * d_out [n_metric][n_par + n_wtan][3]; row n_par + j: slot 2 = lgd * sum relu(U) d w_m / d (credit parameter j), the
 * part of the CVA gradient that flows through the weights; slots 0 / 1 of those rows are 0. */
int mcre_exposure_tangent_sums_paths(const double *d_expo, const double *d_tan, int64_t n_paths, int32_t n_expo, int32_t n_par,
                                     int32_t n_metric, const int32_t *metric_expo, const int32_t *lag, int32_t collateralised,
                                     double threshold, const double *d_w_paths, double lgd, const double *d_w_tan,
                                     int32_t n_wtan, int32_t chunk_paths, double *d_partial, double *d_out, void *stream);
int mcre_eq_unsecured_exposures(const double *d_expo, int64_t n_paths, int32_t n_metric, const int32_t *metric_expo,
                                const int32_t *lag, int32_t collateralised, double threshold, double *d_out, void *stream);
/* d_out [n_rows][2] = sum(v - c), sum((v - c)^2) per row of d_x [n_rows][n], c = d_shift[row], v = x (mode 0),
 * max(x, 0) (mode 1) or -max(-x, 0) (mode 2); fixed-order chunk partials (d_partial:
 * [ceil(n / chunk_paths)][n_rows][2]) + tree, like the simulation kernels. */
int mcre_sum_stats(const double *d_x, int64_t n, int32_t n_rows, int32_t chunk_paths, const double *d_shift,
                   int32_t mode, double *d_partial, double *d_out, void *stream);

/* Pre-simulation pass of the regression-proxy exposures (replaces the path generation + request resolution +
 * cashflow roll feeding controller._perform_regression_for_product, controller.py:294-351, for the equity
 * products, which pay once): the same fused kernel run on the pre-simulation stream spills, date-major,
 * d_x [n_expo][n_assets][n_paths] (spot of every asset per exposure date) and d_cf [n_prod][n_paths] (discounted
 * cashflow of every product rounded to float32 like the reference's accumulators).  The moments / solve per
 * (product, date) then go through mcre_lsm_step without an exercise update. */
int mcre_eq_presim(mcre_eq_plan *plan, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                   double *d_shift, double *d_x, float *d_cf, void *stream);
/* Sensitivities of exposure profiles of equity books (controller.py:609-627 on EPE / ENE / CE / EEPE; Black-Scholes
 * plans with nt = 3).  The accumulator gains [n_metric][n_assets][NS][2][nt] lane-local tangents of sum relu(E) and
 * sum -relu(-E) after the exposure sums (counted by mcre_eq_slots).  Analytic Black-Scholes exposures
 * (european_option.py:123-145) need nothing else; regression proxies need the tangents of their coefficients:
 *  - mcre_eq_presim_tangents: the pre-simulation spill pass on a plan with tangents also writes
 *    d_dx [n_expo][n_assets][nt][n_paths] and d_dcf [n_prod][nt][n_paths] (tangents of the spots and of the deflated
 *    cashflows with respect to the parameters of the product's asset), which feed mcre_lsm_step_tangents;
 *  - mcre_eq_set_exposure_coef_tangents: host xp_tan [n_expo][n_prod][3][nt], d(c0, c1, c2)/d(lane parameters) from the
 *    differentiated normal equations (the reference keeps torch.linalg.lstsq in the autograd graph,
 *    controller.py:368-383); copied to the device;
 *  - mcre_eq_set_exercise_exposure_coef_tangents: the same for exercise products (exposure type 3): host
 *    [n_expo][n_prod][MCRE_LSM_MAX_RIGHTS][3][nt], d(c0, c1, c2)/d(lane parameters) of the continuation value of state
 *    s = rights left at row s - 1 (from the tangent backward induction, mcre_lsm_step_states_tangents); rows of other
 *    products are ignored.  The exposure of state s is (c0 + u (c1 + u c2)) / N(t) on duals, 0 in state 0; the state
 *    itself carries no tangent.  Copied to the device. */
/* Hybrid ModelConfig of Black-Scholes market models + the CIR++ credit model of a counterparty (the reference's
 * tests/exposure_tests/cva_perfprmance_large_netting_set.py): the fused equity kernel also steps the intensity
 * (cirpp.py:155-198, Euler with full truncation or the deterministic mode) on the noise column `noise_col` of the joint
 * draw, correlated with the equity draws through chol_row [noise_dim] = the credit row of the Cholesky factor of the
 * joint correlation (model_config.py:101-142), and accumulates per path
 *     CVA = lgd * sum_{k < n_metric-1} relu(E_k) exp(-logB_lambda(t_k)) (1 - C_k exp(-B_k y_k))     (cva_metric.py:62-100)
 * for the sets with set_cva != 0.  step_cir [n_sub][2] = psi(t1), unused (deterministic: lambda(t1), lambda(t2));
 * cva_coef [n_metric][2] = (C_k, B_k).  Adds [NS][2] = sum(cva - c), sum((cva - c)^2) at the end of the accumulator
 * (counted by mcre_eq_slots).  Value-only plans; host arrays, copied. */
typedef struct {
  int32_t deterministic, noise_col;
  double kappa, theta, sigma, y0, lgd;
  const double *step_cir, *chol_row, *cva_coef;
  const int32_t *set_cva;
} mcre_eq_credit;
int mcre_eq_set_credit(mcre_eq_plan *plan, const mcre_eq_credit *credit);
/* CVA of books split over several launches: the launch that carries the credit factor also writes the default
 * weights d_w [n_metric][n_paths] = exp(-logB_lambda(t_k)) (1 - C_k exp(-B_k y_k)) (0 on the last date); once every
 * launch has added its exposures and mcre_eq_unsecured_exposures has netted them, mcre_eq_cva_paths gives the per-path
 * d_out [n_paths] = lgd * sum_k relu(unsec_k) w_k, finished by mcre_sum_stats. */
int mcre_eq_set_cva_weight_spill(mcre_eq_plan *plan, double *d_w);
/* Tangents of those per-path default weights w.r.t. the CIR++ model's own parameters (kappa, theta, sigma, y0) under a
 * stochastic intensity (cirpp.py:174-198, 246-285 under torch.autograd): the credit factor is replayed from the plan's
 * grid and the same draws (column noise_col of the joint draw through chol_row) with its Euler recursion differentiated
 * by hand.  `credit` as for mcre_eq_set_credit (the plan itself need not carry the factor); dpsi host [n_sub][4] =
 * d psi(t1) / d parameters, dcoef host [n_metric][2][4] = d (C_k, B_k) / d parameters.
 * d_w_tan [n_metric][4][shard->n_paths] (0 on the last date). */
int mcre_eq_credit_weight_tangents(mcre_eq_plan *plan, const mcre_eq_credit *credit, const double *dpsi, const double *dcoef,
                                   const mcre_rng *rng, const mcre_shard *shard, double *d_w_tan, void *stream);
int mcre_eq_cva_paths(const double *d_unsec, const double *d_w, int64_t n_paths, int32_t n_metric, double lgd,
                      double *d_out, void *stream);
int mcre_eq_presim_tangents(mcre_eq_plan *plan, const mcre_rng *rng, const mcre_shard *shard, double *d_partial,
                            double *d_shift, double *d_x, float *d_cf, double *d_dx, double *d_dcf, void *stream);
int mcre_eq_set_exposure_coef_tangents(mcre_eq_plan *plan, const double *xp_tan);
int mcre_eq_set_exercise_exposure_coef_tangents(mcre_eq_plan *plan, const double *tan);

/* ================================================================================
 * Longstaff-Schwartz backward induction on spilled pre-simulation arrays: one call per
 * regression date, latest first.  Replaces the roll of compute_normalized_cashflows over
 * [t_next, last) with its float32 accumulators and the tall lstsq of
 * controller._perform_regression_for_product (controller.py:312-374) for single-right
 * exercise products (state 0 = exercised carries no value):
 *   1. if d_imm != NULL: exercise update at the product date i that enters the window,
 *        cont = c0 + u (c1 + u c2), u = (x_i - shift_i) scale_i   (coef_i == NULL: cont = 0)
 *        ex = imm_i > cont;  V <- fp32(fp32(ex ? imm_i / N_i : 0) + (ex ? 0 : V))
 *   2. moments of regression date k with response Y = N_k * V:
 *        d_moments[0..4] = sum u^0..u^4, d_moments[5..7] = sum Y u^0..u^2, u = (x_k - shift_k) scale_k
 * All arrays are device arrays of length n (this rank's pre-simulation paths); d_value is
 * the running fp32 tail value per path (zero-initialised by the caller).  Per-chunk partial
 * sums + fixed tree, like the other reductions; multi-GPU callers all-reduce d_moments.
 * ============================================================================== */
int mcre_lsm_step(const double *d_xk, const double *d_nk, double shift_k, double scale_k,
                  const double *d_xi, const double *d_ni, const double *d_imm, const double *coef_i /* host[3] or NULL */,
                  double shift_i, double scale_i, float *d_value, int64_t n, int32_t chunk_paths,
                  double *d_partial, double *d_moments, void *stream);
/* Step 2 of mcre_lsm_step (no exercise update, constant numeraire nk) for MANY (product, regression date) pairs in
 * one launch: d_moments [n_jobs][8], bit-identical to the per-pair calls; d_partial [ceil(n / chunk_paths)][n_jobs][8].
 * For the regression proxies of books of thousands of products (controller.py:294-383 per product and exposure date).
 * `jobs` is a host array; x and v are device arrays of length n. */
typedef struct { const double *x; const float *v; double nk, shift, scale; } mcre_lsm_job;
int mcre_lsm_moments_batch(int64_t n_jobs, const mcre_lsm_job *jobs, int64_t n, int32_t chunk_paths,
                           double *d_partial, double *d_moments, void *stream);
/* mcre_lsm_step_states for MANY products in one launch (the lock-step backward inductions of a book: one job per
 * product and round): d_moments [n_jobs][23] (row layout of the 6-rights step, unused tail zero), bit-identical to the
 * per-product calls; d_partial [ceil(n / chunk_paths)][n_jobs][23].  coef: [6][3] continuation coefficients of the
 * product date (has_coef = 0: none); imm NULL: no exercise update.  `jobs` is a host array of device pointers. */
#define MCRE_LSM_MAX_RIGHTS 6   /* exercise rights of a product (FlexiCall); state = rights left */
typedef struct {
  int32_t n_rights, has_coef;
  const double *xk, *nk;
  double shift_k, scale_k;
  const double *xi, *ni, *imm;
  double coef[3 * MCRE_LSM_MAX_RIGHTS];
  double shift_i, scale_i;
  float *value;
} mcre_lsm_step_job;
int mcre_lsm_step_batch(int64_t n_jobs, const mcre_lsm_step_job *jobs, int64_t n, int32_t chunk_paths,
                        double *d_partial, double *d_moments, void *stream);
/* The same with n_rights = 1..6 exercise rights (FlexiCall, src/products/flexicall.py:56-160): the product state
 * is the number of rights left, d_value is [n_rights][n] (state s at row s-1; state 0 carries nothing),
 * coef_i host [n_rights][3] (continuation of state s at product date i), d_moments [5 + 3 n_rights]:
 *   ex_s = imm_i + cont_i(s-1) > cont_i(s), cont(0) = 0;  V_s <- fp32(fp32(ex_s ? imm_i/N_i : 0) + (ex_s ? V_{s-1} : V_s))
 * n_rights = 1 is mcre_lsm_step. */
int mcre_lsm_step_states(int32_t n_rights, const double *d_xk, const double *d_nk, double shift_k, double scale_k,
                         const double *d_xi, const double *d_ni, const double *d_imm, const double *coef_i,
                         double shift_i, double scale_i, float *d_value, int64_t n, int32_t chunk_paths,
                         double *d_partial, double *d_moments, void *stream);

/* Single-right step like mcre_lsm_step_states, with the continuation coefficients of product date i read from
 * DEVICE memory (d_coef_i: 3 doubles, or NULL), and the 3x3 solve of one regression date on the device
 * (d_moments: the 8 moments, all-reduced over the ranks; d_coef: 3 doubles; the minimum-norm convention of
 * torch.linalg.lstsq's gelsy driver, controller.py:368-374): the backward induction of one Bermudan option is then
 * a stream of kernels without a per-date read-back. */
int mcre_lsm_step_dev(const double *d_xk, const double *d_nk, double shift_k, double scale_k, const double *d_xi,
                      const double *d_ni, const double *d_imm, const double *d_coef_i, double shift_i, double scale_i,
                      float *d_value, int64_t n, int32_t chunk_paths, double *d_partial, double *d_moments, void *stream);
int mcre_lsm_solve_dev(const double *d_moments, double *d_coef, void *stream);

/* Tangent companion of mcre_lsm_step (one exercise right), called after it for the same regression date: applies
 * the same hard exercise decision to the running pathwise tangents d_dvalue [nt][n] of the deflated value,
 *   dV <- ex ? (dimm_i - (imm_i / N_i) dN_i) / N_i : dV,
 * and accumulates d_tmoments [nt][9] = sum u^m du (m = 0..3), sum u^i dY (i = 0..2), sum du Y, sum 2 u du Y with
 * Y = N_k V, dY = dN_k V + N_k dV, from which the host differentiates the normal equations (the reference keeps
 * torch.linalg.lstsq inside the autograd graph, controller.py:368-383).  d_dxk, d_dnk, d_dni, d_dimm: [nt][n]. */
int mcre_lsm_step_tangents(int32_t nt, const double *d_xk, const double *d_nk, const double *d_dxk, const double *d_dnk,
                           double shift_k, double scale_k, const double *d_xi, const double *d_ni, const double *d_imm,
                           const double *d_dni, const double *d_dimm, const double *coef_i, double shift_i, double scale_i,
                           const float *d_value, double *d_dvalue, int64_t n, int32_t chunk_paths, double *d_partial,
                           double *d_tmoments, void *stream);
/* The same for 1..6 exercise rights, called after mcre_lsm_step_states for the same regression date (n_rights = 1:
 * exactly mcre_lsm_step_tangents).  Recomputes every state's decision ex_s = imm_i + cont(s-1) > cont(s) with the
 * expressions of the value step and updates the running tangents d_dvalue [n_rights][nt][n] from their values before
 * the update:  dV_s <- ex_s ? (dimm_i - (imm_i / N_i) dN_i) / N_i + dV_{s-1} : dV_s  (dV_0 = 0).  coef_i: host
 * [n_rights][3] or NULL; d_value: the value step's [n_rights][n].  d_tmoments [nt][4 + 5 n_rights]: sum u^m du
 * (m = 0..3), then per state s at 4 + 5 s: sum dY, u dY, u^2 dY, du Y, 2 u du Y with Y = N_k V_s. */
int mcre_lsm_step_states_tangents(int32_t n_rights, int32_t nt, const double *d_xk, const double *d_nk,
                                  const double *d_dxk, const double *d_dnk, double shift_k, double scale_k,
                                  const double *d_xi, const double *d_ni, const double *d_imm, const double *d_dni,
                                  const double *d_dimm, const double *coef_i, double shift_i, double scale_i,
                                  const float *d_value, double *d_dvalue, int64_t n, int32_t chunk_paths,
                                  double *d_partial, double *d_tmoments, void *stream);

/* LSM pre-simulation arrays of an exercise product on equity underlyings, gathered date-major from
 * materialised pre-simulation paths (mcre_generate_paths with seed 42; the pre-simulation is a small
 * fraction of the run): x[k][n] explanatory spot and numeraire[k][n] per regression date k,
 * imm[i][n] = max(sign (U - K_i), 0) per exercise date i with U = sum_j w_j spot_j and K_i = ex_strike[i]
 * (NULL: the same strike on every date).  Spots are state columns, exponentiated where the model keeps
 * log-spot (Heston, Schwartz).  Host arrays unless d_*. */
int mcre_lsm_prepare_equity(const double *d_paths, int64_t n_paths, int32_t n_dates, int32_t state_dim,
                            int32_t n_reg, const int32_t *reg_date, const double *reg_numeraire,
                            int32_t n_ex, const int32_t *ex_date, int32_t x_col, int32_t x_is_log,
                            int32_t n_under, const int32_t *under_col, const double *under_w,
                            const int32_t *under_is_log, double strike, const double *ex_strike, double sign,
                            double *d_x, double *d_n, double *d_imm, void *stream);
/* Pathwise tangents of those arrays (single-asset exercise products), from the tangent spill of the pre-simulation
 * d_dx [n_rows][n_assets][nt][n_paths] (mcre_eq_presim_tangents on a plan whose exposure dates are the spill dates):
 * d_dxs [n_reg][nt][n] = the spill row reg_row[k] of asset x_asset; d_dnum [n_reg][nt][n] = reg_dnum[k] in parameter
 * rate_slot, 0 elsewhere (the numeraire is deterministic); d_dimm [n_ex][nt][n] = sign * 1{imm > 0} * the spill row
 * ex_row[i] of asset u_asset.  d_imm: the value arrays of mcre_lsm_prepare_equity.  Host index tables. */
int mcre_lsm_prepare_equity_tangents(const double *d_dx, int64_t n_paths, int32_t n_assets, int32_t nt, int32_t n_reg,
                                     const int32_t *reg_row, const double *reg_dnum, int32_t rate_slot, int32_t x_asset,
                                     int32_t n_ex, const int32_t *ex_row, int32_t u_asset, double sign,
                                     const double *d_imm, double *d_dxs, double *d_dnum, double *d_dimm, void *stream);

/* ================================================================================
 * Exact order statistics per row (PFE), replaces torch.sort + index in
 * PFEMetric.evaluate_numerically, src/metrics/pfe_metric.py:59-71.
 * MSB-first radix select on the order-preserving 64-bit image of the doubles, 8 bits
 * per pass.  Multi-GPU: the caller all-reduces d_hist between count and scan.
 * ============================================================================== */
typedef struct mcre_select_plan mcre_select_plan;
int mcre_select_create(int32_t n_rows, int32_t n_ranks_per_row, mcre_select_plan **out);
void mcre_select_destroy(mcre_select_plan *p);
/* ranks: host [n_rows][n_ranks_per_row] global 0-based ranks (may repeat). */
int mcre_select_begin(mcre_select_plan *p, const int64_t *ranks, void *stream);
/* one pass = count (fills d_hist [n_rows][n_ranks_per_row][256] uint64) then scan. */
int mcre_select_count(mcre_select_plan *p, const double *d_values, int64_t row_stride, int64_t n_local,
                      int32_t pass, uint64_t *d_hist, void *stream);
/* Optional shortcut after `passes_done` >= 2 count + scan rounds: compacts, per row, the elements that still match
 * one of the row's prefixes; later mcre_select_count calls read those instead of the full rows (rows with more
 * than n_local / 8 candidates keep reading everything).  Exact: only elements that cannot be a wanted order
 * statistic are dropped. */
int mcre_select_compact(mcre_select_plan *plan, const double *d_values, int64_t row_stride, int64_t n_local,
                        int32_t passes_done, void *stream);
int mcre_select_scan(mcre_select_plan *p, int32_t pass, const uint64_t *d_hist, void *stream);
/* after 8 passes: d_out [n_rows][n_ranks_per_row] the selected values. */
int mcre_select_finish(mcre_select_plan *p, double *d_out, void *stream);

/* Correlated joint noise of a ModelConfig, materialised: d_out [n_sub][n_paths][dim] = L z per (sub-step, global path
 * 0 .. n_paths-1) with z the Philox stream of `rng` (normal number sub-step * dim + column of the path) or its injected
 * draws, and chol [dim][dim] (host) the lower Cholesky factor of the joint correlation (model.py:46-73,
 * model_config.py:101-142).  For netting sets that mix products of model families whose fused kernels run separately
 * on columns of one joint draw (mcre/hybrid.py); the fused kernels themselves never materialise noise. */
int mcre_correlated_normals(const mcre_rng *rng, int32_t n_sub, int32_t dim, const double *chol, int64_t n_paths,
                            double *d_out, void *stream);

/* ================================================================================
 * Gas storage on a two-factor log-price model
 * replaces Storage.compute_normalized_cashflows (src/products/storage.py:215-308: inventory moves of the three
 * actions, interpolated continuation grid, arg-max, realised cashflow) and the controller loops that drive it:
 * the backward induction of _perform_regression_for_product (src/controller/controller.py:294-383) and the PV branch
 * of _evaluate_product (:399-410), for SchwartzTwoFactorModel (src/models/schwartz_two_factor.py:147-196).
 * ============================================================================== */
#define MCRE_STORAGE_MAX_KNOTS 8   /* knots per injection / withdrawal rate curve                      */
#define MCRE_STORAGE_RECORD 48     /* doubles per action-date record                                    */
#define MCRE_STORAGE_MAX_STATES 16 /* inventory grid states                                             */
#define MCRE_STORAGE_STEP 24       /* doubles per sub-step record                                       */
#define MCRE_STORAGE_MAX_NOISE 8   /* normals per sub-step of the price model's joint draw              */
#define MCRE_STORAGE_MAX_BASIS 6   /* regression basis functions (polynomial degree + 1)                */
#define MCRE_STORAGE_TAN 7         /* doubles per (sub-step, tangent slot) record of step_tan           */

typedef struct {
  int32_t n_sub;            /* sub-steps of the simulation grid (engine.py:36-123)                         */
  int32_t n_dates;          /* action dates of the storage                                                 */
  int32_t n_pre_dates;      /* leading action dates reached without stepping (at the calibration date)     */
  int32_t n_states;         /* inventory grid states                                                       */
  int32_t n_basis;          /* regression basis functions                                                  */
  double log_spot0;         /* log of the forward curve at the calibration date                            */
  const double *step;       /* [n_sub][MCRE_STORAGE_STEP]: [0] a, [1] k, [2] dt, [3] m, [4] cx, [5] cy, [6] log F(t2),
                               [7] non-zero: Black-Scholes EULER step x' = x + log1p(m + cx w0), log S = log F + x'
                               (m = rate dt, cx = sigma sqrt(dt); black_scholes.py:69-85), [8 + j] bx_j, [16 + j] by_j
                               (j < noise_dim):
                                 w0 = sum_j bx_j z_j, w1 = sum_j by_j z_j   (the model's rows of the joint draw z @ L^T)
                                 x' = (a x - (k x) dt) + cx w0;  y' = (y + m) + cy w1;  log S = log F(t2) + x' + y'
                               Schwartz ANALYTICAL: a = exp(-kappa dt), k = 0, cx = cy = 1, b = rows of the Cholesky
                               factor of the step covariance (schwartz_two_factor.py:124-168); EULER: a = 1, k = kappa,
                               cx / cy = vol sqrt(dt), b = rows of the Cholesky factor of the correlation (:170-196);
                               Black-Scholes single / multi-asset, ANALYTICAL: a = 1, k = 0, cx = 1, cy = 0, m = (rate -
                               sigma^2 / 2) dt, bx = the asset's row of the Cholesky factor of the step covariance of
                               all assets (black_scholes.py:50-67, black_scholes_multi.py:63-79), log F = log spot  */
  const int32_t *step_date; /* [n_sub] action-date index completed by the sub-step, or -1                  */
  const double *date_rec;   /* [n_dates][MCRE_STORAGE_RECORD] per action date:
                               0 vmin of the date's band, 1 inventory per state index, 2 / 3 vmin / vmax of the next
                               date's band, 4 state index per unit inventory on the next date (0: degenerate band),
                               5 period to the next action date, 6 / 7 injection / withdrawal cost, 8 / 9 number of
                               injection / withdrawal knots, 10 non-zero on the last action date (no continuation),
                               16.. injection knots (level, rate) x 8, then withdrawal knots x 8
                               (storage_helpers.py:56-127, storage.py:114-190)                              */
  const double *numeraire;  /* [n_dates] numeraire at the action dates                                     */
  int32_t noise_dim;        /* normals per sub-step of the model's joint draw: 2 (Schwartz two-factor), 1 (Black-Scholes),
                               number of assets (Black-Scholes multi-asset), <= MCRE_STORAGE_MAX_NOISE         */
  int32_t n_tan;            /* 0, or 3 / 4 / 6: pathwise PV sensitivities with respect to that many tangent slots of
                               the storage (spot, volatility, rate of a Black-Scholes asset [, rate of the numeraire
                               model]; the six Schwartz parameters), which the caller maps to the model's parameters */
  const double *step_tan;   /* [n_sub][n_tan][MCRE_STORAGE_TAN] d(A, B00, M, B10, B11, log F, Bw)/d slot of the effective
                               recursion x' = A x + B00 z0, y' = y + M + B10 z0 + B11 z1 (A = a - k dt, B00 = cx bx_0,
                               B10 = cy by_0, B11 = cy by_1), where d(cx w0) also gains dBw w0 (Bw: d log of the asset's
                               row of the joint Cholesky factor; 0 for the one- and two-factor stand-alone steps);
                               Black-Scholes EULER steps: dx' = dx + (dM + dBw w0) / (1 + m + cx w0) with dM = d m,
                               dBw = d cx; entry [0][.][5] also holds d log F(t0)                                */
  const double *dlog_num;   /* [n_dates][n_tan] d log numeraire / d slot                                        */
  /* ---- exposure dates (controller.py:412-447); n_expo = 0: none ---- */
  int32_t n_expo;           /* internal exposure dates                                                         */
  int32_t n_pre_expo;       /* leading exposure dates at the calibration date                                  */
  const int32_t *step_expo; /* [n_sub] exposure index completed by the sub-step, or -1                         */
  const double *expo_numeraire; /* [n_expo]                                                                    */
} mcre_storage_desc;

typedef struct mcre_storage_plan mcre_storage_plan;
int mcre_storage_create(const mcre_storage_desc *desc, mcre_storage_plan **out);
void mcre_storage_destroy(mcre_storage_plan *plan);
/* Pre-simulation forward pass: d_spot [n_dates][shard->n_paths] = spot at every action date; d_spot_expo
 * [n_expo][n_paths] = spot at every exposure date (NULL: not wanted). */
int mcre_storage_spots(mcre_storage_plan *plan, const mcre_rng *rng, const mcre_shard *shard, double *d_spot,
                       double *d_spot_expo, void *stream);
/* One date of the backward induction (controller.py:322-352) for all n paths and all grid states:
 * d_value [n_states][n] holds the normalised value from the next action date on, per state entering it, and is
 * replaced by the same quantity for `date`: float32(best action's cashflow / numeraire) + the float64 tail interpolated
 * at the state the action leads to.  d_coef [2 + n_states * n_basis] (device) = centre, inverse scale and per-state
 * coefficients of the continuation polynomial in u = (spot - centre) * inverse scale at `date` (raw basis of the
 * reference: centre 0, scale 1); ignored on the last action date.  d_spot_row [n] = spot at `date`. */
int mcre_storage_backward(mcre_storage_plan *plan, int32_t date, const double *d_coef, const double *d_spot_row,
                          double *d_value, int64_t n, void *stream);
/* Regression moments of one regression date - an action date or an exposure date in front of the action date whose value
 * grid d_value holds (the Gram / right-hand-side sums of controller.py:353-374 for y_s = numeraire x d_value[s], numeraire
 * and d_spot_row taken at the regression date): d_out [n_states * n_basis + 2 n_basis - 1] = sum u^k y_s (s major), then sum u^q, q < 2 n_basis - 1;
 * fixed-order chunk partials d_partial [ceil(n / chunk_paths)][slots] + tree. */
int64_t mcre_storage_moment_slots(const mcre_storage_plan *plan);
int mcre_storage_moments(mcre_storage_plan *plan, double numeraire, double centre, double inv_scale, const double *d_spot_row,
                         const double *d_value, int64_t n, int32_t chunk_paths, double *d_partial, double *d_out,
                         void *stream);
/* Minimum-norm solution of the normal equations of one regression date on the device: d_mom = the (all-reduced) sums of
 * mcre_storage_moments, d_coef_row [2 + n_states * n_basis]: the coefficients are written behind the (centre, inverse
 * scale) pair the caller keeps in its first two entries.  Eigenvalues of the Gram matrix below rcond x the largest are
 * cut off (numpy.linalg.lstsq(G, rhs, rcond): a date with a deterministic spot fits the mean).  No host synchronisation:
 * the backward induction is one stream of kernels. */
int mcre_storage_solve(mcre_storage_plan *plan, const double *d_mom, double rcond, double *d_coef_row, void *stream);
/* Valuation pass, fused (path stepping + decisions + cashflows): ADDS each local path's discounted cashflows to d_cfs
 * [shard->n_paths]; d_coef [n_dates][2 + n_states * n_basis] (device); d_final_state [n_paths] or NULL.  Plans with
 * n_tan > 0 also ADD the path's pathwise sensitivities to d_tan [n_tan][n_paths]: what torch.autograd.grad of the PV
 * gives in the reference (controller.py:609-627) - decisions and inventory moves carry no gradient, cashflows
 * differentiate through the spot and the numeraire.  d_coef_expo [n_expo][2 + n_states * n_basis] + d_expo
 * [n_expo][n_paths] (both or neither): the path's exposure at every exposure date - the continuation polynomials of that
 * date interpolated at the inventory state after the actions up to it, over the numeraire (controller.py:432-447) - is
 * ADDED to d_expo, for the netting-set terms and exposure metrics of mcre_eq_unsecured_exposures / mcre_sum_stats /
 * mcre_select_*. */
int mcre_storage_mainsim(mcre_storage_plan *plan, const mcre_rng *rng, const mcre_shard *shard, const double *d_coef,
                         double initial_state, double *d_cfs, double *d_final_state, double *d_tan,
                         const double *d_coef_expo, double *d_expo, void *stream);

/* ================================================================================
 * Utilities
 * ============================================================================== */
/* Fixed-order binary-tree sum over chunks: d_partial [n_chunks][n_slots] -> d_out [n_slots]. */
int mcre_tree_reduce(const double *d_partial, int64_t n_chunks, int64_t n_slots, double *d_out, void *stream);
/* Measured FP64 FMA throughput of this GPU (TFLOP/s) from a register-resident DFMA loop;
 * the roofline denominator for the FP64-pipe-bound kernels (SURVEY §8d). */
int mcre_dfma_peak(double *tflops_out, void *stream);
/* Test hook for the branch-free FP64 functions of csrc/fastmath.cuh the fused kernels use instead
 * of libdevice: fn 0 exp, 1 log, 2 sqrt, 3 sin(2 pi x), 4 cos(2 pi x), 5 1/x; y[i] = fn(x[i]). */
int mcre_fastmath_probe(int32_t fn, const double *d_x, double *d_y, int64_t n, void *stream);
/* Kernel launches issued by this library since load (bench.py "gpu_launches"). */
int64_t mcre_launch_count(void);
/* Bytes this library has copied host -> device so far (plan arenas, coefficient uploads, job tables): what
 * bench.py reports as h2d_bytes_per_step of the end-to-end leg (measured, not computed). */
int64_t mcre_h2d_bytes(void);
const char *mcre_last_error(void);
int mcre_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* MCRE_H */
