// Gas storage on a two-factor log-price model: the reference's Storage.compute_normalized_cashflows
// (src/products/storage.py:215-308) and the controller loops around it (src/controller/controller.py:294-383 for the
// backward induction, :399-410 for the valuation pass) as four kernels:
//
//   storage_spots_kernel     pre-simulation forward pass: the spot of every action date, [date][path]
//   storage_backward_kernel  one date of the backward induction for all paths x all grid states in one launch:
//                            continuation grid (polynomial in the spot per state), the three actions, arg-max,
//                            float32 cashflow accumulator + interpolated float64 tail (controller.py:331-352)
//   storage_moments_kernel   Gram / right-hand-side moments of the regression of one date (large path counts)
//   storage_main_kernel      valuation pass, fused: path stepping + decision + realised cashflows per path; no
//                            path or state tensor is materialised
//
// The inventory arithmetic (volume <-> state, rate-curve interpolation, clamps) uses explicit unfused
// multiplies and adds: it is pure +,-,*,/ on contract data and reproduces the reference's doubles bit for bit,
// so a path sits in exactly the reference's state unless a decision differs.
#define MCRE_FAST_MATH 2   // table-driven exp / log / sincos of fastmath.cuh (<= 2 ulp), like the other fused kernels
#include "common.cuh"
#include "launch.cuh"
#include "philox.cuh"

namespace mcre {

constexpr int ST_REC = MCRE_STORAGE_RECORD;
constexpr int ST_KNOTS = MCRE_STORAGE_MAX_KNOTS;
constexpr int ST_MAX_S = MCRE_STORAGE_MAX_STATES;
constexpr int ST_MAX_B = MCRE_STORAGE_MAX_BASIS;
constexpr int ST_THREADS = 128;

struct StorageDev {
  int n_sub, n_dates, n_pre_dates, n_states, n_basis;
  double log_spot0;
  const double *step;       // [n_sub][ST_STEP]: see TwoFactor
  const int *step_date;     // [n_sub]
  const double *rec;        // [n_dates][ST_REC]
  const double *numeraire;  // [n_dates]
  // pathwise PV sensitivities (n_tan > 0) with respect to the storage's own tangent slots (the host scatters them into
  // the model's flattened parameters): tangents of the effective recursion per sub-step and slot, [n_sub][n_tan][ST_TAN]
  // = d(A, B00, M, B10, B11, log F, Bw) with x' = A x + B00 z0 + Bw-scaled w0, y' = y + M + B10 z0 + B11 z1 (see
  // storage_main_kernel), and d log numeraire / d slot per action date [n_dates][n_tan]
  int noise_dim, n_tan;
  const double *step_tan, *dlog_num;
  // exposure dates (controller.py:412-447): n_expo internal exposure dates, the first n_pre_expo at the calibration date;
  // step_expo [n_sub]: exposure index completed by the sub-step or -1; expo_num [n_expo]: numeraire there
  int n_expo, n_pre_expo;
  const int *step_expo;
  const double *expo_num;
};

}  // namespace mcre

struct mcre_storage_plan {
  mcre::StorageDev d;
  mcre::DevArena arena;
  mcre::DevArray<double> step, rec, numeraire, step_tan, dlog_num, expo_num;
  mcre::DevArray<int> step_date, step_expo;
};

namespace mcre {

// storage_helpers.py:96-127: torch.bucketize(point, xp) counts the knots strictly below the point; the segment is
// clamped to the curve, the weight is zero on a degenerate segment (torch.isclose: rtol 1e-5, atol 1e-8), and the
// end rates apply at and beyond the end knots.
__device__ __forceinline__ double curve_rate_dev(double point, const double *__restrict__ kn, int n) {
  if (n == 1) return __ldg(kn + 1);
  int below = 0;
  for (int j = 0; j < n; ++j) below += (__ldg(kn + 2 * j) < point) ? 1 : 0;
  int left = below - 1;
  left = left < 0 ? 0 : (left > n - 2 ? n - 2 : left);
  const double x0 = __ldg(kn + 2 * left), y0 = __ldg(kn + 2 * left + 1);
  const double x1 = __ldg(kn + 2 * left + 2), y1 = __ldg(kn + 2 * left + 3);
  const bool close = fabs(x0 - x1) <= 1e-8 + 1e-5 * fabs(x1);
  const double w = close ? 0.0 : __ddiv_rn(__dsub_rn(point, x0), __dsub_rn(x1, x0));
  double out = __dadd_rn(y0, __dmul_rn(w, __dsub_rn(y1, y0)));
  if (point <= __ldg(kn)) out = __ldg(kn + 1);
  if (point >= __ldg(kn + 2 * (n - 1))) out = __ldg(kn + 2 * (n - 1) + 1);
  return out;
}

struct Moves {
  double ns[3], dv[3];   // next state, volume difference of inject / hold / withdraw
};

// _transition_volume + _state_from_volume (storage.py:114-190) for the three actions from one state
__device__ __forceinline__ Moves transitions(const double *__restrict__ r, double state) {
  const double vmin = __ldg(r + 0), step = __ldg(r + 1), nmin = __ldg(r + 2), nmax = __ldg(r + 3);
  const double scale = __ldg(r + 4), period = __ldg(r + 5);
  const int n_inj = (int)__ldg(r + 8), n_wd = (int)__ldg(r + 9);
  const double vol = __dadd_rn(vmin, __dmul_rn(state, step));
  const double up = __dadd_rn(vol, __dmul_rn(curve_rate_dev(vol, r + 16, n_inj), period));
  const double dn = __dsub_rn(vol, __dmul_rn(curve_rate_dev(vol, r + 16 + 2 * ST_KNOTS, n_wd), period));
  double nv[3];
  nv[0] = fmin(up, nmax);
  nv[1] = fmin(fmax(vol, nmin), nmax);
  nv[2] = fmax(dn, nmin);
  Moves m;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    m.ns[a] = scale == 0.0 ? 0.0 : __dmul_rn(__dsub_rn(nv[a], nmin), scale);
    m.dv[a] = __dsub_rn(nv[a], vol);
  }
  return m;
}

// payoffs of the three actions (storage.py:246-253)
__device__ __forceinline__ void payoffs(const double *__restrict__ r, const Moves &m, double spot, double (&pay)[3]) {
  const double ci = __ldg(r + 6), cw = __ldg(r + 7);
  pay[0] = -m.dv[0] * (spot + ci);
  pay[1] = -m.dv[1] * (m.dv[1] >= 0.0 ? spot + ci : spot - cw);
  pay[2] = -m.dv[2] * (spot - cw);
}

// lookup_state_values (storage.py:200-213): weights of the two neighbouring grid states
__device__ __forceinline__ void neighbours(double state, int S, int &lo, int &hi, double &w) {
  const double b = fmin(fmax(state, 0.0), (double)(S - 1));
  const double f = floor(b);
  lo = (int)f; hi = (int)ceil(b);
  w = b - f;
}

// polynomial of the standardised spot u = (x - centre) * inv_scale; raw basis: centre 0, scale 1
__device__ __forceinline__ double poly(const double *__restrict__ c, int nb, double u) {
  double acc = __ldg(c), p = u;
  for (int k = 1; k < nb; ++k) { acc = fma(__ldg(c + k), p, acc); p *= u; }
  return acc;
}

// first maximum of (inject, hold, withdraw) like torch.argmax (storage.py:286)
__device__ __forceinline__ int best_of(const double (&v)[3]) {
  int a = 0;
  if (v[1] > v[a]) a = 1;
  if (v[2] > v[a]) a = 2;
  return a;
}

// One path of the two-factor log-price model, every scheme / price model in one form with the reference's association
// of operations (unfused):
//   w0 = sum_j bx_j z_j,  w1 = sum_j by_j z_j            (the model's rows of the joint draw z @ L^T, model.py:46-73)
//   x' = (a x - (k x) dt) + cx w0                        y' = (y + m) + cy w1            log S = log F + x' + y'
// Schwartz two-factor (schwartz_two_factor.py:147-196): ANALYTICAL a = exp(-kappa dt), k = 0, cx = cy = 1, b = rows of the
// Cholesky factor of the step covariance; EULER a = 1, k = kappa, cx / cy = sigma sqrt(dt), b = rows of the Cholesky
// factor of the correlation.  Black-Scholes single / multi-asset (black_scholes.py:50-67, black_scholes_multi.py:63-79,
// ANALYTICAL): the log-price accumulates in x (bx = the asset's row of the Cholesky factor of the step covariance over
// ALL assets of the model: the draw is the joint one), its drift in m, log F = log spot.
// Step record: [0] a, [1] k, [2] dt, [3] m, [4] cx, [5] cy, [6] log F, [7] 1: Euler Black-Scholes step (below),
// [8 + j] bx_j, [16 + j] by_j.
constexpr int ST_STEP = MCRE_STORAGE_STEP;
constexpr int ST_NOISE = MCRE_STORAGE_MAX_NOISE;
constexpr int ST_TAN = MCRE_STORAGE_TAN;
struct TwoFactor {
  double x = 0.0, y = 0.0;
  __device__ __forceinline__ double advance(const double *__restrict__ st, double w0, double w1) {
    if (__ldg(st + 7) != 0.0) {
      // Black-Scholes under EULER (black_scholes.py:69-85, black_scholes_multi.py:81-97): S' = S + (r S dt + sigma S
      // sqrt(dt) w) = S (1 + m + cx w0), carried in the log
      x = x + log1p(__dadd_rn(__ldg(st + 3), __dmul_rn(__ldg(st + 4), w0)));
      return __ldg(st + 6) + x;
    }
    const double drift = __dsub_rn(__dmul_rn(__ldg(st + 0), x), __dmul_rn(__dmul_rn(__ldg(st + 1), x), __ldg(st + 2)));
    x = __dadd_rn(drift, __dmul_rn(__ldg(st + 4), w0));
    y = __dadd_rn(__dadd_rn(y, __ldg(st + 3)), __dmul_rn(__ldg(st + 5), w1));
    return __dadd_rn(__dadd_rn(__ldg(st + 6), x), y);
  }
};

// the model's draws of one sub-step (normals number is * dim + j of the path, or the injected stream) folded into the two
// factor noises; z0, z1: the first two draws (tangent recursion of the one- and two-factor price models)
__device__ __forceinline__ void draw_w(const RngDev &rng, NormalStream &ns, int dim, int is, long long gpath,
                                       const double *__restrict__ st, double &w0, double &w1, double &z0, double &z1) {
  w0 = 0.0; w1 = 0.0; z0 = 0.0; z1 = 0.0;
  const double *zp = rng.mode == MCRE_RNG_INJECT ? rng.z + ((size_t)is * rng.n_total + gpath) * dim : nullptr;
  for (int j = 0; j < dim; ++j) {
    const double z = zp ? zp[j] : ns.next();
    if (j == 0) z0 = z;
    if (j == 1) z1 = z;
    const double tx = __dmul_rn(__ldg(st + 8 + j), z), ty = __dmul_rn(__ldg(st + 16 + j), z);
    w0 = j == 0 ? tx : __dadd_rn(w0, tx);
    w1 = j == 0 ? ty : __dadd_rn(w1, ty);
  }
}

__global__ void __launch_bounds__(ST_THREADS) storage_spots_kernel(StorageDev P, RngDev rng, long long path_begin,
                                                                   long long n_paths, double *__restrict__ spot,
                                                                   double *__restrict__ spot_expo) {
  fm_tables_init();
  const long long lp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (lp >= n_paths) return;
  const long long gp = path_begin + lp;
  NormalStream ns; ns.init(rng, (unsigned long long)gp);
  TwoFactor f;
  const double s0 = exp(P.log_spot0);
  for (int d = 0; d < P.n_pre_dates; ++d) spot[(size_t)d * n_paths + lp] = s0;
  if (spot_expo)
    for (int e = 0; e < P.n_pre_expo; ++e) spot_expo[(size_t)e * n_paths + lp] = s0;
  for (int is = 0; is < P.n_sub; ++is) {
    double w0, w1, z0, z1;
    const double *st = P.step + (size_t)is * ST_STEP;
    draw_w(rng, ns, P.noise_dim, is, gp, st, w0, w1, z0, z1);
    const double ls = f.advance(st, w0, w1);
    const int d = __ldg(P.step_date + is);
    const int e = spot_expo ? __ldg(P.step_expo + is) : -1;
    if (d >= 0 || e >= 0) {
      const double sp = fm_exp_t(ls);
      if (d >= 0) spot[(size_t)d * n_paths + lp] = sp;
      if (e >= 0) spot_expo[(size_t)e * n_paths + lp] = sp;
    }
  }
}

// One date of the backward induction.  value [S][n]: on entry the normalised value from the NEXT action date on per
// state entering it, on exit the same for THIS date (in place: a thread owns its path's column).
// coef: [2 + S * NB] = centre, inverse scale, coefficients per state of this date's continuation; unused on the last date.
__global__ void __launch_bounds__(ST_THREADS) storage_backward_kernel(StorageDev P, int date, const double *__restrict__ coef,
                                                                      const double *__restrict__ x, double *__restrict__ value,
                                                                      long long n) {
  // per (action, on-grid state): volume difference, interpolation weight and the two neighbouring states of the state
  // the action leads to - none of them depends on the path (first profile: 315 warp instructions per (path, state)
  // with the moves recomputed per path, profiles/r02_storage_kernels.md)
  __shared__ double s_dv[3 * ST_MAX_S], s_w[3 * ST_MAX_S];
  __shared__ int s_lo[3 * ST_MAX_S], s_hi[3 * ST_MAX_S];      // (offsets of the neighbour states' rows in the tiles below)
  __shared__ double s_val[ST_MAX_S * ST_THREADS], s_grid[ST_MAX_S * ST_THREADS];
  __shared__ double s_coef[2 + ST_MAX_S * ST_MAX_B];
  const int S = P.n_states, NB = P.n_basis, tid = threadIdx.x;
  const double *r = P.rec + (size_t)date * ST_REC;
  const bool last = __ldg(r + 10) != 0.0;
  if (tid < S) {
    const Moves m = transitions(r, (double)tid);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      int lo, hi;
      double w;
      neighbours(m.ns[a], S, lo, hi, w);
      s_dv[a * ST_MAX_S + tid] = m.dv[a]; s_w[a * ST_MAX_S + tid] = w;
      s_lo[a * ST_MAX_S + tid] = lo * ST_THREADS; s_hi[a * ST_MAX_S + tid] = hi * ST_THREADS;
    }
  }
  // the date's continuation coefficients once per block (second profile: 40 dependent read-only loads per path)
  if (!last)
    for (int i = tid; i < 2 + S * NB; i += ST_THREADS) s_coef[i] = coef[i];
  const long long p = (long long)blockIdx.x * blockDim.x + tid;
  const bool live = p < n;
  double spot = 0.0;
  if (live) {
    spot = x[p];
    for (int s = 0; s < S; ++s) s_val[s * ST_THREADS + tid] = value[(size_t)s * n + p];   // (all loads in flight together)
  }
  __syncthreads();
  if (!live) return;
  {
    const double u = last ? 0.0 : (spot - s_coef[0]) * s_coef[1];
    for (int s = 0; s < S; ++s) {
      double g = 0.0;
      if (!last) {
        const double *c = s_coef + 2 + s * NB;
        double pw = u;
        g = c[0];
        for (int k = 1; k < NB; ++k) { g = fma(c[k], pw, g); pw *= u; }
      }
      s_grid[s * ST_THREADS + tid] = g;
    }
  }
  // (a thread reads only its own column of the tiles: no barrier needed between its writes and its reads)
  const double num = __ldg(P.numeraire + date);
  const double ci = __ldg(r + 6), cw = __ldg(r + 7);
  const double buy = spot + ci, sell = spot - cw;      // storage.py:246-253
  const double *gcol = s_grid + tid, *vcol = s_val + tid;
#pragma unroll 2
  for (int s = 0; s < S; ++s) {
    double pay[3], v[3];
    const double dv1 = s_dv[ST_MAX_S + s];
    pay[0] = -s_dv[s] * buy;
    pay[1] = -dv1 * (dv1 >= 0.0 ? buy : sell);
    pay[2] = -s_dv[2 * ST_MAX_S + s] * sell;
    int lo[3], hi[3];
    double w[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = s_lo[a * ST_MAX_S + s]; hi[a] = s_hi[a * ST_MAX_S + s]; w[a] = s_w[a * ST_MAX_S + s];
      const double gl = gcol[lo[a]], gh = gcol[hi[a]];
      v[a] = pay[a] + __dadd_rn(gl, __dmul_rn(w[a], __dsub_rn(gh, gl)));
    }
    const int a = best_of(v);
    const double pa = a == 0 ? pay[0] : a == 1 ? pay[1] : pay[2];
    const int l = a == 0 ? lo[0] : a == 1 ? lo[1] : lo[2], h = a == 0 ? hi[0] : a == 1 ? hi[1] : hi[2];
    const double ww = a == 0 ? w[0] : a == 1 ? w[1] : w[2];
    const double tl = vcol[l], th = vcol[h];
    const double tail = __dadd_rn(tl, __dmul_rn(ww, __dsub_rn(th, tl)));
    // float32 accumulator of the window (controller.py:331, 342); x / 1 is exact, so the division is skipped there
    const double step = (double)(float)(num == 1.0 ? pa : __ddiv_rn(pa, num));
    value[(size_t)s * n + p] = step + tail;
  }
}

// Moments of the regression of `date`: y_s = numeraire(date) * value[s], basis u^k, u = (x - centre) * inv_scale.
// blockIdx.y < S: sum u^k y_s, k < NB -> slots [s * NB + k]; blockIdx.y == S: sum u^q, q < 2 NB - 1 -> slots [S * NB + q].
// One block per (chunk of paths, row); fixed summation order inside the block, chunks combined by mcre_tree_reduce.
__global__ void __launch_bounds__(256) storage_moments_kernel(StorageDev P, double num, double centre, double inv_scale,
                                                              const double *__restrict__ x, const double *__restrict__ value,
                                                              long long n, int chunk, double *__restrict__ partial) {
  __shared__ double stage[8][2 * ST_MAX_B];
  const int S = P.n_states, NB = P.n_basis, row = blockIdx.y;
  const int nv = row < S ? NB : 2 * NB - 1;
  double acc[2 * ST_MAX_B];
#pragma unroll
  for (int k = 0; k < 2 * ST_MAX_B; ++k) acc[k] = 0.0;
  const long long base = (long long)blockIdx.x * chunk;
  // four paths of a thread at a time: their loads are in flight together and their power chains interleave (one path at a
  // time was a chain of dependent multiplies behind two dependent loads: 24 us for 2^18 paths, latency bound)
  constexpr int IT = 4;
  for (int it0 = threadIdx.x; it0 < chunk; it0 += IT * (int)blockDim.x) {
    double u[IT], w[IT];
#pragma unroll
    for (int j = 0; j < IT; ++j) {
      const int it = it0 + j * (int)blockDim.x;
      const long long p = base + it;
      const bool ok = it < chunk && p < n;
      u[j] = ok ? (x[p] - centre) * inv_scale : 0.0;
      w[j] = ok ? (row < S ? num * value[(size_t)row * n + p] : 1.0) : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 2 * ST_MAX_B; ++k)
      if (k < nv) {
        acc[k] += (w[0] + w[1]) + (w[2] + w[3]);
#pragma unroll
        for (int j = 0; j < IT; ++j) w[j] *= u[j];
      }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 2 * ST_MAX_B; ++k) {
    double v = acc[k];
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) stage[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < nv) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += stage[w][threadIdx.x];
    const int n_slots = S * NB + 2 * NB - 1;
    partial[(size_t)blockIdx.x * n_slots + (row < S ? row * NB : S * NB) + threadIdx.x] = s;
  }
}


// Minimum-norm solution of the normal equations of one regression date on the device (the host solver of the
// "moments" mode was one synchronisation per action date: 0.3 ms x 454 dates).  mom: the all-reduced sums of
// storage_moments_kernel.  Thread 0 diagonalises the (NB x NB) Gram matrix by cyclic Jacobi rotations (symmetric positive
// semi-definite: eigenvalues = singular values), threads s < S apply the pseudo-inverse with the cut-off
// lambda_i > rcond * lambda_max to their right-hand side - numpy.linalg.lstsq(G, rhs, rcond) in exact arithmetic,
// including the rank-1 system of a date with a deterministic spot (all u equal -> the mean).
__global__ void __launch_bounds__(32) storage_solve_kernel(int S, int NB, const double *__restrict__ mom, double rcond,
                                                           double *__restrict__ coef) {
  __shared__ double V[ST_MAX_B][ST_MAX_B], lam[ST_MAX_B];
  __shared__ int use_chol;
  __shared__ double Lc[ST_MAX_B][ST_MAX_B];
  if (threadIdx.x == 0) {
    double G[ST_MAX_B][ST_MAX_B];
    double dmax = 0.0;
    for (int a = 0; a < NB; ++a)
      for (int b = 0; b < NB; ++b) { G[a][b] = mom[S * NB + a + b]; V[a][b] = a == b ? 1.0 : 0.0; }
    for (int a = 0; a < NB; ++a) dmax = fmax(dmax, G[a][a]);
    // fast path: a Cholesky factorisation whose pivots stay above 1e-8 of the largest diagonal entry and whose inverse
    // certifies that no eigenvalue is cut: the pseudo-inverse is then the inverse (all but the deterministic-spot
    // dates; the single-thread Jacobi sweeps below cost 80 us, as much as the backward and moments kernels together)
    int ok = 1;
    for (int j = 0; j < NB && ok; ++j) {
      double d = G[j][j];
      for (int k = 0; k < j; ++k) d -= Lc[j][k] * Lc[j][k];
      if (!(d > 1e-8 * dmax)) { ok = 0; break; }
      const double lj = sqrt(d);
      Lc[j][j] = lj;
      for (int i = j + 1; i < NB; ++i) {
        double v = G[i][j];
        for (int k = 0; k < j; ++k) v -= Lc[i][k] * Lc[j][k];
        Lc[i][j] = v / lj;
      }
    }
    // The pivots bound the smallest eigenvalue from above only: Hankel moments of a few support points pass them with
    // lambda_min / lambda_max far below rcond.  So the fast path also needs the lower bound lambda_min >= 1 / |G^-1|_F
    // (G^-1 = L^-T L^-1 from the factor) to exceed rcond * trace(G) >= rcond * lambda_max; otherwise the Jacobi path
    // below applies the cut-off.
    if (ok) {
      double Li[ST_MAX_B][ST_MAX_B];       // L^-1 (lower triangular)
      for (int j = 0; j < NB; ++j) {
        Li[j][j] = 1.0 / Lc[j][j];
        for (int i = j + 1; i < NB; ++i) {
          double v = 0.0;
          for (int k = j; k < i; ++k) v += Lc[i][k] * Li[k][j];
          Li[i][j] = -v / Lc[i][i];
        }
      }
      double fro = 0.0, trace = 0.0;
      for (int a = 0; a < NB; ++a) {
        trace += G[a][a];
        for (int b = 0; b < NB; ++b) {
          double v = 0.0;
          for (int k = a > b ? a : b; k < NB; ++k) v += Li[k][a] * Li[k][b];
          fro += v * v;
        }
      }
      ok = 1.0 / sqrt(fro) > rcond * trace;
    }
    use_chol = ok;
    for (int sweep = 0; sweep < 12 && !ok; ++sweep) {
      double off = 0.0, diag = 0.0;
      for (int a = 0; a < NB; ++a) { diag += G[a][a] * G[a][a]; for (int b = a + 1; b < NB; ++b) off += G[a][b] * G[a][b]; }
      if (off <= 1e-34 * diag) break;
      for (int p = 0; p < NB; ++p)
        for (int q = p + 1; q < NB; ++q) {
          if (G[p][q] == 0.0) continue;
          const double theta = (G[q][q] - G[p][p]) / (2.0 * G[p][q]);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
          for (int k = 0; k < NB; ++k) {       // columns p, q
            const double gkp = G[k][p], gkq = G[k][q];
            G[k][p] = c * gkp - sn * gkq; G[k][q] = sn * gkp + c * gkq;
          }
          for (int k = 0; k < NB; ++k) {       // rows p, q
            const double gpk = G[p][k], gqk = G[q][k];
            G[p][k] = c * gpk - sn * gqk; G[q][k] = sn * gpk + c * gqk;
          }
          for (int k = 0; k < NB; ++k) {
            const double vkp = V[k][p], vkq = V[k][q];
            V[k][p] = c * vkp - sn * vkq; V[k][q] = sn * vkp + c * vkq;
          }
        }
    }
    double top = 0.0;
    for (int a = 0; a < NB; ++a) { lam[a] = G[a][a]; top = fmax(top, fabs(G[a][a])); }
    for (int a = 0; a < NB; ++a) lam[a] = lam[a] > rcond * top ? 1.0 / lam[a] : 0.0;   // (inverse, 0 = cut off)
  }
  __syncthreads();
  if (use_chol) {
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
      double y[ST_MAX_B];
      for (int i = 0; i < NB; ++i) {           // L y = b
        double v = mom[s * NB + i];
        for (int k = 0; k < i; ++k) v -= Lc[i][k] * y[k];
        y[i] = v / Lc[i][i];
      }
      for (int i = NB - 1; i >= 0; --i) {      // L^T c = y
        double v = y[i];
        for (int k = i + 1; k < NB; ++k) v -= Lc[k][i] * y[k];
        y[i] = v / Lc[i][i];
      }
      for (int k = 0; k < NB; ++k) coef[2 + s * NB + k] = y[k];
    }
    return;
  }
  __syncthreads();
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    double y[ST_MAX_B];
    for (int i = 0; i < NB; ++i) {
      double acc = 0.0;
      for (int k = 0; k < NB; ++k) acc += V[k][i] * mom[s * NB + k];
      y[i] = acc * lam[i];
    }
    for (int k = 0; k < NB; ++k) {
      double acc = 0.0;
      for (int i = 0; i < NB; ++i) acc += V[k][i] * y[i];
      coef[2 + s * NB + k] = acc;
    }
  }
}

// Valuation pass (controller.py:399-410 with storage.py:215-308 inlined): one thread per path carries the two factors,
// the inventory state and the running sum of discounted cashflows.  coef: [n_dates][2 + S * NB].
// NT > 0: pathwise sensitivities of the PV with respect to the NT model parameters, the way the reference's autograd sees
// them (controller.py:609-627): the arg-max and the inventory moves carry no gradient, a cashflow
// -dV (S +- cost) / N differentiates to -dV dS / N - cashflow dlogN, and dS = S dlogS follows the tangent recursion of
// the factors:
//   two-factor step     dx' = A dx + dA x + dB00 z0 + dBw w0,  dy' = dy + dM + dB10 z0 + dB11 z1
//                       (dBw w0 = d(sum_j bx_j z_j): a Black-Scholes asset of a joint draw, whose row of the Cholesky
//                       factor of D C D dt is proportional to its own volatility; 0 for the other models)
//   Black-Scholes EULER dx' = dx + (dM + dBw w0) / (1 + m + cx w0)   (dM = d(rate dt), dBw = d(sigma sqrt(dt)))
// NT counts the storage's own tangent slots (3: spot, volatility, rate of a Black-Scholes asset, + 1: the numeraire
// model's rate; 6: the Schwartz parameters), not the parameters of the joint model.
// Per-path tangents are ADDED to tan [NT][n_paths].
template <int NT>
__global__ void __launch_bounds__(ST_THREADS) storage_main_kernel(StorageDev P, RngDev rng, long long path_begin,
                                                                  long long n_paths, const double *__restrict__ coef,
                                                                  double initial_state, double *__restrict__ cfs,
                                                                  double *__restrict__ final_state, double *__restrict__ tan,
                                                                  const double *__restrict__ coef_expo,
                                                                  double *__restrict__ expo) {
  fm_tables_init();
  const long long lp = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (lp >= n_paths) return;
  const long long gp = path_begin + lp;
  NormalStream ns; ns.init(rng, (unsigned long long)gp);
  TwoFactor f;
  const int S = P.n_states, NB = P.n_basis, row = 2 + S * NB;
  double state = initial_state, total = 0.0;
  double dx[NT > 0 ? NT : 1], dy[NT > 0 ? NT : 1], dls[NT > 0 ? NT : 1], dtot[NT > 0 ? NT : 1];
#pragma unroll
  for (int k = 0; k < NT; ++k) { dx[k] = 0.0; dy[k] = 0.0; dls[k] = 0.0; dtot[k] = 0.0; }

  auto act = [&](int d, double spot) {
    const double *r = P.rec + (size_t)d * ST_REC;
    const Moves m = transitions(r, state);
    double pay[3], v[3];
    payoffs(r, m, spot, pay);
    if (__ldg(r + 10) != 0.0) {
#pragma unroll
      for (int a = 0; a < 3; ++a) v[a] = pay[a];
    } else {
      const double *c = coef + (size_t)d * row;
      const double u = (spot - __ldg(c)) * __ldg(c + 1);
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        int lo, hi;
        double w;
        neighbours(m.ns[a], S, lo, hi, w);
        const double gl = poly(c + 2 + lo * NB, NB, u);
        const double gh = hi == lo ? gl : poly(c + 2 + hi * NB, NB, u);
        v[a] = pay[a] + __dadd_rn(gl, __dmul_rn(w, __dsub_rn(gh, gl)));
      }
    }
    const int a = best_of(v);
    state = a == 0 ? m.ns[0] : a == 1 ? m.ns[1] : m.ns[2];
    const double num = __ldg(P.numeraire + d);
    const double cf = __ddiv_rn(a == 0 ? pay[0] : a == 1 ? pay[1] : pay[2], num);
    total += cf;
    if constexpr (NT > 0) {
      const double dvb = a == 0 ? m.dv[0] : a == 1 ? m.dv[1] : m.dv[2];
      const double g = -dvb * spot / num;
#pragma unroll
      for (int k = 0; k < NT; ++k) dtot[k] += g * dls[k] - cf * __ldg(P.dlog_num + (size_t)d * NT + k);
    }
  };

  // exposure at an exposure date (controller.py:432-447): the continuation polynomials of that date, interpolated at the
  // inventory state the path is in after the actions up to that date, over the numeraire; ADDED to expo [n_expo][n_paths]
  auto exposure = [&](int e, double spot) {
    const double *c = coef_expo + (size_t)e * row;
    const double u = (spot - __ldg(c)) * __ldg(c + 1);
    int lo, hi;
    double w;
    neighbours(state, S, lo, hi, w);
    const double gl = poly(c + 2 + lo * NB, NB, u);
    const double gh = hi == lo ? gl : poly(c + 2 + hi * NB, NB, u);
    const double cont = __dadd_rn(gl, __dmul_rn(w, __dsub_rn(gh, gl)));
    expo[(size_t)e * n_paths + lp] += __ddiv_rn(cont, __ldg(P.expo_num + e));
  };

  const double s0 = exp(P.log_spot0);
  if constexpr (NT > 0) {
    // at the calibration date only log F0 depends on the parameters (Black-Scholes: log of the spot parameter);
    // its tangent is stored with the first sub-step
    if (P.n_sub > 0) {
#pragma unroll
      for (int k = 0; k < NT; ++k) dls[k] = __ldg(P.step_tan + (size_t)k * ST_TAN + 5);
    }
  }
  for (int d = 0; d < P.n_pre_dates; ++d) act(d, s0);
  if (expo)
    for (int e = 0; e < P.n_pre_expo; ++e) exposure(e, s0);
  for (int is = 0; is < P.n_sub; ++is) {
    double w0, w1, z0, z1;
    const double x_old = f.x;
    const double *st = P.step + (size_t)is * ST_STEP;
    draw_w(rng, ns, P.noise_dim, is, gp, st, w0, w1, z0, z1);
    const double ls = f.advance(st, w0, w1);
    if constexpr (NT > 0) {
      const double *tt = P.step_tan + (size_t)is * NT * ST_TAN;
      if (__ldg(st + 7) != 0.0) {
        const double inv = 1.0 / (1.0 + __dadd_rn(__ldg(st + 3), __dmul_rn(__ldg(st + 4), w0)));
#pragma unroll
        for (int k = 0; k < NT; ++k) {
          const double *t7 = tt + k * ST_TAN;
          dx[k] = dx[k] + (__ldg(t7 + 2) + __ldg(t7 + 6) * w0) * inv;
          dls[k] = __ldg(t7 + 5) + dx[k];
        }
      } else {
        const double A = __ldg(st + 0) - __ldg(st + 1) * __ldg(st + 2);
#pragma unroll
        for (int k = 0; k < NT; ++k) {
          const double *t7 = tt + k * ST_TAN;
          dx[k] = A * dx[k] + __ldg(t7 + 0) * x_old + __ldg(t7 + 1) * z0;
          dx[k] = fma(__ldg(t7 + 6), w0, dx[k]);
          dy[k] = dy[k] + __ldg(t7 + 2) + __ldg(t7 + 3) * z0 + __ldg(t7 + 4) * z1;
          dls[k] = __ldg(t7 + 5) + dx[k] + dy[k];
        }
      }
    }
    const int d = __ldg(P.step_date + is);
    const int e = expo ? __ldg(P.step_expo + is) : -1;
    if (d >= 0 || e >= 0) {
      const double sp = fm_exp_t(ls);
      if (d >= 0) act(d, sp);          // the action of a date comes before the exposure of the same date (:417-430)
      if (e >= 0) exposure(e, sp);
    }
  }
  cfs[lp] += total;
  if (final_state) final_state[lp] = state;
  if constexpr (NT > 0) {
#pragma unroll
    for (int k = 0; k < NT; ++k) tan[(size_t)k * n_paths + lp] += dtot[k];
  }
}

}  // namespace mcre

using namespace mcre;

extern "C" int mcre_storage_create(const mcre_storage_desc *c, mcre_storage_plan **out) {
  if (!c || !out) return fail(-1, "null argument%s", "");
  if (c->n_states < 2 || c->n_states > ST_MAX_S) return fail(-2, "storage: 2..%s%lld inventory states", "", ST_MAX_S);
  if (c->n_basis < 1 || c->n_basis > ST_MAX_B) return fail(-2, "storage: 1..%s%lld basis functions", "", ST_MAX_B);
  if (c->noise_dim < 1 || c->noise_dim > ST_NOISE) return fail(-2, "storage: 1..8 noise factors%s", "");
  if (c->n_tan != 0 && c->n_tan != 3 && c->n_tan != 4 && c->n_tan != 6)
    return fail(-2, "storage: 0, 3, 4 or 6 tangent directions%s", "");
  if (c->n_tan > 0 && (!c->step_tan || !c->dlog_num)) return fail(-1, "storage: tangent tables missing%s", "");
  if (c->n_expo < 0 || c->n_pre_expo < 0 || c->n_pre_expo > c->n_expo || (c->n_expo > 0 && (!c->expo_numeraire || (c->n_sub > 0 && !c->step_expo))))
    return fail(-2, "storage: bad exposure tables%s", "");
  if (c->n_dates <= 0 || c->n_sub < 0 || c->n_pre_dates < 0 || c->n_pre_dates > c->n_dates)
    return fail(-2, "storage: bad date / step counts%s", "");
  for (int d = 0; d < c->n_dates; ++d) {
    const double *r = c->date_rec + (size_t)d * ST_REC;
    if (r[8] < 1 || r[8] > ST_KNOTS || r[9] < 1 || r[9] > ST_KNOTS) return fail(-2, "storage: 1..8 knots per rate curve%s", "");
  }
  mcre_storage_plan *p = new mcre_storage_plan();
  int rc = 0;
  {
    ArenaScope scope(&p->arena);
    if (!rc) rc = p->step.upload(c->step, (size_t)c->n_sub * ST_STEP);
    if (!rc) rc = p->step_date.upload(c->step_date, (size_t)c->n_sub);
    if (!rc) rc = p->rec.upload(c->date_rec, (size_t)c->n_dates * ST_REC);
    if (!rc) rc = p->numeraire.upload(c->numeraire, (size_t)c->n_dates);
    if (!rc && c->n_expo > 0) rc = p->step_expo.upload(c->step_expo, (size_t)c->n_sub);
    if (!rc && c->n_expo > 0) rc = p->expo_num.upload(c->expo_numeraire, (size_t)c->n_expo);
    if (!rc && c->n_tan > 0) rc = p->step_tan.upload(c->step_tan, (size_t)c->n_sub * c->n_tan * ST_TAN);
    if (!rc && c->n_tan > 0) rc = p->dlog_num.upload(c->dlog_num, (size_t)c->n_dates * c->n_tan);
    if (!rc) rc = p->arena.commit();
  }
  if (rc) { p->arena.release(); delete p; return rc; }
  StorageDev &d = p->d;
  d.n_sub = c->n_sub; d.n_dates = c->n_dates; d.n_pre_dates = c->n_pre_dates; d.n_states = c->n_states;
  d.n_basis = c->n_basis; d.log_spot0 = c->log_spot0;
  d.step = p->step.p; d.step_date = p->step_date.p; d.rec = p->rec.p; d.numeraire = p->numeraire.p;
  d.noise_dim = c->noise_dim; d.n_tan = c->n_tan; d.step_tan = p->step_tan.p; d.dlog_num = p->dlog_num.p;
  d.n_expo = c->n_expo; d.n_pre_expo = c->n_pre_expo; d.step_expo = p->step_expo.p; d.expo_num = p->expo_num.p;
  *out = p;
  return 0;
}

extern "C" void mcre_storage_destroy(mcre_storage_plan *p) {
  if (!p) return;
  p->arena.release();
  delete p;
}

static int storage_rng_ok(const mcre_rng *rng) {
  if (rng->mode == MCRE_RNG_INJECT && !rng->d_z) return fail(-1, "inject mode without normals%s", "");
  return 0;
}

extern "C" int mcre_storage_spots(mcre_storage_plan *p, const mcre_rng *rng, const mcre_shard *shard, double *d_spot,
                                  double *d_spot_expo, void *stream) {
  if (!p || !rng || !shard || !d_spot) return fail(-1, "null argument%s", "");
  if (d_spot_expo && p->d.n_expo <= 0) return fail(-2, "storage: exposure spots requested on a plan without exposure dates%s", "");
  if (int rc = storage_rng_ok(rng)) return rc;
  if (shard->n_paths <= 0) return 0;
  const unsigned blocks = (unsigned)((shard->n_paths + ST_THREADS - 1) / ST_THREADS);
  storage_spots_kernel<<<blocks, ST_THREADS, 0, (cudaStream_t)stream>>>(p->d, make_rng(rng), shard->path_begin,
                                                                         shard->n_paths, d_spot, d_spot_expo);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_storage_backward(mcre_storage_plan *p, int32_t date, const double *d_coef, const double *d_spot_row,
                                     double *d_value, int64_t n, void *stream) {
  if (!p || !d_spot_row || !d_value) return fail(-1, "null argument%s", "");
  if (date < 0 || date >= p->d.n_dates) return fail(-2, "storage: date index out of range%s", "");
  if (n <= 0) return 0;
  const unsigned blocks = (unsigned)((n + ST_THREADS - 1) / ST_THREADS);
  storage_backward_kernel<<<blocks, ST_THREADS, 0, (cudaStream_t)stream>>>(p->d, date, d_coef, d_spot_row, d_value, n);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int64_t mcre_storage_moment_slots(const mcre_storage_plan *p) {
  return p ? (int64_t)p->d.n_states * p->d.n_basis + 2 * p->d.n_basis - 1 : 0;
}

extern "C" int mcre_storage_moments(mcre_storage_plan *p, double numeraire, double centre, double inv_scale,
                                    const double *d_spot_row, const double *d_value, int64_t n, int32_t chunk_paths,
                                    double *d_partial, double *d_out, void *stream) {
  if (!p || !d_spot_row || !d_value || !d_partial || !d_out) return fail(-1, "null argument%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "storage: chunk_paths must be a multiple of 256%s", "");
  const int64_t slots = mcre_storage_moment_slots(p);
  const long long n_chunks = n > 0 ? (n + chunk_paths - 1) / chunk_paths : 0;
  if (n_chunks > 0) {
    dim3 grid((unsigned)n_chunks, (unsigned)(p->d.n_states + 1));
    storage_moments_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(p->d, numeraire, centre, inv_scale, d_spot_row, d_value, n,
                                                                   chunk_paths, d_partial);
    MCRE_LAUNCHED();
  }
  return mcre_tree_reduce(d_partial, n_chunks, slots, d_out, stream);
}

extern "C" int mcre_storage_solve(mcre_storage_plan *p, const double *d_mom, double rcond, double *d_coef_row,
                                  void *stream) {
  if (!p || !d_mom || !d_coef_row) return fail(-1, "null argument%s", "");
  storage_solve_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(p->d.n_states, p->d.n_basis, d_mom, rcond, d_coef_row);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_storage_mainsim(mcre_storage_plan *p, const mcre_rng *rng, const mcre_shard *shard,
                                    const double *d_coef, double initial_state, double *d_cfs, double *d_final_state,
                                    double *d_tan, const double *d_coef_expo, double *d_expo, void *stream) {
  if (!p || !rng || !shard || !d_coef || !d_cfs) return fail(-1, "null argument%s", "");
  if ((d_expo != nullptr) != (d_coef_expo != nullptr) || (d_expo && p->d.n_expo <= 0))
    return fail(-2, "storage: exposures need both the coefficient table and the output, on a plan with exposure dates%s", "");
  if (p->d.n_tan > 0 && !d_tan) return fail(-1, "storage: plan with tangents but d_tan is null%s", "");
  if (int rc = storage_rng_ok(rng)) return rc;
  if (shard->n_paths <= 0) return 0;
  const unsigned blocks = (unsigned)((shard->n_paths + ST_THREADS - 1) / ST_THREADS);
  const RngDev r = make_rng(rng);
  cudaStream_t st = (cudaStream_t)stream;
#define GO(NT) storage_main_kernel<NT><<<blocks, ST_THREADS, 0, st>>>(p->d, r, shard->path_begin, shard->n_paths, d_coef, \
                                                                     initial_state, d_cfs, d_final_state, d_tan, d_coef_expo, d_expo)
  if (p->d.n_tan == 0) GO(0);
  else if (p->d.n_tan == 3) GO(3);
  else if (p->d.n_tan == 4) GO(4);
  else GO(6);
#undef GO
  MCRE_LAUNCHED();
  return 0;
}
