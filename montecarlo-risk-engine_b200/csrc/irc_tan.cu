// Interest-rate / credit family: pre-simulation with pathwise tangents, for sensitivities of
// exposure metrics through the regression proxy.
//
// With differentiate=True the reference's regression coefficients carry gradient: the least
// squares of controller.py:368-383 sits inside the autograd graph, so d(EPE, CVA, ...)/d(theta)
// contains d(coefficients)/d(theta).  Here the pre-simulation propagates forward tangents of the
// explanatory variable x, the numeraire N and the windowed discounted cashflows W along every
// path (same dual arithmetic as the main kernel), and a second kernel accumulates, per
// regression date, unit and model parameter, the nine sums from which the host differentiates
// the normal equations (pseudo-inverse derivative, mcre/lsm.py:regression_tangents):
//   sum u^m du (m = 0..3), sum u^i dY (i = 0..2), sum du Y, sum 2 u du Y,
// with u = (x - shift) scale, du = dx scale, Y = N S, dY = dN S + N dS, S the float32 suffix
// sum of W (values rounded like the reference's float32 accumulators, controller.py:312-351;
// tangents stay FP64).
#include "irc_main.cuh"

namespace mcre {

constexpr int TM_NV = 9;    // tangent moments per (unit, parameter, regression date)
constexpr int TM_IT = 8;    // paths per thread of the tangent moments kernel

// scratch: x [n_reg][n] f64 | N [n_reg][n] f64 | W [n_units][n_reg][n] f32 (as the value-only
// pre-simulation) | dx [n_reg][NT][n] | dN [n_reg][NT][n] | dW [n_units][n_reg][NT][n], f64
template <int NT, bool CIR, int SCHEME>
__global__ void __launch_bounds__(128) irc_presim_forward_tan_kernel(IrcDev P, RngDev rng, ShardDev sh, double *xbuf,
                                                                     double *nbuf, float *wbuf, double *dxbuf,
                                                                     double *dnbuf, double *dwbuf) {
  typedef Dual<NT> R;
  typedef RealTraits<R> T;
  fm_tables_init();
  const long long lpath = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (lpath >= sh.n_paths) return;
  const long long gpath = sh.path_begin + lpath;
  const long long n = sh.n_paths;
  IrcParams<R, CIR> mp;
  irc_load_params<R, CIR>(P, mp);
  NormalStream ns; ns.init(rng, (unsigned long long)gpath);
  IrcState<R> st;
  st.r = mp.r0; st.logB = T::zero(); st.y = mp.y0; st.logBl = T::zero();
  R W[MCRE_IRC_MAX_UNITS];
#pragma unroll
  for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u) W[u] = T::zero();

  auto store_window = [&](int u, int k) {
    wbuf[((size_t)u * P.n_reg + k) * n + lpath] = (float)W[u].v;
#pragma unroll
    for (int i = 0; i < NT; ++i) dwbuf[(((size_t)u * P.n_reg + k) * NT + i) * n + lpath] = W[u].d[i];
  };
  auto eval_date = [&](int di) {
    const int flags = __ldg(P.date_flags + di);
    if (!(flags & (MCRE_DATE_HAS_CASHFLOW | MCRE_DATE_HAS_REGRESSION))) return;
    const R numeraire = r_exp(st.logB);
    if (flags & MCRE_DATE_HAS_CASHFLOW) {
      R cf[MCRE_IRC_MAX_UNITS];
#pragma unroll
      for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u)
        cf[u] = T::lift(u < P.n_units ? __ldg(P.unit_fix + (size_t)u * P.n_dates + di) : 0.0);
      const int j0 = __ldg(P.date_float_off + di), j1 = __ldg(P.date_float_off + di + 1);
      for (int j = j0; j < j1; ++j) {
        const R alpha = T::load(P.float_coef, j * 2), B = T::load(P.float_coef, j * 2 + 1);
        const R libor = (r_exp(B * st.r - alpha) - 1.0) * __ldg(P.float_inv_tau + j);
#pragma unroll
        for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u)
          if (u < P.n_units) cf[u] = cf[u] + libor * __ldg(P.unit_float + (size_t)u * P.n_float + j);
      }
      const R invN = 1.0 / numeraire;
#pragma unroll
      for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u) {
        // float32 accumulator, float64 addend: W <- fp32(fp64(W) + cf / N) (controller.py:330,341)
        W[u] = W[u] + cf[u] * invN;
        W[u].v = (double)(float)W[u].v;
      }
    }
    if (flags & MCRE_DATE_HAS_REGRESSION) {
      const int k = __ldg(P.date_reg + di);
      xbuf[(size_t)k * n + lpath] = st.r.v;
      nbuf[(size_t)k * n + lpath] = numeraire.v;
#pragma unroll
      for (int i = 0; i < NT; ++i) {
        dxbuf[((size_t)k * NT + i) * n + lpath] = st.r.d[i];
        dnbuf[((size_t)k * NT + i) * n + lpath] = numeraire.d[i];
      }
#pragma unroll
      for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u) {
        if (u < P.n_units && k > 0) store_window(u, k - 1);
        W[u] = T::zero();   // cashflows at or before the first regression date never enter a window
      }
    }
  };
  for (int di = 0; di < P.n_pre_dates; ++di) eval_date(di);
  for (int is = 0; is < P.n_sub; ++is) {
    double z0, z1;
    irc_draw<R, CIR>(rng, ns, is, lpath, gpath, z0, z1);
    irc_step<R, CIR, SCHEME, false>(P, mp, st, is, z0, z1);
    const int di = __ldg(P.step_date + is);
    if (di >= 0) eval_date(di);
  }
#pragma unroll
  for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u)
    if (u < P.n_units && P.n_reg > 0) store_window(u, P.n_reg - 1);
}

// grid (chunks, nt, n_units); partial: [chunk][unit][parameter][n_reg][TM_NV]
__global__ void __launch_bounds__(256) irc_presim_tangent_moments_kernel(IrcDev P, ShardDev sh, int nt,
                                                                         const double *xbuf, const double *nbuf,
                                                                         const float *wbuf, const double *dxbuf,
                                                                         const double *dnbuf, const double *dwbuf,
                                                                         double *partial) {
  extern __shared__ double smem[];
  const int nw = blockDim.x >> 5;
  const int n_slots = P.n_reg * TM_NV;
  double *acc = smem;
  double *stage = smem + n_slots;
  const int ip = blockIdx.y, un = blockIdx.z;
  const long long n = sh.n_paths;
  const long long n_chunks = (n + sh.chunk - 1) / sh.chunk;
  for (long long chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) acc[i] = 0.0;
    __syncthreads();
    int parity = 0;
    for (int base = 0; base < sh.chunk; base += TM_IT * (int)blockDim.x) {
      float S[TM_IT];
      double dS[TM_IT];
      long long path[TM_IT];
      bool live[TM_IT];
#pragma unroll
      for (int i = 0; i < TM_IT; ++i) {
        const int in_chunk = base + i * (int)blockDim.x + (int)threadIdx.x;
        const long long lp = chunk * sh.chunk + in_chunk;
        live[i] = in_chunk < sh.chunk && lp < n;
        path[i] = live[i] ? lp : 0;
        S[i] = 0.0f; dS[i] = 0.0;
      }
      for (int k = P.n_reg - 1; k >= 0; --k) {
        const double bs = __ldg(P.reg_basis + k * 2), bc = __ldg(P.reg_basis + k * 2 + 1);
        double vals[TM_NV];
#pragma unroll
        for (int j = 0; j < TM_NV; ++j) vals[j] = 0.0;
#pragma unroll
        for (int i = 0; i < TM_IT; ++i) {
          const size_t at = (size_t)k * n + path[i], dat = ((size_t)k * nt + ip) * n + path[i];
          const double x = xbuf[at], numeraire = nbuf[at];
          const double dx = dxbuf[dat], dnum = dnbuf[dat];
          S[i] = wbuf[((size_t)un * P.n_reg + k) * n + path[i]] + S[i];      // float32 + float32 (controller.py:349)
          dS[i] += dwbuf[(((size_t)un * P.n_reg + k) * nt + ip) * n + path[i]];
          const double keep = live[i] ? 1.0 : 0.0;
          const double uu = (x - bs) * bc, du = keep * dx * bc;
          const double Y = numeraire * (double)S[i];
          const double dY = keep * (dnum * (double)S[i] + numeraire * dS[i]);
          const double u2 = uu * uu;
          vals[0] += du; vals[1] += uu * du; vals[2] += u2 * du; vals[3] += u2 * uu * du;
          vals[4] += dY; vals[5] += uu * dY; vals[6] += u2 * dY;
          vals[7] += du * Y; vals[8] += 2.0 * uu * du * Y;
        }
        block_accumulate<TM_NV>(vals, acc, k * TM_NV, stage, TM_NV, parity);
      }
    }
    __syncthreads();
    double *out = partial + (((size_t)chunk * gridDim.z + un) * nt + ip) * n_slots;
    for (int i = threadIdx.x; i < n_slots; i += blockDim.x) out[i] = acc[i];
    __syncthreads();
  }
}

// Pre-simulation of a Bermudan unit with tangents: like irc_lsm_forward_kernel, plus the pathwise tangents of the
// explanatory variable, the numeraire and the immediate exercise values.
// scratch: x [n_reg][n] | N [n_reg][n] | imm [n_ex][n] | dx [n_reg][NT][n] | dN [n_reg][NT][n] | dimm [n_ex][NT][n]
template <int NT, bool CIR, int SCHEME>
__global__ void __launch_bounds__(128) irc_lsm_forward_tan_kernel(IrcDev P, RngDev rng, ShardDev sh, double *xbuf,
                                                                  double *nbuf, double *ibuf, double *dxbuf, double *dnbuf,
                                                                  double *dibuf) {
  typedef Dual<NT> R;
  typedef RealTraits<R> T;
  fm_tables_init();
  const long long lpath = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (lpath >= sh.n_paths) return;
  const long long gpath = sh.path_begin + lpath;
  const long long n = sh.n_paths;
  IrcParams<R, CIR> mp;
  irc_load_params<R, CIR>(P, mp);
  NormalStream ns; ns.init(rng, (unsigned long long)gpath);
  IrcState<R> st;
  st.r = mp.r0; st.logB = T::zero(); st.y = mp.y0; st.logBl = T::zero();
  auto eval_date = [&](int di) {
    const int flags = __ldg(P.date_flags + di);
    if (flags & MCRE_DATE_HAS_REGRESSION) {
      const int k = __ldg(P.date_reg + di);
      const R num = r_exp(st.logB);
      xbuf[(size_t)k * n + lpath] = st.r.v;
      nbuf[(size_t)k * n + lpath] = num.v;
#pragma unroll
      for (int i = 0; i < NT; ++i) {
        dxbuf[((size_t)k * NT + i) * n + lpath] = st.r.d[i];
        dnbuf[((size_t)k * NT + i) * n + lpath] = num.d[i];
      }
    }
    if (flags & MCRE_DATE_HAS_EXERCISE) {
      const int x0 = __ldg(P.date_ex_off + di), x1 = __ldg(P.date_ex_off + di + 1);
      for (int x = x0; x < x1; ++x) {
        const R imm = irc_exercise_value<R>(P, x, st.r);
        ibuf[(size_t)x * n + lpath] = imm.v;
#pragma unroll
        for (int i = 0; i < NT; ++i) dibuf[((size_t)x * NT + i) * n + lpath] = imm.d[i];
      }
    }
  };
  for (int di = 0; di < P.n_pre_dates; ++di) eval_date(di);
  for (int is = 0; is < P.n_sub; ++is) {
    double z0, z1;
    irc_draw<R, CIR>(rng, ns, is, lpath, gpath, z0, z1);
    irc_step<R, CIR, SCHEME, false>(P, mp, st, is, z0, z1);
    const int di = __ldg(P.step_date + is);
    if (di >= 0) eval_date(di);
  }
}

// Tangent companion of lsm_step_kernel<1> (csrc/lsm.cu), one exercise right: for parameter blockIdx.y it applies
// the SAME exercise decision as the value pass (hard indicator, no derivative) to the running tangent
//     dV <- ex ? d(imm_i / N_i) : dV,   d(imm / N) = (dimm - (imm / N) dN) / N
// and accumulates the nine tangent moments of regression date k (see the header of this file) with Y = N_k V,
// dY = dN_k V + N_k dV, V the float32 running value the value pass has already updated for this date.
// dvalue: [nt][n] f64; partial: [chunk][nt][9].
__global__ void __launch_bounds__(256) lsm_step_tan_kernel(int nt, const double *__restrict__ xk, const double *__restrict__ nk,
                                                           const double *__restrict__ dxk, const double *__restrict__ dnk,
                                                           double shift_k, double scale_k, const double *__restrict__ xi,
                                                           const double *__restrict__ ni, const double *__restrict__ imm,
                                                           const double *__restrict__ dni, const double *__restrict__ dimm,
                                                           int has_coef, double c0, double c1, double c2, double shift_i,
                                                           double scale_i, const float *__restrict__ value,
                                                           double *__restrict__ dvalue, long long n, int chunk,
                                                           double *__restrict__ partial) {
  __shared__ double acc[TM_NV];
  __shared__ double stage[2 * 8 * TM_NV];
  const int ip = blockIdx.y;
  const long long n_chunks = (n + chunk - 1) / chunk;
  for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
    if (threadIdx.x < TM_NV) acc[threadIdx.x] = 0.0;
    __syncthreads();
    int parity = 0;
    double vals[TM_NV];
#pragma unroll
    for (int j = 0; j < TM_NV; ++j) vals[j] = 0.0;
    for (int it = 0; it < chunk; it += blockDim.x) {
      const long long p = ch * chunk + it + threadIdx.x;
      if (it + (int)threadIdx.x < chunk && p < n) {
        double dv = dvalue[(size_t)ip * n + p];
        if (imm) {
          const double im = imm[p];
          double cont = 0.0;
          if (has_coef) {
            const double ui = (xi[p] - shift_i) * scale_i;
            cont = c0 + ui * (c1 + ui * c2);
          }
          if (im > cont) {
            const double inv = 1.0 / ni[p];
            dv = (dimm[(size_t)ip * n + p] - im * inv * dni[(size_t)ip * n + p]) * inv;
          }
          dvalue[(size_t)ip * n + p] = dv;
        }
        const double uu = (xk[p] - shift_k) * scale_k, du = dxk[(size_t)ip * n + p] * scale_k;
        const double V = (double)value[p];
        const double Y = nk[p] * V, dY = dnk[(size_t)ip * n + p] * V + nk[p] * dv;
        const double u2 = uu * uu;
        vals[0] += du; vals[1] += uu * du; vals[2] += u2 * du; vals[3] += u2 * uu * du;
        vals[4] += dY; vals[5] += uu * dY; vals[6] += u2 * dY;
        vals[7] += du * Y; vals[8] += 2.0 * uu * du * Y;
      }
    }
    block_accumulate<TM_NV>(vals, acc, 0, stage, TM_NV, parity);
    __syncthreads();
    if (threadIdx.x < TM_NV) partial[((size_t)ch * nt + ip) * TM_NV + threadIdx.x] = acc[threadIdx.x];
    __syncthreads();
  }
}

}  // namespace mcre

using namespace mcre;

extern "C" int mcre_lsm_step_tangents(int32_t nt, const double *d_xk, const double *d_nk, const double *d_dxk,
                                      const double *d_dnk, double shift_k, double scale_k, const double *d_xi,
                                      const double *d_ni, const double *d_imm, const double *d_dni, const double *d_dimm,
                                      const double *coef_i, double shift_i, double scale_i, const float *d_value,
                                      double *d_dvalue, int64_t n, int32_t chunk_paths, double *d_partial,
                                      double *d_tmoments, void *stream) {
  if (!d_xk || !d_nk || !d_dxk || !d_dnk || !d_value || !d_dvalue || !d_partial || !d_tmoments)
    return fail(-1, "null argument%s", "");
  if (nt < 1) return fail(-1, "lsm tangents: nt must be positive%s", "");
  if (d_imm && (!d_xi || !d_ni || !d_dni || !d_dimm)) return fail(-1, "lsm tangents: exercise update needs its arrays%s", "");
  if (chunk_paths <= 0 || chunk_paths % 256 != 0) return fail(-2, "lsm: chunk_paths must be a positive multiple of 256%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  if (n <= 0) {
    MCRE_CUDA(cudaMemsetAsync(d_tmoments, 0, (size_t)nt * TM_NV * sizeof(double), st));
    return 0;
  }
  const long long n_chunks = (n + chunk_paths - 1) / chunk_paths;
  long long gx = (long long)sm_count() * 4;
  if (gx > n_chunks) gx = n_chunks;
  dim3 grid((unsigned)gx, (unsigned)nt);
  lsm_step_tan_kernel<<<grid, 256, 0, st>>>(nt, d_xk, d_nk, d_dxk, d_dnk, shift_k, scale_k, d_xi, d_ni, d_imm, d_dni, d_dimm,
                                            coef_i != nullptr, coef_i ? coef_i[0] : 0.0, coef_i ? coef_i[1] : 0.0,
                                            coef_i ? coef_i[2] : 0.0, shift_i, scale_i, d_value, d_dvalue, n, chunk_paths,
                                            d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, (int64_t)nt * TM_NV, d_tmoments, stream);
}

template <int NT>
static int launch_lsm_forward_tan(const IrcDev &d, const RngDev &r, const ShardDev &sh, double *x, double *nn, double *im,
                                  double *dx, double *dn, double *di, cudaStream_t st) {
  const int threads = 128;
  const unsigned blocks = (unsigned)((sh.n_paths + threads - 1) / threads);
  if (d.has_cir) irc_lsm_forward_tan_kernel<NT, true, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, x, nn, im, dx, dn, di);
  else if (d.scheme == MCRE_SCHEME_ANALYTICAL)
    irc_lsm_forward_tan_kernel<NT, false, MCRE_SCHEME_ANALYTICAL><<<blocks, threads, 0, st>>>(d, r, sh, x, nn, im, dx, dn, di);
  else irc_lsm_forward_tan_kernel<NT, false, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, x, nn, im, dx, dn, di);
  MCRE_LAUNCHED();
  return 0;
}

// called by mcre_irc_lsm_forward when the plan carries tangents
int irc_lsm_forward_tangent_pass(mcre_irc_plan *p, const RngDev &r, const ShardDev &sh, void *d_scratch, cudaStream_t st) {
  const IrcDev &d = p->d;
  const long long n = sh.n_paths;
  double *x = (double *)d_scratch;
  double *nn = x + (size_t)d.n_reg * n;
  double *im = nn + (size_t)d.n_reg * n;
  double *dx = im + (size_t)d.n_ex * n;
  double *dn = dx + (size_t)d.n_reg * d.nt * n;
  double *di = dn + (size_t)d.n_reg * d.nt * n;
  return d.nt == 4 ? launch_lsm_forward_tan<4>(d, r, sh, x, nn, im, dx, dn, di, st)
                   : launch_lsm_forward_tan<8>(d, r, sh, x, nn, im, dx, dn, di, st);
}

extern "C" int64_t mcre_irc_presim_tangent_slots(const mcre_irc_plan *p) {
  return (int64_t)p->d.n_units * p->d.nt * p->d.n_reg * TM_NV;
}

template <int NT>
static int launch_forward_tan(const IrcDev &d, const RngDev &r, const ShardDev &sh, double *xbuf, double *nbuf,
                              float *wbuf, double *dx, double *dn, double *dw, cudaStream_t st) {
  const int threads = 128;
  const unsigned blocks = (unsigned)((sh.n_paths + threads - 1) / threads);
  if (d.has_cir)
    irc_presim_forward_tan_kernel<NT, true, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf, dx, dn, dw);
  else if (d.scheme == MCRE_SCHEME_ANALYTICAL)
    irc_presim_forward_tan_kernel<NT, false, MCRE_SCHEME_ANALYTICAL><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf, dx, dn, dw);
  else
    irc_presim_forward_tan_kernel<NT, false, MCRE_SCHEME_EULER><<<blocks, threads, 0, st>>>(d, r, sh, xbuf, nbuf, wbuf, dx, dn, dw);
  MCRE_LAUNCHED();
  return 0;
}

static size_t tangent_moments_smem(const IrcDev &d) { return ((size_t)d.n_reg * TM_NV + 2 * (256 / 32) * TM_NV) * sizeof(double); }

// Checks that the tangent moments kernel fits the plan's regression dates (and requests its shared memory); called by
// mcre_irc_presim before anything is launched.
int irc_presim_tangent_fit(const mcre_irc_plan *p) {
  MCRE_SMEM(irc_presim_tangent_moments_kernel, tangent_moments_smem(p->d),
            "irc tangent presim kernel does not fit: too many regression dates (%s%lld bytes of shared memory)");
  return 0;
}

// Forward pass with tangents + tangent moments; the value moments of the same scratch are
// accumulated by mcre_irc_presim (which calls this first when the plan carries tangents).
int irc_presim_tangent_pass(mcre_irc_plan *p, const RngDev &r, const ShardDev &sh, void *d_scratch, double *d_partial,
                            double *d_tmoments, cudaStream_t st) {
  const IrcDev &d = p->d;
  const long long n = sh.n_paths;
  double *xbuf = (double *)d_scratch;
  double *nbuf = xbuf + (size_t)d.n_reg * n;
  float *wbuf = (float *)(nbuf + (size_t)d.n_reg * n);
  const size_t wcount = (size_t)d.n_units * d.n_reg * n;
  double *dx = (double *)(wbuf + ((wcount + 1) & ~(size_t)1));
  double *dn = dx + (size_t)d.n_reg * d.nt * n;
  double *dw = dn + (size_t)d.n_reg * d.nt * n;
  int rc = d.nt == 4 ? launch_forward_tan<4>(d, r, sh, xbuf, nbuf, wbuf, dx, dn, dw, st)
                     : launch_forward_tan<8>(d, r, sh, xbuf, nbuf, wbuf, dx, dn, dw, st);
  if (rc) return rc;
  const int threads = 256;
  const size_t smem = tangent_moments_smem(d);
  const long long n_chunks = (n + sh.chunk - 1) / sh.chunk;
  auto k = irc_presim_tangent_moments_kernel;
  int per_sm = 1;
  MCRE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, threads, smem));
  if (per_sm < 1) return fail(-3, "irc tangent presim kernel does not fit: too many regression dates%s", "");
  long long gx = (long long)sm_count() * per_sm;
  if (gx > n_chunks) gx = n_chunks;
  dim3 grid((unsigned)gx, (unsigned)d.nt, (unsigned)d.n_units);
  k<<<grid, threads, smem, st>>>(d, sh, d.nt, xbuf, nbuf, wbuf, dx, dn, dw, d_partial);
  MCRE_LAUNCHED();
  return mcre_tree_reduce(d_partial, n_chunks, mcre_irc_presim_tangent_slots(p), d_tmoments, st);
}
