// Device side of the exposure regression of linear rate products: solves the 3x3 normal equations of every
// regression date from the all-reduced moments and patches the coefficients into the main plan's per-date records,
// so that pre-simulation -> solve -> main simulation is one stream of kernels without a device-to-host round trip.
//
// Replaces torch.linalg.lstsq of controller.py:368-374 (driver gelsy: minimum-norm solution for rank-deficient
// designs - at t = 0 every path has the same explanatory value) with the same decision rule as the host solver
// mcre/lsm.py:solve_normal_equations: equilibrate the Gram matrix by its diagonal; full rank (smallest / largest
// eigenvalue of the equilibrated matrix > 1e-10): Gaussian elimination with partial pivoting; otherwise the
// pseudo-inverse of the unscaled Gram matrix with the same relative threshold on its eigenvalues.
#include "irc_main.cuh"
#include "solve3.cuh"

namespace mcre {

// One thread per regression date: coefficients of every unit and their per-set sums.
// moments [n_reg][5 + 3 nu_t]; unit_set[u] = netting-set row of unit u (or -1); coef_unit [n_units][n_reg][3];
// coef_sum [n_reg][n_sets][3].
struct UnitSets { int row[MCRE_IRC_MAX_UNITS]; };
__global__ void irc_solve_kernel(const double *__restrict__ moments, int n_reg, int n_units, int nu_t, int n_sets,
                                 UnitSets unit_set, double *__restrict__ coef_unit, double *__restrict__ coef_sum) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_reg) return;
  const double *m = moments + (size_t)k * (5 + 3 * nu_t);
  for (int r = 0; r < n_sets; ++r)
    for (int j = 0; j < 3; ++j) coef_sum[((size_t)k * n_sets + r) * 3 + j] = 0.0;
  for (int u = 0; u < n_units; ++u) {
    double c[3];
    solve_normal_equations_dev(m, m + 5 + 3 * u, c);
    for (int j = 0; j < 3; ++j) coef_unit[((size_t)u * n_reg + k) * 3 + j] = c[j];
    const int r = unit_set.row[u];
    if (r >= 0 && r < n_sets)
      for (int j = 0; j < 3; ++j) coef_sum[((size_t)k * n_sets + r) * 3 + j] += c[j];
  }
}

// Patches value-only coefficients [n_expo][n_sets][3] (standardised basis) into the main plan on the device: the
// expo_coef table, the packed per-date records of the general kernel and, for the CVA-only kernel, the event records
// (raw monomial basis, scaled by g_k = 1/2 exp(-sum psi dt), see irc_cva.cu).
__global__ void irc_patch_coefficients_kernel(const double *__restrict__ coef, int n_dates, int n_sets, int DR,
                                              const int *__restrict__ date_expo, double *__restrict__ expo_coef,
                                              double *__restrict__ date_rec, double *__restrict__ cva_rec, int n_events) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_dates) {
    const int e = date_expo[i];
    if (e >= 0) {
      double *r = date_rec + (size_t)i * DR + DATE_HDR + 2;
      for (int k = 0; k < 3 * n_sets; ++k) {
        const double cv = coef[(size_t)e * 3 * n_sets + k];
        r[k] = cv;
        expo_coef[(size_t)e * 3 * n_sets + k] = cv;
      }
    }
  }
  if (cva_rec && i < n_events) {
    double *r = cva_rec + (size_t)i * CVA_REC;
    const int di = __double2loint(r[23]) - 1;      // date closed by the event (+1), 0: none
    if (di >= 0) {
      const int e = date_expo[di];
      const double g = r[22];
      if (e >= 0) {
        const double *dr = date_rec + (size_t)di * DR;
        const double sh = dr[4], sc = dr[5];
        double raw[3];
        irc_raw_basis(coef[(size_t)e * 3], coef[(size_t)e * 3 + 1], coef[(size_t)e * 3 + 2], sh, sc, raw);
        r[12] = __dmul_rn(g, raw[2]);
        r[11] = __dmul_rn(g, raw[1]);
        r[10] = __dmul_rn(g, raw[0]);
      }
    }
  }
}

}  // namespace mcre

using namespace mcre;

static int nu_template_(int n_units) { return n_units <= 1 ? 1 : (n_units <= 2 ? 2 : 4); }

extern "C" int mcre_irc_solve_coefficients(const mcre_irc_plan *pre, const double *d_moments, const int32_t *unit_set,
                                           int32_t n_sets, double *d_coef_unit, double *d_coef_sum, void *stream) {
  if (!pre || !d_moments || !unit_set || !d_coef_unit || !d_coef_sum) return fail(-1, "null argument%s", "");
  if (pre->d.nt != 0) return fail(-1, "irc solve: value-only plans only (tangent plans are solved on the host)%s", "");
  const int n_reg = pre->d.n_reg, n_units = pre->d.n_units;
  if (n_reg == 0 || n_units == 0) return 0;
  if (n_sets < 1 || n_sets > MCRE_IRC_MAX_SETS) return fail(-1, "irc solve: n_sets out of range%s", "");
  cudaStream_t st = (cudaStream_t)stream;
  UnitSets us;
  for (int u = 0; u < MCRE_IRC_MAX_UNITS; ++u) us.row[u] = u < n_units ? unit_set[u] : -1;
  irc_solve_kernel<<<(n_reg + 63) / 64, 64, 0, st>>>(d_moments, n_reg, n_units, nu_template_(n_units), n_sets, us,
                                                     d_coef_unit, d_coef_sum);
  MCRE_LAUNCHED();
  return 0;
}

extern "C" int mcre_irc_set_coefficients_device(mcre_irc_plan *p, const double *d_coef, void *stream) {
  if (!p || !d_coef) return fail(-1, "null argument%s", "");
  if (p->d.nt != 0) return fail(-1, "irc: device coefficients are value-only%s", "");
  if (p->expo_coef_count == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int n = p->cva_only ? (p->d.n_dates > p->cva.n_pre_dates + p->cva.n_sub ? p->d.n_dates : p->cva.n_pre_dates + p->cva.n_sub)
                            : p->d.n_dates;
  irc_patch_coefficients_kernel<<<(n + 127) / 128, 128, 0, st>>>(
      d_coef, p->d.n_dates, p->d.n_sets, p->date_stride, p->d.date_expo, p->d.expo_coef, (double *)p->d.date_rec,
      p->cva_only ? p->cva_rec_dev : nullptr, p->cva_only ? p->cva.n_pre_dates + p->cva.n_sub : 0);
  MCRE_LAUNCHED();
  return 0;
}
