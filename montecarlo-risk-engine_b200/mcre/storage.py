"""Backend for books of gas storages on a Schwartz two-factor model (csrc/storage.cu).

Replaces, for `products.storage.Storage`, the reference's pre-simulation + backward induction
(src/controller/controller.py:272-383) and valuation pass (:385-471, PV branch) with

  pre-simulation : one forward launch spilling the spot of every action date, then one launch per action date
                   (backwards) that advances the value grid [state][path] of ALL paths and states;
  regression     : per action date a tall least squares of the value grid on the polynomial basis of the spot.
                   Two solvers (`SimulationController.storage_regression`):
                     "lapack"  - the design matrix and the value grid are read back and solved by LAPACK gelsy
                                 through torch.linalg.lstsq, the very routine the reference calls.  Default up to
                                 LAPACK_MAX_PATHS pre-simulation paths, because the reference's results depend on that
                                 routine's rank decisions wherever prices are (nearly) deterministic: on the
                                 reference's own `storage1` known answer a mathematically equivalent solver moves the
                                 PV by 1.7e-3 (exact ties between "inject today" and "inject tomorrow" are broken
                                 by the least-squares noise).  Only the [N x basis] solve runs on the host - paths,
                                 decisions and value grids stay on the GPU;
                     "moments" - Gram / right-hand-side moments of the standardised basis accumulated on the device
                                 (fixed-order chunk tree, all-reduced over ranks), (basis x basis) normal equations
                                 solved on the device by Jacobi diagonalisation with a minimum-norm cut-off: the whole
                                 induction is one stream of kernels; paths are sharded over the GPUs.  Default above
                                 that size;
  main simulation: one fused launch per product (stepping + decisions + cashflows), per-path totals of a netting
                   set accumulated on the device, mean and standard error by mcre_sum_stats.
"""
from __future__ import annotations

import ctypes as C
import math
import time

import numpy as np
import torch

from common.enums import SimulationScheme
from mcre import binding as B
from mcre import runtime as RT
from mcre.finish import mean_and_error
from mcre.timegrid import build_time_grid

#: largest pre-simulation for which the regression is solved by LAPACK on the host by default
LAPACK_MAX_PATHS = 1 << 16
STEP = 24
MAX_NOISE = 8
TAN = 7


def _is_storage(p):
    from products.storage import Storage
    return isinstance(p, Storage)


def _is_bs(model):
    from models.black_scholes import BlackScholesModel
    return type(model) is BlackScholesModel


def _is_bsm(model):
    from models.black_scholes_multi import BlackScholesMulti
    return isinstance(model, BlackScholesMulti)


def price_model_of(model, asset_id):
    """(sub-model that simulates `asset_id`, its first noise column in the model's joint draw, joint noise dimension,
    numeraire model).  A plain model is its own price and numeraire model; in a ModelConfig (model_config.py:8-77) the
    sub-models' draws are concatenated."""
    from models.model_config import ModelConfig
    if not isinstance(model, ModelConfig):
        return model, 0, int(model.simulation_dim), model
    off = 0
    for m in model.models:
        if asset_id in m.asset_ids:
            return m, off, int(model.simulation_dim), model.models[model.id_to_model["numeraire"]]
        off += int(m.simulation_dim)
    raise ValueError(f"Asset id '{asset_id}' not found in model asset ids {list(model.asset_ids)}.")


def rate_of(model):
    """Rate parameter of a (numeraire) model."""
    return model.param_values()[2 * model.num_assets if _is_bsm(model) else (2 if _is_bs(model) else 0)]


def tangent_slots(model, asset_id=None):
    """-> (slots, numeraire slot): the flattened parameter index of each tangent slot of a storage on `asset_id`, and the
    slot of the numeraire model's rate.  The slots are the parameters the storage's step depends on - the lane
    parameters of mcre/equity.py:family_of (spot, volatility, rate of a Black-Scholes asset; the six Schwartz
    parameters) - and, when the numeraire is another model of a ModelConfig, that model's rate (its discount factors)."""
    from mcre.equity import EquityBackend, family_of
    from models.model_config import ModelConfig
    fam = family_of(model)
    if fam is None:
        raise NotImplementedError("gas storage: sensitivities on Schwartz two-factor, Black-Scholes and Black-Scholes "
                                  "multi-asset models, or a ModelConfig of Black-Scholes models")
    _, assets = fam
    asset = assets[0] if len(assets) == 1 else next(a for a in assets if a.asset_id == asset_id)
    if isinstance(model, ModelConfig):
        num_idx = model.id_to_model["numeraire"]
        num_global = model.param_offsets()[num_idx] + EquityBackend._rate_index(model.models[num_idx])
    else:
        num_global = EquityBackend._rate_index(model)
    slots = list(asset.gmap)
    if num_global not in slots:
        slots.append(num_global)
    return slots, slots.index(num_global)


def step_table(model, grid, scheme, nt=0, asset_id=None, kernel_record=False):
    """-> (steps [n_sub][STEP], tangents [n_sub][nt][6] or None): records of csrc/storage.cu:TwoFactor and, for
    pathwise sensitivities, d(A, B00, M, B10, B11, log F) / d(slot) of the effective recursion x' = A x + B00 z0,
    y' = y + M + B10 z0 + B11 z1, or of the Black-Scholes EULER step (host duals, mcre/dual.py); kernel_record: the
    kernel's [n_sub][nt][TAN] records, which also hold d Bw, the tangent that scales the combined draw w0.  The
    slots are the storage's own (tangent_slots): nt = 6 Schwartz parameters, or 3 (spot, volatility, rate of the asset's
    model) + an optional 4th, the numeraire model's rate, on which no step depends.
    Schwartz two-factor (schwartz_two_factor.py:124-196), parameters [rate, kappa, sigma_s, mu_l, sigma_l, rho]:
      ANALYTICAL  a = exp(-kappa dt), b = Cholesky factor of the step covariance (cached per nominal dt, model.py:45-64)
      EULER       a = 1, k = kappa, cx / cy = sigma sqrt(dt), b = Cholesky factor of the correlation - which the
                  reference builds before requires_grad(): rho is a constant of its autograd graph there
    Black-Scholes (black_scholes.py:50-67, parameters [spot, sigma, rate]), ANALYTICAL: the log-price accumulates in
    x (bx_0 = sqrt(sigma^2 dt)), its drift (rate - sigma^2 / 2) dt in m, log F = log spot.
    Black-Scholes multi-asset (black_scholes_multi.py:63-79) or a Black-Scholes model of a ModelConfig, ANALYTICAL: the
    same for the asset `asset_id` with bx = its row of the Cholesky factor of the step covariance D C D dt of all assets
    - the draw is the model's joint one.  That row is sigma_a sqrt(dt) L_C[a, :], so d bx = bx d log sigma_a: the
    tangent multiplies the combined draw w0 (Bw = log sigma_a), and the other assets' volatilities do not reach it.
    EULER (black_scholes.py:69-85, black_scholes_multi.py:81-97): x' = x + log1p(m + cx w0), m = rate dt,
    cx = sigma sqrt(dt), bx = the asset's row of the Cholesky factor of the correlation (a constant); the tangent record
    holds dM = d m, dBw = d cx and d log F."""
    from mcre.dual import D, dexp, dlog, dsqrt
    joint = model
    model, noise_off, noise_dim, _ = price_model_of(joint, asset_id)
    if noise_dim > MAX_NOISE:
        raise NotImplementedError(f"gas storage: price models with at most {MAX_NOISE} noise factors")
    zero, one = D(0.0, None, nt), D(1.0, None, nt)
    out = np.zeros((max(grid.n_sub, 1), STEP))
    tan = np.zeros((max(grid.n_sub, 1), nt, TAN)) if nt else None
    chol = {}
    black_scholes = _is_bs(model) or _is_bsm(model)
    if black_scholes:
        n = model.num_assets if _is_bsm(model) else 1
        ai = model.asset_ids.index(asset_id) if _is_bsm(model) else 0
        vals = model.param_values()
        # (slots 0, 1, 2: spot, volatility, rate of the asset; the same order as dual_params of a BlackScholesModel)
        spot, sig, rate = [D.var(v, k, nt) if nt else D(v, None, 0) for k, v in enumerate((vals[ai], vals[n + ai], vals[2 * n]))]
    else:
        p = model.dual_params(0, nt)
    if black_scholes and scheme not in (SimulationScheme.ANALYTICAL, SimulationScheme.EULER):
        raise NotImplementedError(f"gas storage on Black-Scholes models: scheme {scheme}")

    def joint_factor(key):
        """Lower Cholesky factor of the joint step covariance (ANALYTICAL) / correlation (EULER) of the whole draw
        (model.py:50-73, model_config.py:101-221; raises like the reference for pairs without a joint covariance)."""
        from mcre.paths import joint_matrix
        if key not in chol:
            chol[key] = np.linalg.cholesky(np.array(joint_matrix(joint, scheme, key)))
        return chol[key]
    for s in range(grid.n_sub):
        dt = grid.dt[s]
        bx, by = [zero] * MAX_NOISE, [zero] * MAX_NOISE
        bw = zero
        euler_bs = 0.0
        if black_scholes:
            col = noise_off + ai
            a, k, cx, cy, lf = one, zero, one, zero, dlog(spot)
            if scheme == SimulationScheme.EULER:
                # S' = S + (r S dt + sigma S sqrt(dt) w): multiplicative, carried as log1p in the kernel
                L = joint_factor(None)
                m, cx, euler_bs = rate * dt, sig * math.sqrt(dt), 1.0
                bx = [D(float(L[col, j]), None, nt) if j <= col else zero for j in range(MAX_NOISE)]
            elif _is_bs(model) and joint is model:
                m = rate * dt - 0.5 * dt * sig * sig
                bx = [dsqrt(sig * sig * grid.dt_nominal[s])] + [zero] * (MAX_NOISE - 1)
            else:
                L = joint_factor(grid.dt_nominal[s])
                m = (rate - 0.5 * sig * sig) * dt if _is_bsm(model) else rate * dt - 0.5 * dt * sig * sig
                bx = [D(float(L[col, j]), None, nt) if j <= col else zero for j in range(MAX_NOISE)]
                bw = dlog(sig)
        else:
            rate, kappa, sig_s, mu, sig_l, rho = p
            if scheme == SimulationScheme.ANALYTICAL:
                key = grid.dt_nominal[s]            # the reference caches the factor per nominal dt
                if key not in chol:
                    if abs(kappa.v) <= 1e-12:
                        var_s = sig_s * sig_s * key
                    else:
                        var_s = sig_s * sig_s * (1.0 - dexp(-2.0 * kappa * key)) / (2.0 * kappa)
                    var_l = sig_l * sig_l * key
                    cov = rho * dsqrt(var_s * var_l)
                    l00 = dsqrt(var_s)
                    l10 = cov / l00
                    chol[key] = (l00, l10, dsqrt(var_l - l10 * l10))
                a = one if abs(kappa.v) <= 1e-12 else dexp(-kappa * dt)
                k, m, cx, cy = zero, mu * dt, one, one
                bx = [chol[key][0]] + [zero] * (MAX_NOISE - 1)
                by = [chol[key][1], chol[key][2]] + [zero] * (MAX_NOISE - 2)
            elif scheme == SimulationScheme.EULER:
                sq = math.sqrt(dt)
                rho_c = rho.v                         # constant of the reference's graph under EULER
                a, k, m = one, kappa, mu * dt
                cx, cy = sig_s * sq, sig_l * sq
                bx = [one] + [zero] * (MAX_NOISE - 1)
                by = [D(rho_c, None, nt), D(math.sqrt(1.0 - rho_c * rho_c), None, nt)] + [zero] * (MAX_NOISE - 2)
            else:
                raise NotImplementedError(f"storage: scheme {scheme} is not defined for the Schwartz two-factor model")
            lf = D(math.log(model.curve_value(grid.t2[s])), None, nt)
        val = lambda x: x.v if isinstance(x, D) else x   # noqa: E731
        out[s, :7] = [val(x) for x in (a, k, dt, m, cx, cy, lf)]
        out[s, 7] = euler_bs
        out[s, 8:8 + MAX_NOISE] = [val(x) for x in bx]
        out[s, 16:16 + MAX_NOISE] = [val(x) for x in by]
        if nt:
            if euler_bs:
                eff = (zero, zero, m, zero, zero, lf, cx)
            else:
                eff = (a - k * dt, cx * bx[0], m, cy * by[0], cy * by[1], lf, bw)
            for j, e in enumerate(eff):
                tan[s, :, j] = D.lift(e, nt).t
    return out, (tan if tan is None or kernel_record else tan[:, :, :6])


def log_spot_scale(model, t):
    """Standard deviation of log S(t) under the model: a per-date scale for the standardised basis."""
    from models.model_config import ModelConfig
    if isinstance(model, ModelConfig):
        return max(log_spot_scale(m, t) for m in model.models if _is_bs(m) or _is_bsm(m))
    tau = max(t - model.t0(), 0.0)
    if _is_bs(model):
        return model.param_values()[1] * math.sqrt(tau)
    if _is_bsm(model):
        return max(model.param_values()[model.num_assets:2 * model.num_assets]) * math.sqrt(tau)
    _, kappa, sig_s, _, sig_l, rho = model.param_values()
    if abs(kappa) <= 1e-12:
        var_s, cov = sig_s * sig_s * tau, rho * sig_s * sig_l * tau
    else:
        var_s = sig_s * sig_s * (1.0 - math.exp(-2.0 * kappa * tau)) / (2.0 * kappa)
        cov = rho * sig_s * sig_l * (1.0 - math.exp(-kappa * tau)) / kappa
    return math.sqrt(max(var_s + sig_l * sig_l * tau + 2.0 * cov, 0.0))


class StorageBackend:
    @staticmethod
    def supports(ctrl):
        return any(_is_storage(p) for p in ctrl.products)

    def __init__(self, ctrl):
        from maths.regression import PolyomialRegression
        from metrics.metric import MetricType
        from models.schwartz_two_factor import SchwartzTwoFactorModel
        self.c = c = ctrl
        #: storages next to other equity products in the same run (the reference's 50k-product book,
        #: tests/pv_tests/pv_performance_large_netting_set.py): the storages' per-path cashflows start the PV
        #: accumulators of the equity launches (mcre/equity.py:_run_split_book, extra_pv)
        self.mixed = not all(_is_storage(p) for p in c.products)
        from models.cirpp import CIRPPModel
        from models.model_config import ModelConfig
        subs = list(c.model.models) if isinstance(c.model, ModelConfig) else [c.model]
        self.standalone = not isinstance(c.model, ModelConfig)
        for m in subs:
            ok = _is_bs(m) or _is_bsm(m) or (isinstance(m, SchwartzTwoFactorModel) and self.standalone) \
                or (isinstance(m, CIRPPModel) and not self.standalone)
            if not ok:
                raise NotImplementedError("gas storage: SchwartzTwoFactorModel, BlackScholesModel, BlackScholesMulti, or a "
                                          f"ModelConfig of Black-Scholes models and a credit model (got {type(m).__name__})")
        kinds = {m.metric_type for m in c.risk_metrics.metrics}
        if MetricType.CVA in kinds and not self.mixed:
            raise NotImplementedError("gas storage: CVA of a book of storages alone (the default weights ride with an equity "
                                      "launch of the same netting set)")
        self.need_expo = c.risk_metrics.requires_exposure_profiles()
        if c.differentiate and self.need_expo:
            raise NotImplementedError("gas storage: sensitivities of exposure metrics and CVA (PV sensitivities only)")
        if c.differentiate and any(isinstance(m, CIRPPModel) for m in subs):
            raise NotImplementedError("gas storage: sensitivities in a ModelConfig with a credit model")
        for p in c.products:
            if _is_storage(p):
                price_model_of(c.model, p.get_asset_id())      # raises for an unknown asset id
        num_model = price_model_of(c.model, [p for p in c.products if _is_storage(p)][0].get_asset_id())[3]
        self.num_rate = rate_of(num_model)
        #: tangent slots of each storage (tangent_slots): asset id -> (flattened parameter index per slot, numeraire slot)
        self.slots = {}
        if c.differentiate:
            for p in c.products:
                if _is_storage(p) and p.get_asset_id() not in self.slots:
                    self.slots[p.get_asset_id()] = tangent_slots(c.model, p.get_asset_id())
        #: tangent slots per storage lane (csrc/storage.cu:storage_main_kernel<NT>); 0: values only
        self.nt = max(len(g) for g, _ in self.slots.values()) if self.slots else 0
        self.noise_dim = int(c.model.simulation_dim)
        if self.noise_dim > MAX_NOISE:
            raise NotImplementedError(f"gas storage: price models with at most {MAX_NOISE} noise factors")
        rf = c.regression_function
        if type(rf) is not PolyomialRegression or not 0 <= rf.degree < B_MAX_BASIS:
            raise NotImplementedError(f"gas storage: PolyomialRegression of degree 0..{B_MAX_BASIS - 1} (the kernels "
                                      "evaluate monomials of the spot)")
        self.n_basis = rf.degree + 1
        mode = getattr(c, "storage_regression", "auto")
        if mode not in ("auto", "lapack", "moments"):
            raise ValueError("storage_regression must be 'auto', 'lapack' or 'moments'")
        if mode == "auto":
            mode = "lapack" if c.num_paths_presim <= LAPACK_MAX_PATHS else "moments"
        self.mode = mode

    # ------------------------------------------------------------------ plan
    def _spot0(self, prod):
        m = price_model_of(self.c.model, prod.get_asset_id())[0]
        if _is_bsm(m):
            return m.param_values()[m.asset_ids.index(prod.get_asset_id())]
        return m.param_values()[0] if _is_bs(m) else m.curve_value(m.t0())

    def _create(self, prod, grid, steps, steps_tan):
        c = self.c
        sim_dates = grid.index_map()
        acts = prod.product_timeline.tolist()
        date_of = {sim_dates[t]: k for k, t in enumerate(acts)}
        step_date = np.array([date_of.get(d, -1) if d >= 0 else -1 for d in grid.date_after], dtype=np.int32)
        n_pre = sum(1 for t in acts if sim_dates[t] < grid.n_pre_dates)
        rec = prod.lower()
        t0 = self._t0()
        rate = self.num_rate
        numeraire = np.array([math.exp(rate * (t - t0)) for t in acts])
        slots, num_slot = self.slots.get(prod.get_asset_id(), ([], 0))
        nt = len(slots)
        dlog_num = np.zeros((len(acts), max(nt, 1)))
        if nt:
            dlog_num[:, num_slot] = [t - t0 for t in acts]
        keep = []
        d = B.StorageDesc()
        d.n_sub, d.n_dates, d.n_pre_dates = grid.n_sub, len(acts), n_pre
        d.n_states, d.n_basis = prod.num_states, self.n_basis
        d.log_spot0 = math.log(self._spot0(prod))
        d.noise_dim, d.n_tan = self.noise_dim, nt
        expo_times = c.exposure_timeline.tolist() if self.need_expo else []
        for t in expo_times:
            # two dates one rounding error apart share a simulation date; the kernel acts before it reads the exposure of
            # that date, which is the reference's order only if the action date is not the later of the two
            if any(sim_dates[ta] == sim_dates[t] and ta > t for ta in acts):
                raise NotImplementedError(f"exposure date {t!r} lies one rounding error before an action date of a storage")
        expo_of = {sim_dates[t]: e for e, t in enumerate(expo_times)}
        step_expo = np.array([expo_of.get(di, -1) if di >= 0 else -1 for di in grid.date_after], dtype=np.int32)
        d.n_expo = len(expo_times)
        d.n_pre_expo = sum(1 for t in expo_times if sim_dates[t] < grid.n_pre_dates)
        expo_num = np.array([math.exp(rate * (t - t0)) for t in expo_times]) if expo_times else np.zeros(1)
        for name, arr, conv in (("step_expo", step_expo if (grid.n_sub and expo_times) else np.zeros(1, np.int32), B.as_ip),
                                ("expo_numeraire", expo_num, B.as_dp),
                                ("step_tan", steps_tan if nt else np.zeros(1), B.as_dp), ("dlog_num", dlog_num, B.as_dp),
                                ("step", steps, B.as_dp), ("step_date", step_date if grid.n_sub else np.zeros(1, np.int32), B.as_ip),
                                ("date_rec", rec, B.as_dp), ("numeraire", numeraire, B.as_dp)):
            a, ptr = conv(arr)
            keep.append(a)
            setattr(d, name, ptr)
        plan = C.c_void_p()
        B.check(B.lib().mcre_storage_create(C.byref(d), C.byref(plan)))
        return plan, numeraire, acts, expo_num

    def _rng(self, which, seed, n_total):
        c = self.c
        rng = B.Rng()
        rng.seed, rng.stream, rng.n_paths_total = seed, c.rng_stream, n_total
        z = c.injected_normals.get(which) if c.injected_normals else None
        if z is not None:
            if z.shape[1] != n_total or z.shape[2] != self.noise_dim:
                raise ValueError(f"injected {which} normals must be [n_sub, {n_total}, {self.noise_dim}]")
            rng.mode, rng.d_z = B.RNG_INJECT, z.data_ptr()
        else:
            rng.mode = B.RNG_PHILOX
        return rng, z

    # ------------------------------------------------------------------ pre-simulation + regression
    def _t0(self):
        m = self.c.model
        return (m if self.standalone else m.models[0]).t0()

    def _forward(self, t, prod):
        m = price_model_of(self.c.model, prod.get_asset_id())[0]
        if _is_bs(m) or _is_bsm(m):
            return self._spot0(prod) * math.exp(rate_of(m) * (t - m.t0()))
        return m.curve_value(t)

    def _regress(self, prod, plan, numeraire, acts, expo_num, dev):
        """-> (coef [n_dates][2 + S * NB], coef_expo [n_expo][2 + S * NB] or None) on the device: (centre, inverse scale,
        coefficients per state) of the continuation polynomials per action date and per exposure date.
        controller.py:294-383: walking the dates backwards, the value grid of action date k (per state entering it) is
        regressed on the spot of the action date before it and on the spot of every exposure date in (T_k-1, T_k)
        (and of one equal to T_k-1: the same system); exposure dates from the last action date on get zeros."""
        c, L = self.c, B.lib()
        S, NB, n_dates = prod.num_states, self.n_basis, len(acts)
        row = 2 + S * NB
        n_total = c.num_paths_presim
        rank, world = RT.dist_info()
        chunk = 256 if n_total < (1 << 18) else 4096
        if self.mode == "lapack" or world == 1:
            begin, count = 0, n_total            # (lapack: every rank solves the same full-size systems)
        else:
            begin, count = RT.shard_range(n_total, chunk)
        rng, _keep = self._rng("pre", 42, n_total)
        shard = B.Shard(begin, count, chunk)
        expo_times = c.exposure_timeline.tolist() if self.need_expo else []
        n_expo = len(expo_times)
        # value grid each exposure date is regressed on: the first action date AFTER it (an action on the exposure date
        # itself has been taken when the exposure is read, controller.py:417-430)
        next_action = [int(np.searchsorted(acts, t, side="right")) for t in expo_times]
        expo_of_k = {}
        for e, k in enumerate(next_action):
            expo_of_k.setdefault(k, []).append(e)
        spot = torch.empty((n_dates, max(count, 1)), dtype=torch.float64, device=dev)
        spot_e = torch.empty((n_expo, max(count, 1)), dtype=torch.float64, device=dev) if n_expo else None
        B.check(L.mcre_storage_spots(plan, C.byref(rng), C.byref(shard), spot.data_ptr(),
                                     spot_e.data_ptr() if n_expo else None, RT.stream_ptr()))

        def basis_rows(times):
            h = np.zeros((len(times), row))
            h[:, 1] = 1.0
            if self.mode == "moments":
                for i, t in enumerate(times):
                    f = self._forward(t, prod)
                    sd = f * log_spot_scale(c.model, t)
                    h[i, 0], h[i, 1] = f, (1.0 / sd if sd > 1e-300 else 0.0)
            return h
        coef_h, coef_eh = basis_rows(acts), basis_rows(expo_times)
        coef = torch.from_numpy(coef_h.copy()).to(dev)
        coef_e = torch.from_numpy(coef_eh.copy()).to(dev) if n_expo else None
        value = torch.zeros((S, max(count, 1)), dtype=torch.float64, device=dev)
        if self.mode == "lapack":
            spot_h = RT.to_host(spot)
            spot_eh = RT.to_host(spot_e) if n_expo else None
        else:
            slots = L.mcre_storage_moment_slots(plan)
            n_chunks = (count + chunk - 1) // chunk
            partial = torch.empty(max(n_chunks, 1) * slots, dtype=torch.float64, device=dev)
            mom = torch.zeros(slots, dtype=torch.float64, device=dev)
        value_h = [None]

        def solve(x_host, x_dev, num, host_row, dev_row):
            """Regression of numeraire x value grid on the basis of one date's spot -> host_row / dev_row [2 + S NB]."""
            if self.mode == "lapack":
                # controller.py:361-374: A = [x^0 .. x^degree], solution of min |A c - numeraire * value| by gelsy
                if value_h[0] is None:
                    value_h[0] = torch.from_numpy(RT.to_host(value)).transpose(0, 1)
                A = c.regression_function.get_regression_matrix(torch.from_numpy(x_host))
                sol = torch.linalg.lstsq(A, value_h[0] * float(num)).solution            # [NB, S]
                host_row[2:] = sol.transpose(0, 1).reshape(-1).numpy()
                dev_row.copy_(torch.from_numpy(host_row), non_blocking=False)
            else:
                B.check(L.mcre_storage_moments(plan, float(num), host_row[0], host_row[1], x_dev.data_ptr(), value.data_ptr(),
                                               count, chunk, partial.data_ptr(), mom.data_ptr(), RT.stream_ptr()))
                # normal equations solved on the device, coefficients written straight into the row the next backward
                # step reads: no host synchronisation inside the induction (NCCL's all-gather is stream ordered)
                B.check(L.mcre_storage_solve(plan, RT.all_reduce_tree(mom).data_ptr(), 1e-12, dev_row.data_ptr(),
                                             RT.stream_ptr()))
        first = 0 if 0 in expo_of_k else 1
        for k in range(n_dates - 1, first - 1, -1):
            B.check(L.mcre_storage_backward(plan, k, coef[k].data_ptr(), spot[k].data_ptr(), value.data_ptr(), count,
                                            RT.stream_ptr()))
            value_h[0] = None
            if k >= 1:
                solve(spot_h[k - 1] if self.mode == "lapack" else None, spot[k - 1], numeraire[k - 1], coef_h[k - 1], coef[k - 1])
            for e in expo_of_k.get(k, []):
                solve(spot_eh[e] if self.mode == "lapack" else None, spot_e[e], expo_num[e], coef_eh[e], coef_e[e])
        if self.mode == "moments":
            coef_h = RT.to_host(coef)
            coef_eh = RT.to_host(coef_e) if n_expo else coef_eh
        # regression coefficients of the product, as the reference stores them ([date][state][basis]); in "moments"
        # mode they refer to the standardised spot (spot - centre) * inverse scale, kept next to them
        prod.regression_coeffs = torch.from_numpy(coef_h[:, 2:].reshape(n_dates, S, NB).copy())
        prod.regression_basis_shift_scale = torch.from_numpy(coef_h[:, :2].copy())
        if n_expo:
            c.regression_coeffs[prod.product_id] = torch.from_numpy(coef_eh[:, 2:].reshape(n_expo, S, NB).copy())
        return coef, coef_e

    # ------------------------------------------------------------------ run
    def run(self):
        c, L = self.c, B.lib()
        dev = RT.compute_device()
        t_start = time.perf_counter()
        grid = build_time_grid(self._t0(), c.simulation_timeline.tolist(), c.num_steps)
        step_cache = {}

        def steps_of(prod):
            key = None if (self.standalone and not _is_bsm(c.model)) else prod.get_asset_id()
            if key not in step_cache:
                nt = len(self.slots[prod.get_asset_id()][0]) if self.nt else 0
                step_cache[key] = step_table(c.model, grid, c.simulation_scheme, nt, asset_id=key, kernel_record=True)
            return step_cache[key]
        n_main = c.num_paths_mainsim
        if self.mixed or self.need_expo:
            from mcre.equity import main_chunk
            chunk = main_chunk(n_main)       # the equity launches' reduction chunk: one summation tree for the whole set
        else:
            chunk = 256 if n_main < (1 << 18) else 4096
        begin, count = RT.shard_range(n_main, chunk)
        rng_main, _keep = self._rng("main", 43, n_main)
        shard = B.Shard(begin, count, chunk)
        plans, t_pre = [], 0.0
        cfs = [torch.zeros(max(count, 1), dtype=torch.float64, device=dev) for _ in c.netting_sets]
        n_expo = len(c.exposure_timeline) if self.need_expo else 0
        expos = [torch.zeros((n_expo, max(count, 1)), dtype=torch.float64, device=dev) if n_expo else None
                 for _ in c.netting_sets]
        # per-path tangents, one buffer per (netting set, tangent slots): the storages of a set that share their slots add
        # into one buffer, whose fixed-order chunk sums are scattered into the set's gradient at the end
        tans = [{} for _ in c.netting_sets]
        try:
            for pi, prod in enumerate(c.products):
                if not _is_storage(prod):
                    continue
                plan, numeraire, acts, expo_num = self._create(prod, grid, *steps_of(prod))
                plans.append(plan)
                t0 = time.perf_counter()
                coef, coef_e = self._regress(prod, plan, numeraire, acts, expo_num, dev)
                torch.cuda.current_stream().synchronize()
                t_pre += time.perf_counter() - t0
                si = c.product_to_netting_set_idx[pi]
                tan = None
                if self.nt:
                    key = tuple(self.slots[prod.get_asset_id()][0])
                    if key not in tans[si]:
                        tans[si][key] = torch.zeros((len(key), max(count, 1)), dtype=torch.float64, device=dev)
                    tan = tans[si][key]
                B.check(L.mcre_storage_mainsim(plan, C.byref(rng_main), C.byref(shard), coef.data_ptr(),
                                               float(prod.get_initial_state()), cfs[si].data_ptr(), None,
                                               tan.data_ptr() if self.nt else None,
                                               coef_e.data_ptr() if n_expo else None,
                                               expos[si].data_ptr() if n_expo else None, RT.stream_ptr()))
            n_chunks = max((count + chunk - 1) // chunk, 1)
            partial = torch.empty(n_chunks * 2 * max(self.nt, 1) + 1, dtype=torch.float64, device=dev)
            grads = [self._gradient(t, count, chunk, partial, dev) for t in tans] if self.nt else None
            if self.mixed or self.need_expo:
                return self._finish_mixed(cfs, expos, grads, chunk, dev, t_start, t_pre)
            raw = []
            unconnected = c.model.unconnected_params(c.simulation_scheme)
            used = [i not in unconnected for i in range(len(c.model.model_params))]
            for si in range(len(c.netting_sets)):
                # shift = the set's value on global path 0 (lives on the rank that owns it; summed over the ranks)
                shift = cfs[si][0:1].clone() if (begin == 0 and count > 0) else torch.zeros(1, dtype=torch.float64, device=dev)
                shift = RT.all_reduce_tree(shift)
                out = torch.zeros(2, dtype=torch.float64, device=dev)
                B.check(L.mcre_sum_stats(cfs[si].data_ptr(), count, 1, chunk, shift.data_ptr(), 0, partial.data_ptr(),
                                         out.data_ptr(), RT.stream_ptr()))
                s = RT.to_host(RT.all_reduce_tree(out))
                pv = mean_and_error(float(s[0]), float(s[1]), float(RT.to_host(shift)[0]), n_main)
                raw.append({"pv": (pv, grads[si] if self.nt else None), "param_used": lambda kind: used})
        finally:
            torch.cuda.current_stream().synchronize()
            for plan in plans:
                L.mcre_storage_destroy(plan)
        total = time.perf_counter() - t_start
        return raw, {"preprocessing": t_pre, "path_generation": total - t_pre, "request_resolution": 0.0}


    def _gradient(self, tans, count, chunk, partial, dev):
        """PV gradient [n_params] of one netting set's storages: the sums of the per-path tangents of each buffer
        {slots: [len(slots)][count]} in the fixed chunk order of mcre_sum_stats (shift 0) and the rank tree - the same
        bits on any number of GPUs - over the path count, scattered to the slots' parameters."""
        L = B.lib()
        grad = np.zeros(len(self.c.model.model_params))
        for slots, tan in tans.items():
            nt = len(slots)
            zero = torch.zeros(nt, dtype=torch.float64, device=dev)
            out_t = torch.zeros(nt * 2, dtype=torch.float64, device=dev)
            B.check(L.mcre_sum_stats(tan.data_ptr(), count, nt, chunk, zero.data_ptr(), 0, partial.data_ptr(),
                                     out_t.data_ptr(), RT.stream_ptr()))
            grad[list(slots)] += RT.to_host(RT.all_reduce_tree(out_t)).reshape(nt, 2)[:, 0] / self.c.num_paths_mainsim
        return grad

    def _finish_mixed(self, cfs, expos, grads, chunk, dev, t_start, t_pre):
        """The other products of the run through the equity backend's accumulating launches, starting from the
        storages' per-path discounted cashflows and exposures (same Philox streams: the draw is the model's joint one);
        that path also applies threshold / collateral and finishes EPE / ENE / PFE - for books of storages alone, too.
        With sensitivities (PV only) the equity launches run with tangents, and a set's gradient is theirs plus the
        storages' `grads`."""
        import copy
        from mcre.equity import EquityBackend, is_equity_exercise
        c = self.c
        sub = copy.copy(c)
        sub.netting_sets = []
        for ns in c.netting_sets:
            view = copy.copy(ns)
            view.products = [p for p in ns.products if not _is_storage(p)]
            sub.netting_sets.append(view)
        sub.products = [p for ns in sub.netting_sets for p in ns.products]
        sub.product_to_netting_set_idx = [i for i, ns in enumerate(sub.netting_sets) for _ in ns.products]
        sub.requires_regression = any(sub._product_requires_regression(p) for p in sub.products)
        eb = EquityBackend(sub)
        t1 = time.perf_counter()
        eb.presim_exercise_all([p for p in sub.products if is_equity_exercise(p)], dev)
        if self.need_expo:
            reg = [p for p in sub.products if not sub._can_use_analytic_exposure_for_product(p) and not is_equity_exercise(p)]
            if reg:
                eb.presim_regression(reg, dev)
        torch.cuda.synchronize(dev)
        t_pre += time.perf_counter() - t1
        n_params = len(c.model.model_params)
        raw = []
        for si in range(len(c.netting_sets)):
            res = eb._run_split_book(si, dev, c.num_paths_mainsim, n_params, chunk=chunk, extra_pv=cfs[si],
                                     extra_expo=expos[si])
            if grads is not None:
                pv, grad = res["pv"]
                res["pv"] = (pv, grad + grads[si])
            raw.append(res)
        torch.cuda.synchronize(dev)
        total = time.perf_counter() - t_start
        return raw, {"preprocessing": t_pre, "path_generation": total - t_pre, "request_resolution": 0.0}


B_MAX_BASIS = 6
