"""Plan compiler + driver for the equity family (csrc/equity.cu).

Lowers (Black-Scholes single / multi asset / ModelConfig of equity models, Heston, Schwartz
two-factor; European / binary / basket / Asian / barrier payoffs; PV metrics) into the flat
tables of ``mcre_eq_desc`` (include/mcre.h) and runs the fused kernel: path stepping,
correlation, payoff, PV and pathwise sensitivities in one pass, nothing per-path in HBM.
What it takes the place of in the reference:
  request collection / resolution   src/request_interface/request_interface.py:22-130
  evaluate_products (PV branch)     src/controller/controller.py:385-471, 565-661
  torch.autograd.grad               src/controller/controller.py:609-627
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
from mcre.dual import D, cholesky_dual
from mcre.finish import mean_and_error
from mcre.timegrid import build_time_grid
from metrics.metric import MetricType
from models.black_scholes import BlackScholesModel
from models.black_scholes_multi import BlackScholesMulti
from models.cirpp import CIRPPModel
from models.heston import HestonModel
from models.model_config import ModelConfig
from models.schwartz_two_factor import SchwartzTwoFactorModel
from products.asian_option import AsianAveragingType, AsianOption
from products.barrier_option import BarrierOption, BarrierOptionType
from products.basket_option import BasketOption, BasketOptionType
from products.bermudan_option import BermudanOption
from products.binary_option import BinaryOption
from products.equity import Equity
from products.european_option import EuropeanOption
from products.flexicall import FlexiCall
from products.product import OptionType

CHUNK_PATHS = 4096


def main_chunk(n_total):
    """Paths per reduction chunk (= per block pass) of the main pass: a pure function of the TOTAL path count, so
    the summation tree - and every bit of the result - does not depend on the number of GPUs.  Small runs
    (books of many products on ~1000 paths) use small chunks, otherwise one block would do all the work."""
    if n_total >= (1 << 18):
        return CHUNK_PATHS
    return 256 if n_total >= (1 << 14) else 32
EQ_BS, EQ_HESTON, EQ_SCHWARTZ = 0, 1, 2
P_EUROPEAN, P_BINARY, P_BASKET, P_ASIAN, P_BARRIER, P_EXERCISE = 0, 1, 2, 3, 4, 5
EV_OBSERVE, EV_PAY, EV_FIRST, EV_EXERCISE = 1, 2, 4, 8
EQ_PR, EQ_PAR, EQ_MAX_SETS, EQ_XP, EQ_EVD, EQ_MAX_LAG, EQ_MAX_RIGHTS = 16, 8, 4, 32, 32, 4, 6


def eq_ntrk(nt):
    """Path-dependent / exercise trackers per launch (csrc/equity.cu:eq_ntrk)."""
    return 64 if nt == 0 else 2
_NPAR = {EQ_BS: 3, EQ_HESTON: 7, EQ_SCHWARTZ: 6}
_BARRIER_CODE = {BarrierOptionType.UPANDOUT: 1, BarrierOptionType.DOWNANDOUT: 2,
                 BarrierOptionType.UPANDIN: 3, BarrierOptionType.DOWNANDIN: 4}


class EqDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("scheme", C.c_int32), ("nt", C.c_int32), ("smoothing", C.c_int32),
        ("n_assets", C.c_int32), ("noise_dim", C.c_int32), ("n_uniform", C.c_int32),
        ("asset_par", B.c_dp), ("asset_noise", B.c_ip), ("asset_uniform", B.c_ip),
        ("col_asset", B.c_ip), ("col_elem", B.c_ip),
        ("n_sub", C.c_int32), ("n_dates", C.c_int32), ("n_pre_dates", C.c_int32), ("n_chol", C.c_int32),
        ("step_dt", B.c_dp), ("step_sq", B.c_dp), ("step_date", B.c_ip), ("step_chol", B.c_ip),
        ("step_aux", B.c_dp), ("init_aux", B.c_dp),
        ("corr_mode", C.c_int32), ("chol", B.c_dp), ("chol_dual", B.c_dp),
        ("date_ev_off", B.c_ip), ("ev_prod", B.c_ip), ("ev_flags", B.c_ip),
        ("n_prod", C.c_int32), ("prod", B.c_dp), ("prod_w", B.c_dp), ("n_sets", C.c_int32),
        ("ev_data", B.c_dp), ("prod_x", B.c_dp),
        ("n_expo", C.c_int32), ("n_metric", C.c_int32), ("acc_flags", C.c_int32),
        ("date_expo", B.c_ip), ("date_metric", B.c_ip), ("xp", B.c_dp),
        ("set_threshold", B.c_dp), ("set_flags", B.c_ip), ("set_lag", B.c_ip),
    ]


class EqCredit(C.Structure):
    """mcre_eq_credit (include/mcre.h)."""
    _fields_ = [("deterministic", C.c_int32), ("noise_col", C.c_int32),
                ("kappa", C.c_double), ("theta", C.c_double), ("sigma", C.c_double), ("y0", C.c_double), ("lgd", C.c_double),
                ("step_cir", B.c_dp), ("chol_row", B.c_dp), ("cva_coef", B.c_dp), ("set_cva", B.c_ip)]


def credit_of(model):
    """(CIR++ credit model, its index in the ModelConfig) of a hybrid equity + credit ModelConfig, else (None, None):
    the credit model rides after the market models (the joint Cholesky factor keeps the reference's asset order)."""
    if isinstance(model, ModelConfig) and len(model.models) >= 2 and isinstance(model.models[-1], CIRPPModel):
        return model.models[-1], len(model.models) - 1
    return None, None


class Asset:
    """One simulated asset = one lane of a path group."""

    def __init__(self, asset_id, model, par, gmap):
        self.asset_id, self.model = asset_id, model
        self.par = par        # lane parameter values in the kernel's order
        self.gmap = gmap      # lane parameter k -> index in the controller's flattened parameter list


def _sub_models(model):
    return list(model.models) if isinstance(model, ModelConfig) else [model]


def family_of(model):
    """(kind, assets) or None if the model is not an equity-family model."""
    subs = _sub_models(model)
    offs = model.param_offsets() if isinstance(model, ModelConfig) else [0]
    kinds, assets = set(), []
    credit, _ = credit_of(model)
    if credit is not None:
        subs = subs[:-1]
    for m, off in zip(subs, offs):
        pv = m.param_values()
        if isinstance(m, BlackScholesModel):
            kinds.add(EQ_BS)
            assets.append(Asset(m.asset_ids[0], m, pv, [off, off + 1, off + 2]))
        elif isinstance(m, BlackScholesMulti):
            kinds.add(EQ_BS)
            n = m.num_assets
            for a in range(n):
                assets.append(Asset(m.asset_ids[a], m, [pv[a], pv[n + a], pv[2 * n]],
                                    [off + a, off + n + a, off + 2 * n]))
        elif isinstance(m, HestonModel):
            kinds.add(EQ_HESTON)
            assets.append(Asset(m.asset_ids[0], m, pv, [off + k for k in range(7)]))
        elif isinstance(m, SchwartzTwoFactorModel):
            kinds.add(EQ_SCHWARTZ)
            assets.append(Asset(m.asset_ids[0], m, pv, [off + k for k in range(6)]))
        else:
            return None
    if len(kinds) != 1:
        return None
    kind = kinds.pop()
    if kind == EQ_SCHWARTZ and len(assets) != 1:
        return None
    if credit is not None and kind != EQ_BS:
        return None      # the credit factor rides with Black-Scholes market models
    return kind, assets


def is_equity_exercise(p):
    return isinstance(p, (BermudanOption, FlexiCall)) and isinstance(p.underlying, Equity)


def exercise_strikes(p):
    """Strike per exercise date: one strike (Bermudan / American) or the strip's strikes (FlexiCall)."""
    if isinstance(p, FlexiCall):
        return list(p.strikes)
    return [float(p.strike)] * len(p.product_timeline)


def _is_path_dependent(p):
    return isinstance(p, (AsianOption, BarrierOption)) or is_equity_exercise(p)


def _is_equity_product(p):
    if isinstance(p, EuropeanOption):
        return isinstance(p.underlying, Equity)
    if is_equity_exercise(p):
        return True
    return isinstance(p, (BinaryOption, BasketOption, AsianOption, BarrierOption))


class EquityBackend:
    @staticmethod
    def supports(ctrl):
        if family_of(ctrl.model) is None:
            return False
        if not all(_is_equity_product(p) for p in ctrl.products):
            return False
        if ctrl.risk_metrics.requires_exposure_profiles():
            # exposure profiles: the analytic Black-Scholes exposure of European options (the reference's
            # own no-regression branch, controller.py:204-229), else the regression proxy of products that
            # pay once; no CVA here (needs a credit model in the same ModelConfig: hybrid books are next)
            if any(m.metric_type == MetricType.CVA for m in ctrl.risk_metrics.metrics):
                # CVA of equity books: hybrid ModelConfig of Black-Scholes market models + the counterparty's CIR++
                credit, _ = credit_of(ctrl.model)
                return credit is not None and all(m.counterparty_id in credit.asset_ids for m in ctrl.risk_metrics.metrics
                                                  if m.metric_type == MetricType.CVA)
            return True
        return True

    def _param_used(self, kind):
        """Which model parameters a metric's value is connected to in the reference's autograd graph."""
        n = len(self.c.model.model_params)
        off = self.c.model.unconnected_params(self.c.simulation_scheme) if hasattr(self.c.model, "unconnected_params") else set()
        return [i not in off for i in range(n)]

    def __init__(self, ctrl):
        self.c = ctrl
        self.kind, self.assets = family_of(ctrl.model)
        self.A = len(self.assets)
        self.credit, self.credit_idx = credit_of(ctrl.model)
        if self.credit is not None:
            if ctrl.differentiate and not getattr(ctrl, "_credit_passenger", False):
                # (mcre/hybrid.py:EquityCreditGreeks runs the tangent pass with the credit factor as a value-only
                # passenger of the joint draw and differentiates the metrics on per-path duals)
                raise NotImplementedError("sensitivities of hybrid equity + credit runs are not implemented")
            if ctrl.simulation_scheme != SimulationScheme.EULER:
                # same restriction as the reference: only Black-Scholes pairs have a joint exact covariance (model_config.py:216-221)
                raise NotImplementedError("Analytical covariance is currently only supported for Black-Scholes-type model pairs.")
        if self.A > 32:
            raise NotImplementedError("at most 32 jointly simulated assets per path group")
        scheme = ctrl.simulation_scheme
        if self.kind == EQ_HESTON:
            if scheme not in (SimulationScheme.EULER, SimulationScheme.QE):
                raise NotImplementedError(f"Scheme {scheme} is not defined for the Heston model.")
            if isinstance(ctrl.model, ModelConfig) and scheme != SimulationScheme.QE:
                raise NotImplementedError("Several correlated Heston assets are simulated with the QE scheme only.")
        elif scheme not in (SimulationScheme.EULER, SimulationScheme.ANALYTICAL):
            raise NotImplementedError(f"Scheme {scheme} is not defined for this model.")
        self.scheme = scheme
        self.npar = _NPAR[self.kind]
        self.nt = self.npar if ctrl.differentiate else 0
        self.id_to_asset = {a.asset_id: i for i, a in enumerate(self.assets)}
        self.exercise_coef = {}        # id(product) -> (coef [n_ex, rights, 3] standardised basis, basis [n_ex, 2])
        self.exercise_expo_coef = {}   # id(product) -> (coef [n_expo, rights, 3], basis [n_expo, 2]) per exposure date
        self.exercise_expo_dcoef = {}  # id(product) -> d coef / d (lane parameters of the product's asset) [n_expo, rights, nt, 3]
        self.expo_coef = {}       # id(product) -> (coef [n_expo, 3] standardised basis, basis [n_expo, 2])
        self.expo_dcoef = {}      # id(product) -> d coef / d (lane parameters of the product's asset) [n_expo, nt, 3]
        subs = _sub_models(ctrl.model)
        num_idx = ctrl.model.id_to_model["numeraire"] if isinstance(ctrl.model, ModelConfig) else 0
        self.num_model = subs[num_idx]
        offs = ctrl.model.param_offsets() if isinstance(ctrl.model, ModelConfig) else [0]
        self.num_rate_global = offs[num_idx] + self._rate_index(self.num_model)
        self.num_rate = self.num_model.param_values()[self._rate_index(self.num_model)]
        #: pathwise Hessians (compute_higher_derivatives, controller.py:253-255, 631-648): Black-Scholes lanes carry
        #: Dual2<3> numbers - value, 3 first and 6 second derivatives w.r.t. (spot, volatility, rate) of the lane's asset
        self.second = bool(ctrl.differentiate and getattr(ctrl, "requires_higher_order_derivatives", False))
        if self.second:
            if (self.kind != EQ_BS or self.credit is not None or ctrl.risk_metrics.requires_exposure_profiles()
                    or any(a.gmap[2] != self.num_rate_global for a in self.assets)):
                raise NotImplementedError("second-order sensitivities of Monte Carlo values: present values of books on "
                                          "one Black-Scholes model (single or multi-asset)")
            for p in ctrl.products:
                if ctrl._can_skip_monte_carlo_for_product(p):
                    continue
                if (is_equity_exercise(p) or isinstance(p, BasketOption) or getattr(p, "basket", None) is not None
                        or getattr(p, "use_brownian_bridge", False)):
                    # (second derivatives across assets do not live in one lane; exercise products would need the
                    # second-order dependence of the regression coefficients)
                    raise NotImplementedError("second-order sensitivities of Monte Carlo values: single-asset products "
                                              "that pay once (European, binary, barrier, Asian options)")
            self.nt = 9
        if ctrl.differentiate and ctrl.risk_metrics.requires_exposure_profiles():
            # checked before any device work (the same conditions guard the lowering)
            if self.kind not in (EQ_BS, EQ_HESTON) or any(a.gmap[2] != self.num_rate_global for a in self.assets):
                raise NotImplementedError("sensitivities of exposure profiles of equity books: one Black-Scholes "
                                          "model (single or multi-asset) or one Heston model")
            if any(m.metric_type == MetricType.PFE for m in ctrl.risk_metrics.metrics) and not getattr(ctrl, "_credit_passenger", False):
                # (the fused kernel reduces tangent sums; the gradient of an order statistic is the tangent of ONE path:
                # mcre/hybrid.py:EquityCreditGreeks takes it from the per-path duals of the accumulating tangent pass)
                raise NotImplementedError("PFE sensitivities are not implemented for equity books")

    @staticmethod
    def _rate_index(m):
        if isinstance(m, BlackScholesMulti):
            return 2 * m.num_assets
        if isinstance(m, SchwartzTwoFactorModel):
            return 0
        return 2

    # ------------------------------------------------------------------ lowering
    def _asset_index(self, asset_id):
        if self.A == 1:
            return 0
        if asset_id not in self.id_to_asset:
            raise ValueError(f"Asset id '{asset_id}' not found in model asset ids {list(self.id_to_asset)}.")
        return self.id_to_asset[asset_id]

    def _inv_numeraire(self, t):
        """1 / N(t) and its rate derivative: deterministic money-market account of the
        numeraire model (black_scholes.py:104-106, heston.py:272-274)."""
        tau = t - self.num_model.t0()
        inv = math.exp(-self.num_rate * tau)
        return inv, -tau * inv

    def basis_at(self, a, t):
        """Standardisation (shift, scale) of the spot of asset a at time t from the model's own first two moments
        (log-normal with the model's average variance).  A pure conditioning aid: the fitted values do not depend
        on it, and - unlike sample statistics - it does not depend on how the paths are sharded over GPUs, so
        results stay bit-identical across GPU counts (SURVEY 8e)."""
        asset = self.assets[a]
        m, par = asset.model, asset.par
        tau = t - m.t0()
        if self.kind == EQ_BS:
            s0, sig, r = par
            mean, var_log = s0 * math.exp(r * max(tau, 0.0)), sig * sig * tau
        elif self.kind == EQ_HESTON:
            s0, _, r, _, kappa, theta, v0 = par
            kt = kappa * tau
            avg = theta + (v0 - theta) * ((1.0 - math.exp(-kt)) / kt if kt > 1e-12 else 1.0)
            mean, var_log = s0 * math.exp(r * max(tau, 0.0)), max(avg, 1e-12) * tau
        else:
            _, ks, ss, _, sl, rho = par
            mean = m.curve_value(t)
            e1 = (1.0 - math.exp(-ks * tau)) / ks if ks > 1e-12 else tau
            e2 = (1.0 - math.exp(-2.0 * ks * tau)) / (2.0 * ks) if ks > 1e-12 else tau
            var_log = ss * ss * e2 + sl * sl * tau + 2.0 * rho * ss * sl * e1
        if tau <= 0.0 or var_log <= 0.0:
            return (mean if tau > 0.0 else self._spot0(a), 1.0)
        std = mean * math.sqrt(math.expm1(min(var_log, 50.0)))
        return (mean, 1.0 / std if std > 0.0 else 1.0)

    def _spot0(self, a):
        asset = self.assets[a]
        if self.kind == EQ_SCHWARTZ:
            return asset.model.curve_value(asset.model.t0())
        return asset.par[0]

    def _product_record(self, p, set_local, slot, date_idx):
        """-> (record[16], weights[A], events [(date index, flags)])."""
        rec = np.zeros(EQ_PR)
        w = np.zeros(self.A)
        rec[1] = set_local
        rec[14] = -1
        sign = 1.0 if p.option_type == OptionType.CALL else -1.0
        rec[2], rec[3] = (0.0 if isinstance(p, FlexiCall) else float(p.strike)), sign
        basket = getattr(p, "basket", None)   # extension: path-dependent payoffs on a weighted basket
        if isinstance(p, EuropeanOption):
            rec[0] = P_EUROPEAN
            w[self._asset_index(p.underlying.get_asset_id())] = 1.0
            t_pay = float(p.exercise_date)
            events = [(date_idx[t_pay], EV_PAY)]
            t_num = t_pay
        elif isinstance(p, BinaryOption):
            rec[0] = P_BINARY
            w[self._asset_index(p.get_asset_id())] = 1.0
            rec[8] = float(p.payment_amount)
            t_pay = float(p.maturity)
            events = [(date_idx[t_pay], EV_PAY)]
            t_num = t_pay
        elif isinstance(p, BasketOption):
            rec[0] = P_BASKET
            for aid, wi in zip(p.asset_ids, p.weights.tolist()):
                w[self._asset_index(aid)] += wi
            geo = p.basket_option_type == BasketOptionType.GEOMETRIC
            rec[6] = (1 if geo else 0) | (2 if p.use_variation_reduction else 0)
            if p.use_variation_reduction:
                rec[7] = float(p.compute_pv_analytically(self.c.model).reshape(-1)[0])
            t_pay = float(p.maturity)
            events = [(date_idx[t_pay], EV_PAY)]
            t_num = t_pay
        elif isinstance(p, (AsianOption, BarrierOption)):
            obs = p.modeling_timeline.tolist()        # (iterating a tensor element by element costs microseconds each)
            if basket is not None:
                for aid, wi in zip(*basket):
                    w[self._asset_index(aid)] += float(wi)
            else:
                w[self._asset_index(p.get_asset_id())] = 1.0
            rec[13], rec[14] = len(obs), slot
            if isinstance(p, AsianOption):
                rec[0] = P_ASIAN
                rec[6] = 1 if p.averaging_type == AsianAveragingType.GEOMETRIC else 0
            else:
                rec[0] = P_BARRIER
                if getattr(p, "use_brownian_bridge", False):
                    if basket is not None or not isinstance(self.c.model, BlackScholesModel):
                        raise NotImplementedError("Brownian-bridge barrier monitoring: single Black-Scholes model, "
                                                  "one monitored asset")
                    rec[6] = 4
                rec[9], rec[10] = float(p.barrier1), _BARRIER_CODE[p.barrier_option_type1]
                if p.barrier2 is not None and p.barrier_option_type2 is not None:
                    rec[11], rec[12] = float(p.barrier2), _BARRIER_CODE[p.barrier_option_type2]
            events = []
            for i, t in enumerate(obs):
                f = EV_OBSERVE | (EV_FIRST if i == 0 else 0) | (EV_PAY if i == len(obs) - 1 else 0)
                events.append((date_idx[t], f))
            # the reference divides by the numeraire request of index 0 = the FIRST monitoring
            # date (asian_option.py:90, barrier_option.py:312)
            t_num = obs[0]
        elif is_equity_exercise(p):
            rec[0] = P_EXERCISE
            rec[13], rec[14] = p.num_exercise_rights, slot
            if p.num_exercise_rights > EQ_MAX_RIGHTS:
                raise NotImplementedError(f"at most {EQ_MAX_RIGHTS} exercise rights per product")
            w[self._asset_index(p.underlying.get_asset_id())] = 1.0
            ex = p.product_timeline.tolist()
            events = [(date_idx[t], EV_EXERCISE | (EV_FIRST if i == 0 else 0)) for i, t in enumerate(ex)]
            t_num = ex[0]
        else:
            raise TypeError(type(p))
        rec[4], rec[5] = self._inv_numeraire(t_num)
        return rec, w, events

    def _correlation_tables(self, grid, nt):
        """-> (corr_mode, chol [n_chol,d,d] or None, chol_dual list of D or None, step_chol)."""
        model, scheme = self.c.model, self.scheme
        n_sub = grid.n_sub
        zero_idx = [0] * n_sub
        if self.kind == EQ_BS:
            if self.A == 1 and self.credit is None:
                return 0, None, None, zero_idx
            # ANALYTICAL: chol(diag(s) C diag(s) dt) = diag(s sqrt(dt)) chol(C): one factor for all steps
            if isinstance(model, ModelConfig):
                ps = [m.dual_params() for m in model.models]
                corr = [[x.v for x in row] for row in model.joint_correlation(SimulationScheme.EULER, ps)]
            else:
                corr = model.correlation_matrix.numpy().tolist()
            Lm = cholesky_dual([[D(x, None, 0) for x in row] for row in corr])
            return 2, np.array([[[x.v for x in row] for row in Lm]]), None, zero_idx
        if self.kind == EQ_HESTON:
            if self.A == 1:
                if scheme == SimulationScheme.QE:
                    return 0, None, None, zero_idx
                p = self.assets[0].model.dual_params(0, nt)
                L = cholesky_dual(self.assets[0].model.intra_correlation(scheme, p))
                return 1, None, [L[0][0], L[0][1], L[1][0], L[1][1]], zero_idx
            # extension: spot normals of the assets correlated by the ModelConfig's inter-asset
            # matrix, variance normals independent (QE draws them independently, heston.py:85-90)
            A = self.A
            corr = np.eye(2 * A)
            idx = 0
            for i in range(A):
                for j in range(i + 1, A):
                    rho = float(np.asarray(model.inter_asset_correlation_matrix[idx]).reshape(-1)[0])
                    corr[2 * i, 2 * j] = corr[2 * j, 2 * i] = rho
                    idx += 1
            return 2, np.linalg.cholesky(corr)[None], None, zero_idx
        # Schwartz two-factor
        m = self.assets[0].model
        p = m.dual_params(0, nt)
        if scheme == SimulationScheme.EULER:
            L = cholesky_dual(m.intra_correlation(scheme, p))
            return 1, None, [L[0][0], L[0][1], L[1][0], L[1][1]], zero_idx
        chol_dual, step_chol, seen = [], [], {}
        for s in range(n_sub):
            key = grid.dt_nominal[s]
            if key not in seen:
                L = cholesky_dual(m.exact_covariance(p, key))
                seen[key] = len(chol_dual) // 4
                chol_dual += [L[0][0], L[0][1], L[1][0], L[1][1]]
            step_chol.append(seen[key])
        return 1, None, chol_dual, step_chol

    def lower(self, set_indices, presim_products=None, subset=None, presim_tangents=False, spill_times=None):
        """Plan of the main pass for a group of netting sets, or (presim_products given) of the
        pre-simulation spill pass for a group of products (all in one dummy set).  `subset`: the
        products to keep (book splitting: one launch evaluates a part of a large netting set).
        `spill_times` (spill pass): the dates to spill spots at instead of the exposure dates."""
        c, nt, A = self.c, self.nt, self.A
        if presim_products is not None and not presim_tangents:
            nt = 0
        grid = build_time_grid(self.assets[0].model.t0(), c.simulation_timeline.tolist(), c.num_steps)
        dates = grid.dates
        date_idx = grid.index_map()
        n_dates, n_sub = len(dates), grid.n_sub
        two = self.kind != EQ_BS
        d = (2 if two else 1) * A + (1 if self.credit is not None else 0)     # the credit factor draws the last column
        asset_noise = np.array([[2 * a, 2 * a + 1] if two else [a, -1] for a in range(A)], dtype=np.int32)
        col_asset = np.array([min(j // 2 if two else j, A - 1) for j in range(d)], dtype=np.int32)
        col_elem = np.array([j % 2 if two else 0 for j in range(d)], dtype=np.int32)
        par = np.zeros((A, EQ_PAR))
        for a, asset in enumerate(self.assets):
            par[a, :self.npar] = asset.par
        corr_mode, chol, chol_dual, step_chol = self._correlation_tables(grid, nt)
        analytical = self.scheme == SimulationScheme.ANALYTICAL
        step_sq = [math.sqrt(x) for x in (grid.dt_nominal if analytical else grid.dt)]
        step_aux = np.zeros((max(n_sub, 1), A))
        init_aux = np.zeros(A)
        if self.kind == EQ_SCHWARTZ:
            m = self.assets[0].model
            init_aux[0] = math.log(m.curve_value(m.t0()))
            for s in range(n_sub):
                step_aux[s, 0] = math.log(m.curve_value(grid.t2[s]))

        # ---- products / events ------------------------------------------------------------
        recs, weights, xweights, events = [], [], [], [[] for _ in range(n_dates)]
        owners = []
        slot = 0
        if presim_products is not None:
            book = [(0, p) for p in presim_products]
        elif subset is not None:
            book = [(0, p) for p in subset]      # book splitting: one netting set, products in netting-set order
        else:
            book = [(r, p) for r, si in enumerate(set_indices) for p in c.netting_sets[si].products]
        for r, p in book:
            if True:
                if c._can_skip_monte_carlo_for_product(p):
                    continue
                use_slot = -1
                if _is_path_dependent(p):
                    use_slot = slot
                    slot += 1
                rec, w, evs = self._product_record(p, r, use_slot, date_idx)
                pi = len(recs)
                recs.append(rec)
                weights.append(w)
                xw = np.zeros(A)
                aid = p.asset_ids[0] if getattr(p, "asset_ids", None) else None
                if self.A == 1 or aid in self.id_to_asset:
                    xw[self._asset_index(aid)] = 1.0   # explanatory variable: spot of the product's first asset
                xweights.append(xw)
                owners.append(p)
                for di, f in evs:
                    events[di].append((pi, f))
        if slot > eq_ntrk(nt):
            raise NotImplementedError(f"at most {eq_ntrk(nt)} path-dependent / exercise products per launch group")
        ev_off, ev_prod, ev_flags, ev_data = [0], [], [], []
        ex_count = {}
        bridge = []   # (tracker slot, product id, intervals) of Brownian-bridge barrier options
        for di in range(n_dates):
            for pi, f in events[di]:
                ev_prod.append(pi)
                ev_flags.append(f)
                row = np.zeros(EQ_EVD)
                if f & EV_EXERCISE:
                    p = owners[pi]
                    i = ex_count.get(pi, 0)
                    ex_count[pi] = i + 1
                    coef, basis = self.exercise_coef[id(p)]          # [n_ex, rights, 3], [n_ex, 2]
                    row[0:3], row[3:5] = coef[i, 0], basis[i]
                    for st in range(1, coef.shape[1]):
                        row[16 + 3 * (st - 1):19 + 3 * (st - 1)] = coef[i, st]
                    row[5], row[6] = self._inv_numeraire(dates[di])
                    row[7] = 1.0 if i == len(p.product_timeline) - 1 else 0.0
                    row[14] = exercise_strikes(p)[i]
                elif (f & EV_OBSERVE) and getattr(owners[pi], "use_brownian_bridge", False):
                    # Brownian-bridge draws of the interval ending at this observation (csrc/equity.cu)
                    p = owners[pi]
                    i = ex_count.get(pi, 0)
                    ex_count[pi] = i + 1
                    n_obs = len(p.modeling_timeline)
                    sigma = self.assets[self._asset_index(p.get_asset_id())].par[1]
                    row[0] = float(p.product_id * 4096 + max(i - 1, 0))
                    row[1] = -2.0 / (sigma * sigma * float(p.maturity) / n_obs)
                    row[2] = float(max(i - 1, 0))
                    if i == 0:
                        bridge.append((int(recs[pi][14]), int(p.product_id), n_obs - 1))
                ev_data.append(row)
            ev_off.append(len(ev_prod))

        t = {}

        def fp(name, arr):
            t[name], ptr = B.as_dp(arr)
            return ptr

        def ip(name, arr):
            t[name], ptr = B.as_ip(arr)
            return ptr

        desc = EqDesc()
        desc.kind = self.kind
        desc.scheme = {SimulationScheme.EULER: B.SCHEME_EULER, SimulationScheme.ANALYTICAL: B.SCHEME_ANALYTICAL,
                       SimulationScheme.QE: B.SCHEME_QE}[self.scheme]
        desc.nt = nt
        desc.smoothing = int(any(a.model.perform_smoothing for a in self.assets))
        desc.n_assets, desc.noise_dim = A, d
        desc.n_uniform = A if (self.kind == EQ_HESTON and self.scheme == SimulationScheme.QE) else 1
        desc.asset_par = fp("par", par)
        desc.asset_noise, desc.asset_uniform = ip("noise", asset_noise), ip("uni", np.arange(A))
        desc.col_asset, desc.col_elem = ip("col_asset", col_asset), ip("col_elem", col_elem)
        desc.n_sub, desc.n_dates, desc.n_pre_dates = n_sub, n_dates, grid.n_pre_dates
        desc.n_chol = (len(chol_dual) // 4) if chol_dual else (len(chol) if chol is not None else 0)
        desc.step_dt = fp("dt", grid.dt if n_sub else [0.0])
        desc.step_sq = fp("sq", step_sq if n_sub else [0.0])
        desc.step_date = ip("step_date", grid.date_after if n_sub else [0])
        desc.step_chol = ip("step_chol", step_chol if n_sub else [0])
        desc.step_aux, desc.init_aux = fp("step_aux", step_aux), fp("init_aux", init_aux)
        desc.corr_mode = corr_mode
        desc.chol = fp("chol", chol if chol is not None else np.zeros(1))
        desc.chol_dual = fp("chol_dual", np.concatenate([x.pack() for x in chol_dual]) if chol_dual else np.zeros(1))
        desc.date_ev_off = ip("ev_off", ev_off)
        desc.ev_prod, desc.ev_flags = ip("ev_prod", ev_prod or [0]), ip("ev_flags", ev_flags or [0])
        desc.n_prod = len(recs)
        desc.prod = fp("prod", np.stack(recs) if recs else np.zeros(EQ_PR))
        desc.prod_w = fp("prod_w", np.stack(weights) if weights else np.zeros(A))
        desc.n_sets = len(set_indices) if presim_products is None else 1
        desc.ev_data = fp("ev_data", np.stack(ev_data) if ev_data else np.zeros(EQ_EVD))
        desc.prod_x = fp("prod_x", np.stack(xweights) if xweights else np.zeros(A))

        # ---- exposure profiles ---------------------------------------------------------------
        n_expo = n_metric = acc = 0
        if c.risk_metrics.requires_exposure_profiles():
            if nt and presim_products is None:
                # sensitivities of EPE / ENE / CE through the analytic Black-Scholes exposure: tangents in the fused kernel
                # (csrc/equity.cu, exposure tangents).  The numeraire term lands on the lane-local rate, so every asset
                # must share the numeraire's rate parameter (BlackScholesModel, BlackScholesMulti).
                if self.kind not in (EQ_BS, EQ_HESTON) or any(a.gmap[2] != self.num_rate_global for a in self.assets):
                    raise NotImplementedError("sensitivities of exposure profiles of equity books: one Black-Scholes "
                                              "model (single or multi-asset) or one Heston model")
                for p in owners:
                    if c._can_use_analytic_exposure_for_product(p) or is_equity_exercise(p):
                        continue      # (exercise products: tangent backward induction, exercise_expo_dcoef)
                    if id(p) not in self.expo_dcoef:
                        raise NotImplementedError("sensitivities of exposure profiles of equity books: not implemented for "
                                                  "baskets (regression proxies on several assets)")
                if any(m.metric_type == MetricType.PFE for m in c.risk_metrics.metrics) and not getattr(c, "_credit_passenger", False):
                    raise NotImplementedError("PFE sensitivities are not implemented for equity books")
            expo_times, metric_times = c.exposure_timeline.tolist(), c.metric_exposure_timeline.tolist()
            if spill_times is not None:
                expo_times = list(spill_times)
            n_expo, n_metric = len(expo_times), len(metric_times)
            date_expo = np.full(n_dates, -1, dtype=np.int32)
            date_metric = np.full(n_dates, -1, dtype=np.int32)
            for e, te in enumerate(expo_times):
                date_expo[date_idx[te]] = e
            for m, tm in enumerate(metric_times):
                date_metric[date_idx[tm]] = m
            xp = np.zeros((n_expo, max(len(recs), 1), EQ_XP))
            xp_tan = np.zeros((n_expo, max(len(recs), 1), 3, max(nt, 1))) if (nt and presim_products is None) else None
            xp_ex_tan = None      # [n_expo][n_prod][EQ_MAX_RIGHTS][3][nt], exercise products only
            # per product, all exposure dates at once (books of thousands of products x ~100 dates: no Python in the
            # (date, product) loop)
            te_arr = np.asarray(expo_times, dtype=np.float64)
            invs = np.array([self._inv_numeraire(te) for te in expo_times]).reshape(n_expo, 2)
            inv, dinv = invs[:, 0], invs[:, 1]
            for pi, p in enumerate(owners):
                if presim_products is not None:
                    break                           # the spill pass evaluates no exposures
                if c._can_use_analytic_exposure_for_product(p):
                    ttm = float(p.exercise_date) - te_arr
                    on = ttm > 0.0                  # matured options carry no exposure (european_option.py:129-131)
                    xp[on, pi, 0], xp[on, pi, 1], xp[on, pi, 2] = 1.0, ttm[on], inv[on]
                    xp[on, pi, 7] = dinv[on]        # d (1 / N(t)) / d rate, for the exposure tangents
                elif is_equity_exercise(p):
                    coef, basis = self.exercise_expo_coef[id(p)]     # [n_expo, rights, 3], [n_expo, 2]
                    on = np.any(coef != 0.0, axis=(1, 2))
                    xp[on, pi, 0], xp[on, pi, 1], xp[on, pi, 2] = 3.0, coef[on, 0, 0], inv[on]
                    xp[on, pi, 3], xp[on, pi, 4] = coef[on, 0, 1], coef[on, 0, 2]
                    xp[on, pi, 5], xp[on, pi, 6] = basis[on, 0], basis[on, 1]
                    for st in range(1, coef.shape[1]):
                        xp[on, pi, 16 + 3 * (st - 1):19 + 3 * (st - 1)] = coef[on, st]
                    xp[on, pi, 7] = dinv[on]
                    if xp_tan is not None:
                        if xp_ex_tan is None:
                            xp_ex_tan = np.zeros((n_expo, len(recs), EQ_MAX_RIGHTS, 3, nt))
                        dcoef = self.exercise_expo_dcoef[id(p)]                  # [n_expo, rights, nt, 3]
                        xp_ex_tan[on, pi, :coef.shape[1]] = np.transpose(dcoef[on], (0, 1, 3, 2))
                else:
                    coef, basis = self.expo_coef[id(p)]              # [n_expo, 3], [n_expo, 2]
                    on = np.any(coef != 0.0, axis=1)
                    xp[on, pi, 0], xp[on, pi, 1], xp[on, pi, 2] = 2.0, coef[on, 0], inv[on]
                    xp[on, pi, 3], xp[on, pi, 4] = coef[on, 1], coef[on, 2]
                    xp[on, pi, 5], xp[on, pi, 6], xp[on, pi, 7] = basis[on, 0], basis[on, 1], dinv[on]
                    if xp_tan is not None:
                        xp_tan[on, pi] = np.transpose(self.expo_dcoef[id(p)][on], (0, 2, 1))   # [nt, 3] -> [3, nt]
            kinds = {m.metric_type for m in c.risk_metrics.metrics}
            if kinds & {MetricType.CE, MetricType.EPE, MetricType.EEPE}:
                acc |= B.ACC_POS
            if MetricType.ENE in kinds:
                acc |= B.ACC_NEG
            if MetricType.PFE in kinds:
                acc |= B.ACC_SPILL
            sets = [c.netting_sets[i] for i in set_indices] if presim_products is None else [c.netting_sets[0]]
            if presim_products is not None:
                set_indices, acc = [0], 0
            set_flags = np.zeros(len(sets), dtype=np.int32)
            set_lag = np.full((len(sets), n_metric), -1, dtype=np.int32)
            for r, (si, ns) in enumerate(zip(set_indices, sets)):
                if ns.is_collateralized() and presim_products is None:
                    set_flags[r] |= 1
                    delayed = c.netting_set_delayed_exposure_indices[si].tolist()
                    for m in range(n_metric):
                        if delayed[m] >= 0:
                            lag = int(c.metric_exposure_indices[m]) - delayed[m]
                            if lag >= EQ_MAX_LAG:
                                raise NotImplementedError(
                                    f"MPoR look-back spans {lag} exposure dates; the fused kernel keeps {EQ_MAX_LAG - 1}")
                            set_lag[r, m] = lag
            desc.date_expo, desc.date_metric = ip("date_expo", date_expo), ip("date_metric", date_metric)
            desc.xp = fp("xp", xp)
            desc.set_threshold = fp("set_thr", np.array([ns.threshold for ns in sets], dtype=np.float64))
            desc.set_flags, desc.set_lag = ip("set_flags", set_flags), ip("set_lag", set_lag)
        desc.n_expo, desc.n_metric, desc.acc_flags = n_expo, n_metric, acc
        info = dict(grid=grid, noise_dim=d, n_uniform=desc.n_uniform, owners=owners, recs=recs, n_metric=n_metric, acc=acc,
                    bridge=bridge, chol=chol, set_indices=list(set_indices), xp_tan=xp_tan if (n_expo and presim_products is None) else None,
                    xp_ex_tan=xp_ex_tan if (n_expo and presim_products is None) else None)
        return desc, t, info

    def _set_credit(self, plan, info):
        """Hands the plan the CIR++ credit factor of a hybrid ModelConfig and the CVA weights (mcre_eq_set_credit);
        returns the CVA metric or None.  Closed forms from models/cirpp.py (psi, conditional survival coefficients)."""
        c, cir = self.c, self.credit
        cvas = [m for m in c.risk_metrics.metrics if m.metric_type == MetricType.CVA]
        if cir is None or not cvas or not info["n_metric"]:
            return None
        if len({m.counterparty_id for m in cvas}) > 1 or len({m.recovery_rate for m in cvas}) > 1:
            raise NotImplementedError("one CVA counterparty / recovery per run is supported for now")
        metric = cvas[0]
        grid, d = info["grid"], info["noise_dim"]
        pv = cir.param_values()                   # [kappa, theta, sigma, y0]
        metric_times = c.metric_exposure_timeline.tolist()
        n_metric = len(metric_times)
        t0 = cir.t0()
        step = np.zeros((max(grid.n_sub, 1), 2))
        coef = np.zeros((n_metric, 2))
        if cir.deterministic:
            for s_ in range(grid.n_sub):
                step[s_] = (cir.market_hazard(grid.t1[s_]), cir.market_hazard(grid.t2[s_]))
            for m in range(n_metric - 1):
                coef[m] = (cir.market_survival(metric_times[m + 1]) / cir.market_survival(metric_times[m]), 0.0)
            y0 = cir.market_hazard(t0)
        else:
            if grid.n_sub:
                step[:grid.n_sub, 0] = cir.psi_values(pv, grid.t1)
            if n_metric > 1:
                Cs, Bs = cir.conditional_survival_values(pv, metric_times[:-1], metric_times[1:])
                coef[:-1, 0], coef[:-1, 1] = Cs, Bs
            y0 = pv[3]
        cr = EqCredit()
        cr.deterministic, cr.noise_col = int(cir.deterministic), d - 1
        cr.kappa, cr.theta, cr.sigma, cr.y0, cr.lgd = pv[0], pv[1], pv[2], y0, 1.0 - metric.recovery_rate
        keep = {}
        keep["step"], cr.step_cir = B.as_dp(step.reshape(-1))
        keep["row"], cr.chol_row = B.as_dp(np.asarray(info["chol"])[0, d - 1, :])
        keep["coef"], cr.cva_coef = B.as_dp(coef.reshape(-1))
        flags = [int(c.netting_sets[si].counterparty_id is None or c.netting_sets[si].counterparty_id == metric.counterparty_id)
                 for si in info["set_indices"]]
        keep["flags"], cr.set_cva = B.as_ip(flags)
        B.check(B.lib().mcre_eq_set_credit(plan, C.byref(cr)))
        return metric

    def _credit_weight_tangents(self, plan, info, rng, sh, n, dev):
        """d (per-path default weights) / d (kappa, theta, sigma, y0) of a stochastic CIR++ counterparty,
        [n_metric][4][n] (mcre_eq_credit_weight_tangents): the closed forms psi(t) and (C_k, B_k) as host duals
        (models/cirpp.py), the factor's Euler recursion differentiated in the kernel."""
        c, cir = self.c, self.credit
        grid, d = info["grid"], info["noise_dim"]
        pv = cir.param_values()
        pc = cir.dual_params(0, 4)
        metric_times = c.metric_exposure_timeline.tolist()
        n_metric = len(metric_times)
        step = np.zeros((max(grid.n_sub, 1), 2))
        dpsi = np.zeros((max(grid.n_sub, 1), 4))
        for s_ in range(grid.n_sub):
            ps = cir.psi(pc, grid.t1[s_])
            step[s_, 0], dpsi[s_] = ps.v, ps.t
        coef, dcoef = np.zeros((n_metric, 2)), np.zeros((n_metric, 2, 4))
        for m in range(n_metric - 1):
            Ck, Bk = cir.conditional_survival_coefficients(pc, metric_times[m], metric_times[m + 1])
            coef[m] = (Ck.v, Bk.v)
            dcoef[m, 0], dcoef[m, 1] = Ck.t, Bk.t
        cr = EqCredit()
        cr.deterministic, cr.noise_col = 0, d - 1
        cr.kappa, cr.theta, cr.sigma, cr.y0, cr.lgd = pv[0], pv[1], pv[2], pv[3], 1.0
        keep = {}
        keep["step"], cr.step_cir = B.as_dp(step.reshape(-1))
        keep["row"], cr.chol_row = B.as_dp(np.asarray(info["chol"])[0, d - 1, :])
        keep["coef"], cr.cva_coef = B.as_dp(coef.reshape(-1))
        keep["dpsi"], dpsi_p = B.as_dp(dpsi.reshape(-1))
        keep["dcoef"], dcoef_p = B.as_dp(dcoef.reshape(-1))
        w_tan = torch.zeros((n_metric, 4, n), dtype=torch.float64, device=dev)
        B.check(B.lib().mcre_eq_credit_weight_tangents(plan, C.byref(cr), dpsi_p, dcoef_p, C.byref(rng), C.byref(sh),
                                                       w_tan.data_ptr(), RT.stream_ptr()))
        return w_tan

    # ------------------------------------------------------------------ execution
    def _rng(self, seed, n_total):
        c = self.c
        r = B.Rng()
        r.seed, r.stream, r.n_paths_total = seed, c.rng_stream, n_total
        z = c.injected_normals.get("main") if c.injected_normals else None
        if z is not None:
            r.mode, r.d_z = B.RNG_INJECT, z.data_ptr()
            u = getattr(c, "injected_uniforms", None)
            u = u.get("main") if u else None
            if u is not None:
                dev = RT.compute_device()
                u = torch.as_tensor(u, dtype=torch.float64).to(dev).contiguous()
                self._keep_u = u
                r.d_u = u.data_ptr()
        else:
            r.mode = B.RNG_PHILOX
        return r

    def _control_variate_gradient(self, owners, recs, set_local, n_params):
        """d/d(params) of the closed-form control-variate constants (basket_option.py:72-78):
        they enter every path's payoff, so their parameter derivative adds invN * dc."""
        out = np.zeros(n_params)
        for p, rec in zip(owners, recs):
            if int(rec[1]) != set_local or not (isinstance(p, BasketOption) and p.use_variation_reduction):
                continue
            params = self.c.model.model_params
            leaves = [q.detach().clone().requires_grad_(True) for q in params]
            saved = list(params)
            try:
                self._swap_params(leaves)
                val = p.compute_pv_analytically(self.c.model).reshape(-1)[0]
                grads = torch.autograd.grad(val, leaves, allow_unused=True)
            finally:
                self._swap_params(saved)
            for i, g in enumerate(grads):
                if g is not None:
                    out[i] += rec[4] * float(g)
        return out

    def _swap_params(self, new):
        model = self.c.model
        if isinstance(model, ModelConfig):
            o = 0
            for m in model.models:
                k = len(m.model_params)
                m.model_params = list(new[o:o + k])
                o += k
            model.model_params = [q for m in model.models for q in m.model_params]
        else:
            model.model_params = list(new)

    def _state_columns(self):
        """(state column, is log-spot) of every asset in the joint state vector of the path generator."""
        cols, off = [], 0
        for m in _sub_models(self.c.model):
            if isinstance(m, BlackScholesModel):
                cols.append((off, 0))
            elif isinstance(m, BlackScholesMulti):
                cols += [(off + a, 0) for a in range(m.num_assets)]
            else:                       # Heston [logS, v], Schwartz [logS, x, y]
                cols.append((off, 1))
            off += m.state_dim
        return cols

    def presim_exercise_all(self, prods, dev):
        """Longstaff-Schwartz pre-simulation of every exercise product of the run: the backward inductions of
        the products advance in lock-step (one moment all-reduce + one device-to-host read per step for all
        of them, mcre/lsm.py:run_backward_inductions) instead of one synchronisation per product and date.
        Memory is bounded by processing the products in batches."""
        from mcre.lsm import run_backward_inductions
        if not prods:
            return
        c = self.c
        n_expo = len(c.exposure_timeline) if c.risk_metrics.requires_exposure_profiles() else 0
        nt = self.nt if n_expo else 0       # tangents of the induction: sensitivities of exposure metrics only
        _, count = RT.shard_range(c.num_paths_presim, CHUNK_PATHS)
        # value arrays (xs, nums, imm) + f32 values; with tangents dxs, dnums, dimm, the running tangents and the
        # product's share of the tangent spill of every asset
        per_product = max(((3 + nt * (3 + self.A)) * (len(p.product_timeline) + n_expo) + 2 + 2 * nt * p.num_exercise_rights)
                          * max(count, 1) * 8 for p in prods)
        batch = max(1, min(64, int(6e9 // per_product)))
        expo_times = c.exposure_timeline.tolist() if n_expo else []
        for b0 in range(0, len(prods), batch):
            group = prods[b0:b0 + batch]
            spill = None
            if nt:
                times = {t for p in group for t in p.regression_timeline.tolist() + p.product_timeline.tolist()}
                spill = self.presim_tangent_spill(times | set(expo_times), dev)
            prepared = [self.presim_exercise(p, dev, prepare_only=True, spill=spill) for p in group]
            coefs = run_backward_inductions([g for g, _ in prepared])
            for (_, finish), coef in zip(prepared, coefs):
                finish(coef)
            del spill, prepared
        self._presim_paths = None

    def presim_exercise(self, prod, dev, prepare_only=False, spill=None):
        """Longstaff-Schwartz pre-simulation of a Bermudan / American / FlexiCall option on equity underlyings
        (controller.py:294-383): pre-simulation paths from the path generator (seed 42), gathered
        date-major by mcre_lsm_prepare_equity, then the shared backward induction (mcre/lsm.py).
        With tangents and exposure metrics the induction also differentiates the exposure coefficients: the tangents
        of the gathered arrays come from the tangent spill of the pre-simulation (`spill` = presim_tangent_spill of
        dates covering the product's regression dates, else one of its own) through mcre_lsm_prepare_equity_tangents;
        the value arrays, and so every exercise decision and coefficient, are those of the value-only run.
        prepare_only: return (generator of the backward induction, finish(coef)) for the lock-step driver."""
        from mcre import paths as P
        from mcre.lsm import backward_induction_steps, run_backward_inductions, to_raw_basis
        c = self.c
        L = B.lib()
        n_pre = c.num_paths_presim
        if n_pre <= 0:
            raise ValueError("Exercise products need a pre-simulation: num_paths_presim must be positive.")
        ptl = prod.product_timeline.tolist()
        expo_times = c.exposure_timeline.tolist() if c.risk_metrics.requires_exposure_profiles() else []
        reg_times = sorted(set(prod.regression_timeline.tolist()) | set(expo_times))
        R = int(prod.num_exercise_rights)
        sim = c.simulation_timeline.tolist()
        date_idx = {t: i for i, t in enumerate(sim)}
        begin, count = RT.shard_range(n_pre, CHUNK_PATHS)
        n = max(count, 1)
        inj = c.injected_normals.get("pre") if c.injected_normals else None
        inj_u = getattr(c, "injected_uniforms", None)
        inj_u = inj_u.get("pre") if inj_u else None
        paths = getattr(self, "_presim_paths", None)
        if paths is None:
            # one set of pre-simulation paths serves every exercise product of the run (the reference
            # generates them once per run too, controller.py:272-292)
            paths = P.generate(c.model, sim, n, c.num_steps, self.scheme, 42, inject_z=inj, inject_u=inj_u,
                               stream_id=c.rng_stream, path_begin=begin, n_total=n_pre)
            self._presim_paths = paths
        cols = self._state_columns()
        xi = self._asset_index(prod.get_asset_id())
        ui = self._asset_index(prod.underlying.get_asset_id())
        t0 = self.num_model.t0()
        n_reg, n_ex = len(reg_times), len(ptl)
        buf = torch.empty((2 * n_reg + n_ex) * n, dtype=torch.float64, device=dev)
        xs, nums, imm = buf[:n_reg * n].view(n_reg, n), buf[n_reg * n:2 * n_reg * n].view(n_reg, n), buf[2 * n_reg * n:].view(n_ex, n)
        keep = []

        def ip(a):
            arr, ptr = B.as_ip(a)
            keep.append(arr)
            return ptr

        def fp(a):
            arr, ptr = B.as_dp(a)
            keep.append(arr)
            return ptr

        L.mcre_lsm_prepare_equity.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, B.c_ip, B.c_dp, C.c_int32,
                                              B.c_ip, C.c_int32, C.c_int32, C.c_int32, B.c_ip, B.c_dp, B.c_ip, C.c_double,
                                              B.c_dp, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        sign = 1.0 if prod.option_type == OptionType.CALL else -1.0
        B.check(L.mcre_lsm_prepare_equity(
            paths.data_ptr(), count, len(sim), paths.shape[2], n_reg, ip([date_idx[t] for t in reg_times]),
            fp([math.exp(self.num_rate * (t - t0)) for t in reg_times]), n_ex, ip([date_idx[t] for t in ptl]),
            cols[xi][0], cols[xi][1], 1, ip([cols[ui][0]]), fp([1.0]), ip([cols[ui][1]]), 0.0, fp(exercise_strikes(prod)), sign,
            xs.data_ptr(), nums.data_ptr(), imm.data_ptr(), RT.stream_ptr()))
        del paths
        tangents = None
        nt = self.nt if expo_times else 0
        if nt:
            if xi != ui:
                raise NotImplementedError("sensitivities of exposure profiles of exercise products: the explanatory "
                                          "variable must be the underlying's spot")
            dx, rows = spill if spill is not None else self.presim_tangent_spill(reg_times, dev)
            tbuf = torch.empty((2 * n_reg + n_ex) * nt * n, dtype=torch.float64, device=dev)
            dxs = tbuf[:n_reg * nt * n].view(n_reg, nt, n)
            dnums = tbuf[n_reg * nt * n:2 * n_reg * nt * n].view(n_reg, nt, n)
            dimm = tbuf[2 * n_reg * nt * n:].view(n_ex, nt, n)
            # d numeraire / d rate = (t - t0) exp(r (t - t0)), on the lane's rate (parameter 2, the numeraire's rate)
            B.check(L.mcre_lsm_prepare_equity_tangents(
                dx.data_ptr(), count, self.A, nt, n_reg, ip([rows[t] for t in reg_times]),
                fp([(t - t0) * math.exp(self.num_rate * (t - t0)) for t in reg_times]), 2, xi, n_ex,
                ip([rows[t] for t in ptl]), ui, sign, imm.data_ptr(), dxs.data_ptr(), dnums.data_ptr(), dimm.data_ptr(),
                RT.stream_ptr()))
            del dx
            tangents = dict(nt=nt, dxs=dxs, dnums=dnums, dimm=dimm)
        # standardisation of the explanatory variable per date: model moments (shard independent)
        basis = np.array([self.basis_at(xi, t) for t in reg_times]).reshape(n_reg, 2)
        gen = backward_induction_steps(xs, nums, imm, ptl, reg_times, basis, count, CHUNK_PATHS, dev, n_rights=R,
                                       tangents=tangents, batched=prepare_only)

        def finish(out):
            coef, dcoef = out if tangents is not None else (out, None)
            coef = coef.reshape(n_reg, R, 3)
            ridx = {t: k for k, t in enumerate(reg_times)}
            rows = [ridx[t] for t in ptl]
            self.exercise_coef[id(prod)] = (coef[rows], basis[rows])
            degen = [t <= t0 for t in reg_times]
            raw = np.stack([to_raw_basis(coef[:, st, :], basis, degen) for st in range(R)], axis=1)   # [n_reg, R, 3]
            # state s = rights left keeps its coefficients at row s, like the reference's [date, state, basis] tensors
            rrows = [ridx[t] for t in prod.regression_timeline.tolist()]
            if rrows:
                prod.regression_coeffs[:len(rrows), 1:R + 1, :] = torch.from_numpy(raw[rrows])
            if expo_times:
                erows = [ridx[t] for t in expo_times]
                self.exercise_expo_coef[id(prod)] = (coef[erows], basis[erows])
                c.regression_coeffs[prod.product_id][:, 1:R + 1, :] = torch.tensor(raw[erows])
                if dcoef is not None:
                    self.exercise_expo_dcoef[id(prod)] = dcoef.reshape(n_reg, R, nt, 3)[erows]

        if prepare_only:
            return gen, finish
        finish(run_backward_inductions([gen])[0])

    def _presim_rng(self, dev):
        """Draws of the pre-simulation (seed 42): Philox, or the injected reference stream."""
        c = self.c
        inj = c.injected_normals.get("pre") if c.injected_normals else None
        rng = B.Rng()
        rng.seed, rng.stream, rng.n_paths_total = 42, c.rng_stream, c.num_paths_presim
        if inj is not None:
            rng.mode, rng.d_z = B.RNG_INJECT, inj.data_ptr()
            iu = getattr(c, "injected_uniforms", None)
            iu = iu.get("pre") if iu else None
            if iu is not None:
                self._keep_u_pre = torch.as_tensor(iu, dtype=torch.float64).to(dev).contiguous()
                rng.d_u = self._keep_u_pre.data_ptr()
        else:
            rng.mode = B.RNG_PHILOX
        return rng

    def presim_tangent_spill(self, times, dev):
        """Pathwise tangents of every asset's spot at `times` on the pre-simulation paths: the spill pass of the fused
        kernel (mcre_eq_presim_tangents) on a plan without products whose spill dates are `times`, replaying the
        pre-simulation draws with tangents (under EULER the sub-steps between dates are not stored, so the tangents
        cannot come from the materialised paths).  -> (dx [len(times), A, nt, n] device, {time: row})."""
        c, L = self.c, B.lib()
        n_pre = c.num_paths_presim
        begin, count = RT.shard_range(n_pre, CHUNK_PATHS)
        n = max(count, 1)
        times = sorted(set(times))
        x = torch.zeros((len(times), self.A, n), dtype=torch.float64, device=dev)
        dx = torch.zeros((len(times), self.A, self.nt, n), dtype=torch.float64, device=dev)
        cf = torch.zeros(1, dtype=torch.float32, device=dev)          # (no products: no cashflows)
        dcf = torch.zeros(1, dtype=torch.float64, device=dev)
        desc, keep, info = self.lower([], presim_products=[], presim_tangents=True, spill_times=times)
        plan = C.c_void_p()
        B.check(L.mcre_eq_create(C.byref(desc), C.byref(plan)))
        try:
            slots = L.mcre_eq_slots(plan)
            spill_chunk = main_chunk(n_pre)
            partial = torch.empty(((n + spill_chunk - 1) // spill_chunk) * slots + slots + 1, dtype=torch.float64, device=dev)
            shift = torch.zeros(slots, dtype=torch.float64, device=dev)
            rng = self._presim_rng(dev)
            sh = B.Shard(begin, count, spill_chunk)
            B.check(L.mcre_eq_presim_tangents(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), shift.data_ptr(),
                                              x.data_ptr(), cf.data_ptr(), dx.data_ptr(), dcf.data_ptr(), RT.stream_ptr()))
        finally:
            L.mcre_eq_destroy(plan)
        return dx, {t: i for i, t in enumerate(times)}

    def presim_regression(self, products, dev):
        """Regression-proxy exposure coefficients of products that pay once (controller.py:294-383): the
        fused kernel run on the pre-simulation stream spills spots per exposure date and every product's
        float32 discounted cashflow (mcre_eq_presim); per (product, exposure date before its payment) the 8
        moments come from mcre_lsm_step, all solved in one batch after one all-reduce."""
        from mcre.lsm import solve_normal_equations_batch, to_raw_basis
        c, A = self.c, self.A
        L = B.lib()
        n_pre = c.num_paths_presim
        if n_pre <= 0:
            raise ValueError("Exposure metrics need a pre-simulation: num_paths_presim must be positive.")
        expo_times = c.exposure_timeline.tolist()
        n_expo = len(expo_times)
        begin, count = RT.shard_range(n_pre, CHUNK_PATHS)
        n = max(count, 1)
        n_chunks = (n + CHUNK_PATHS - 1) // CHUNK_PATHS
        xs = torch.zeros((n_expo, A, n), dtype=torch.float64, device=dev)
        cfs = {}
        # sensitivities through the regression (differentiate=True): the spill pass runs on a plan with tangents and
        # also writes the tangents of spots and deflated cashflows; the normal equations are differentiated below
        nt = self.nt
        if nt:
            if self.kind not in (EQ_BS, EQ_HESTON):
                raise NotImplementedError("sensitivities of regression-proxy exposures: Black-Scholes and Heston models")
            for p in products:
                ids = set(getattr(p, "asset_ids", None) or [])
                if len(ids) > 1 or getattr(p, "basket", None) is not None:
                    raise NotImplementedError("sensitivities of regression-proxy exposures: single-asset products only")
            dxs = torch.zeros((n_expo, A, nt, n), dtype=torch.float64, device=dev)
            dcfs = {}
        groups, cur, trk = [], [], 0
        for p in products:
            t = int(_is_path_dependent(p))
            if cur and trk + t > eq_ntrk(nt):
                groups.append(cur)
                cur, trk = [], 0
            cur.append(p)
            trk += t
        if cur:
            groups.append(cur)
        for group in groups:
            desc, keep, info = self.lower([], presim_products=group, presim_tangents=bool(nt))
            plan = C.c_void_p()
            B.check(L.mcre_eq_create(C.byref(desc), C.byref(plan)))
            try:
                slots = L.mcre_eq_slots(plan)
                cf = torch.zeros((len(group), n), dtype=torch.float32, device=dev)
                dcf = torch.zeros((len(group), nt, n), dtype=torch.float64, device=dev) if nt else None
                # the spill pass uses none of the kernel's sums, so its reduction chunk is free: small chunks for small
                # pre-simulations (one 4096-path chunk would put a 1000-path book on a single SM)
                spill_chunk = main_chunk(n_pre)
                partial = torch.empty(((n + spill_chunk - 1) // spill_chunk) * slots + slots + 1, dtype=torch.float64, device=dev)
                shift = torch.zeros(slots, dtype=torch.float64, device=dev)
                rng = self._presim_rng(dev)
                keep_bridge = self._set_bridge_uniforms(plan, info, "pre", n_pre, dev)
                sh = B.Shard(begin, count, spill_chunk)
                if nt:
                    B.check(L.mcre_eq_presim_tangents(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), shift.data_ptr(),
                                                      xs.data_ptr(), cf.data_ptr(), dxs.data_ptr(), dcf.data_ptr(),
                                                      RT.stream_ptr()))
                else:
                    B.check(L.mcre_eq_presim(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), shift.data_ptr(),
                                             xs.data_ptr(), cf.data_ptr(), RT.stream_ptr()))
            finally:
                L.mcre_eq_destroy(plan)
            for u, p in enumerate(group):
                cfs[id(p)] = cf[u]
                if nt:
                    dcfs[id(p)] = dcf[u]
        # standardisation of each asset's spot per date: model moments (shard independent)
        bs = np.array([[self.basis_at(a, t) for a in range(A)] for t in expo_times]).reshape(n_expo, A, 2)
        mean, scale = bs[:, :, 0], bs[:, :, 1]
        # moments per (product, date strictly before the payment)
        te_arr = np.asarray(expo_times, dtype=np.float64)
        n_before = [int(np.searchsorted(te_arr, float(p.product_timeline[-1]), side="left")) for p in products]
        jobs = [(p, k) for p, nb in zip(products, n_before) for k in range(nb)]   # expo_times is sorted
        moments = torch.zeros((max(len(jobs), 1), 8), dtype=torch.float64, device=dev)
        t0 = self.num_model.t0()
        nk_of = [math.exp(self.num_rate * (t - t0)) for t in expo_times]
        if jobs:
            # all (product, date) moments in one launch (mcre_lsm_moments_batch): job = device pointers of the date's
            # spots of the product's asset and of the product's float32 cashflows + numeraire / standardisation
            table = np.zeros(len(jobs), dtype=[("x", "u8"), ("v", "u8"), ("nk", "f8"), ("shift", "f8"), ("scale", "f8")])
            x_base, row_bytes = xs.data_ptr(), n * 8
            nk_arr, j0 = np.asarray(nk_of), 0
            for p, nb in zip(products, n_before):
                if nb == 0:
                    continue
                a, ks = self._asset_index(p.asset_ids[0]), np.arange(nb)
                seg = table[j0:j0 + nb]
                seg["x"] = x_base + (ks * A + a) * row_bytes
                seg["v"] = cfs[id(p)].data_ptr()
                seg["nk"], seg["shift"], seg["scale"] = nk_arr[:nb], mean[:nb, a], scale[:nb, a]
                j0 += nb
            partial = torch.empty(n_chunks * len(jobs) * 8 + 1, dtype=torch.float64, device=dev)
            B.check(L.mcre_lsm_moments_batch(len(jobs), table.ctypes.data, count, CHUNK_PATHS, partial.data_ptr(),
                                             moments.data_ptr(), RT.stream_ptr()))
        if nt:
            # the numeraire exp(r (t - t0)) is deterministic: its only tangent is the rate's (lane parameter 2)
            nconst = torch.empty(n, dtype=torch.float64, device=dev)
            dnconst = torch.zeros((nt, n), dtype=torch.float64, device=dev)
            tmoments = torch.zeros((max(len(jobs), 1), nt * 9), dtype=torch.float64, device=dev)
            tpartial = torch.empty(n_chunks * nt * 9 + 1, dtype=torch.float64, device=dev)
            last_k = None
            for j, (p, k) in enumerate(jobs):
                a = self._asset_index(p.asset_ids[0])
                if k != last_k:
                    nconst.fill_(nk_of[k])
                    dnconst[2].fill_((expo_times[k] - t0) * nk_of[k])
                    last_k = k
                B.check(L.mcre_lsm_step_tangents(nt, xs[k, a].data_ptr(), nconst.data_ptr(), dxs[k, a].data_ptr(),
                                                 dnconst.data_ptr(), float(mean[k, a]), float(scale[k, a]),
                                                 None, None, None, None, None, None, 0.0, 1.0, cfs[id(p)].data_ptr(),
                                                 dcfs[id(p)].data_ptr(), count, CHUNK_PATHS, tpartial.data_ptr(),
                                                 tmoments[j].data_ptr(), RT.stream_ptr()))
        m = RT.all_reduce_tree(moments).cpu().numpy()
        G = m[:, [[0, 1, 2], [1, 2, 3], [2, 3, 4]]]
        sol = solve_normal_equations_batch(G, m[:, 5:8]) if jobs else np.zeros((0, 3))
        if nt:
            from mcre.lsm import regression_tangents
            tm = RT.all_reduce_tree(tmoments).cpu().numpy().reshape(-1, nt, 9)
            for p in products:
                self.expo_dcoef[id(p)] = np.zeros((n_expo, nt, 3))
            for j, ((p, k), cvec) in enumerate(zip(jobs, sol)):
                self.expo_dcoef[id(p)][k] = regression_tangents(G[j], m[j, 5:8], cvec, tm[j])
        for p in products:
            a = self._asset_index(p.asset_ids[0])
            self.expo_coef[id(p)] = (np.zeros((n_expo, 3)), np.stack([mean[:, a], scale[:, a]], axis=1))
        j0 = 0
        for p, nb in zip(products, n_before):
            self.expo_coef[id(p)][0][:nb] = sol[j0:j0 + nb]
            j0 += nb
        for p in products:
            coef, basis = self.expo_coef[id(p)]
            c.regression_coeffs[p.product_id][:, 0, :] = torch.tensor(to_raw_basis(coef, basis, [t <= t0 for t in expo_times]))

    @staticmethod
    def _set_coef_tangents(plan, info):
        """Hands a plan with tangents the coefficient tangents of its regression-proxy and exercise exposures."""
        L = B.lib()
        if info.get("xp_tan") is not None:
            _, ptr = B.as_dp(info["xp_tan"].reshape(-1))     # (copied to the device by the call)
            B.check(L.mcre_eq_set_exposure_coef_tangents(plan, ptr))
        if info.get("xp_ex_tan") is not None:
            _, ptr = B.as_dp(info["xp_ex_tan"].reshape(-1))
            B.check(L.mcre_eq_set_exercise_exposure_coef_tangents(plan, ptr))

    def _set_bridge_uniforms(self, plan, info, which, n_total, dev):
        """RNG compatibility mode: hand the launch the reference's numpy uniforms of its Brownian-bridge barrier
        options (mcre/compat.py:inject_reference_stream); returns the device table to keep alive, or None."""
        inj = getattr(self.c, "injected_bridge", None)
        if not inj or not info["bridge"] or which not in inj:
            return None
        stride = max(n_int for _, _, n_int in info["bridge"])
        table = torch.zeros((max(sl for sl, _, _ in info["bridge"]) + 1, 2, n_total, stride), dtype=torch.float64)
        for slot, pid, n_int in info["bridge"]:
            u1, u2 = inj[which][pid]
            table[slot, 0, :, :n_int] = torch.as_tensor(u1)
            if u2 is not None:
                table[slot, 1, :, :n_int] = torch.as_tensor(u2)
        table = table.to(dev).contiguous()
        B.check(B.lib().mcre_eq_set_bridge_uniforms(plan, table.data_ptr(), stride))
        return table

    def _run_split_book(self, si, dev, n_main, n_params, chunk=None, extra_expo=None, extra_pv=None):
        """PV (and pathwise Greeks) of one netting set with more path-dependent / exercise products than a launch
        can track: the products are split over launches that replay the same Philox streams; every launch adds
        its per-path discounted cashflows to one accumulator (mcre_eq_set_pv_accumulator), the pilot shifts and
        the tangent sums add up linearly, and mcre_sum_stats finishes mean / standard error.
        `extra_expo` [n_expo][n] / `extra_pv` [n]: per-path netted exposures / discounted cashflows of products of
        ANOTHER model family of the same netting set, on the same paths (mcre/hybrid.py): the accumulators start from
        them, so that threshold / collateral, the positive parts and the CVA integrand see the whole netting set
        (controller.py:506-563 sums all products of a set before netting_set.compute_unsecured_exposure_profiles)."""
        c = self.c
        L = B.lib()
        ntrk = eq_ntrk(self.nt)
        prods = [p for p in c.netting_sets[si].products if not c._can_skip_monte_carlo_for_product(p)]
        order = {id(p): i for i, p in enumerate(c.netting_sets[si].products)}
        tracked = [p for p in prods if _is_path_dependent(p)]
        plain = [p for p in prods if not _is_path_dependent(p)]
        books = [tracked[i:i + ntrk] for i in range(0, len(tracked), ntrk)]
        if plain and books:
            books[0] = books[0] + plain
        elif plain:
            books = [plain]
        chunk = main_chunk(n_main) if chunk is None else chunk
        begin, count = RT.shard_range(n_main, chunk)
        n = max(count, 1)
        n_chunks = (n + chunk - 1) // chunk
        need_expo = c.risk_metrics.requires_exposure_profiles()
        if need_expo and self.nt:
            raise NotImplementedError("sensitivities of exposure profiles of books split over several launches")
        if need_expo and MetricType.CVA in {m.metric_type for m in c.risk_metrics.metrics} and not books:
            raise NotImplementedError("CVA of a netting set without simulated equity products in a hybrid ModelConfig: "
                                      "the default weights ride with the first equity launch")
        kinds = {m.metric_type for m in c.risk_metrics.metrics}
        n_expo, n_metric = len(c.exposure_timeline), len(c.metric_exposure_timeline)
        accum = torch.zeros(n, dtype=torch.float64, device=dev) if extra_pv is None else extra_pv.clone()
        accum_e = None
        if need_expo:
            accum_e = torch.zeros((n_expo, n), dtype=torch.float64, device=dev) if extra_expo is None else extra_expo.clone()
        # (the shift of the PV sums is the book's value on global path 0, which lives on the rank that owns it)
        shift_sum = torch.zeros(1, dtype=torch.float64, device=dev)
        if extra_pv is not None:
            first_pv = extra_pv[0:1].clone() if (begin == 0 and count > 0) else torch.zeros(1, dtype=torch.float64, device=dev)
            shift_sum += RT.all_reduce_tree(first_pv)
        grad, numtan = (np.zeros(n_params) if self.nt else None), 0.0
        cva_metric, cva_w = None, None
        for bi, book in enumerate(books):
            desc, keep, info = self.lower([si], subset=sorted(book, key=lambda p: order[id(p)]))
            plan = C.c_void_p()
            B.check(L.mcre_eq_create(C.byref(desc), C.byref(plan)))
            try:
                slots = L.mcre_eq_slots(plan)
                acc = torch.zeros(slots, dtype=torch.float64, device=dev)
                shift = torch.zeros(slots, dtype=torch.float64, device=dev)
                partial = torch.empty(n_chunks * slots + 1, dtype=torch.float64, device=dev)
                B.check(L.mcre_eq_set_pv_accumulator(plan, accum.data_ptr()))
                if need_expo:
                    B.check(L.mcre_eq_set_exposure_accumulator(plan, accum_e.data_ptr()))
                if bi == 0 and need_expo and MetricType.CVA in kinds:
                    # the first launch carries the credit factor and spills the default weights per (metric date, path)
                    cva_metric = self._set_credit(plan, info)
                    if cva_metric is not None:
                        cva_w = torch.zeros((n_metric, n), dtype=torch.float64, device=dev)
                        B.check(L.mcre_eq_set_cva_weight_spill(plan, cva_w.data_ptr()))
                        slots = L.mcre_eq_slots(plan)
                        acc = torch.zeros(slots, dtype=torch.float64, device=dev)
                        shift = torch.zeros(slots, dtype=torch.float64, device=dev)
                        partial = torch.empty(n_chunks * slots + 1, dtype=torch.float64, device=dev)
                keep_bridge = self._set_bridge_uniforms(plan, info, "main", n_main, dev)
                rng = self._rng(43, n_main)
                sh = B.Shard(begin, count, chunk)
                B.check(L.mcre_eq_mainsim(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), acc.data_ptr(),
                                          shift.data_ptr(), None, RT.stream_ptr()))
                if self.nt:
                    acc_h = RT.all_reduce_tree(acc).cpu().numpy()
                    tang = acc_h[3:3 + self.A * self.nt].reshape(self.A, 1, self.nt)
                    for a, asset in enumerate(self.assets):
                        for k, g in enumerate(asset.gmap):
                            grad[g] += tang[a, 0, k] / n_main
                    numtan += acc_h[2] / n_main
                    grad += self._control_variate_gradient(info["owners"], info["recs"], 0, n_params)
                shift_sum += shift[0:1]      # pilot values add up: the book's value on global path 0
            finally:
                L.mcre_eq_destroy(plan)
        partial = torch.empty(n_chunks * 2 * max(n_metric, 1) + 1, dtype=torch.float64, device=dev)
        out = torch.zeros(2, dtype=torch.float64, device=dev)
        B.check(L.mcre_sum_stats(accum.data_ptr(), count, 1, chunk, shift_sum.data_ptr(), 0, partial.data_ptr(),
                                 out.data_ptr(), RT.stream_ptr()))
        s = RT.all_reduce_tree(out).cpu().numpy()
        pv = mean_and_error(s[0], s[1], float(shift_sum[0]), n_main)
        if self.nt:
            grad[self.num_rate_global] += numtan
        res = {"pv": (pv, grad), "param_used": self._param_used, "_expo": accum_e, "_cva_w": cva_w}
        if need_expo:
            # netting-set terms on the accumulated exposures, then the metric sums (shift = the value on global path 0,
            # which lives on rank 0: summed over the ranks so that every rank uses the same one)
            ns = c.netting_sets[si]
            metric_expo = np.asarray(c.metric_exposure_indices.tolist(), dtype=np.int32)
            lag = np.full(n_metric, -1, dtype=np.int32)
            if ns.is_collateralized():
                delayed = c.netting_set_delayed_exposure_indices[si].tolist()
                for m in range(n_metric):
                    if delayed[m] >= 0:
                        lag[m] = int(metric_expo[m]) - delayed[m]
            spill = torch.zeros((1, n_metric, n), dtype=torch.float64, device=dev)
            me_k, me_p = B.as_ip(metric_expo)
            lg_k, lg_p = B.as_ip(lag)
            B.check(L.mcre_eq_unsecured_exposures(accum_e.data_ptr(), count, n_metric, me_p, lg_p,
                                                  int(ns.is_collateralized()), float(ns.threshold), spill.data_ptr(),
                                                  RT.stream_ptr()))
            first = spill[0, :, 0].clone() if (RT.dist_info()[0] == 0 and count > 0) else torch.zeros(n_metric, dtype=torch.float64, device=dev)
            first = RT.all_reduce_tree(first)
            for key, mode, flag in (("pos", 1, B.ACC_POS), ("neg", 2, B.ACC_NEG)):
                want = (kinds & {MetricType.CE, MetricType.EPE, MetricType.EEPE}) if key == "pos" else (MetricType.ENE in kinds)
                if not want:
                    continue
                c_shift = torch.clamp(first, min=0.0) if mode == 1 else -torch.clamp(-first, min=0.0)
                out_m = torch.zeros(n_metric * 2, dtype=torch.float64, device=dev)
                B.check(L.mcre_sum_stats(spill.data_ptr(), count, n_metric, chunk, c_shift.data_ptr(), mode,
                                         partial.data_ptr(), out_m.data_ptr(), RT.stream_ptr()))
                sm = RT.all_reduce_tree(out_m).cpu().numpy().reshape(n_metric, 2)
                ch = c_shift.cpu().numpy()
                res[key] = ([mean_and_error(sm[m, 0], sm[m, 1], ch[m], n_main) for m in range(n_metric)], [None] * n_metric)
            res["_unsec"] = spill
            if MetricType.PFE in kinds:
                from mcre.select import order_statistics
                res["pfe"] = order_statistics(c, spill, count, n_main)[0]
            if cva_metric is not None:
                cp = ns.counterparty_id
                if cp is None or cp == cva_metric.counterparty_id:
                    cva_paths = torch.zeros(n, dtype=torch.float64, device=dev)
                    B.check(L.mcre_eq_cva_paths(spill.data_ptr(), cva_w.data_ptr(), count, n_metric,
                                                1.0 - cva_metric.recovery_rate, cva_paths.data_ptr(), RT.stream_ptr()))
                    first_c = cva_paths[0:1].clone() if (RT.dist_info()[0] == 0 and count > 0) else torch.zeros(1, dtype=torch.float64, device=dev)
                    first_c = RT.all_reduce_tree(first_c)
                    out_c = torch.zeros(2, dtype=torch.float64, device=dev)
                    B.check(L.mcre_sum_stats(cva_paths.data_ptr(), count, 1, chunk, first_c.data_ptr(), 0, partial.data_ptr(),
                                             out_c.data_ptr(), RT.stream_ptr()))
                    sc_ = RT.all_reduce_tree(out_c).cpu().numpy()
                    res["cva"] = (mean_and_error(sc_[0], sc_[1], float(first_c[0]), n_main), None)
                else:
                    res["cva"] = ((0.0, 0.0), None)
        return res

    def exposure_tangent_pass(self, si, dev, n_main, chunk, credit_out=None):
        """Tangent twin of _run_split_book for hybrid books (mcre/hybrid.py): the launches of netting set `si` in
        accumulating mode on a plan with tangents.  -> (per-path tangents of the netted exposure of the set's equity
        products [n_expo][assets][nt][n] w.r.t. the lane-local parameters (spot, volatility, rate) of each asset,
        PV gradient [parameters of this backend's model] or None)."""
        c = self.c
        L = B.lib()
        ntrk = eq_ntrk(self.nt)
        prods = [p for p in c.netting_sets[si].products if not c._can_skip_monte_carlo_for_product(p)]
        order = {id(p): i for i, p in enumerate(c.netting_sets[si].products)}
        tracked = [p for p in prods if _is_path_dependent(p)]
        plain = [p for p in prods if not _is_path_dependent(p)]
        books = [tracked[i:i + ntrk] for i in range(0, len(tracked), ntrk)]
        if plain and books:
            books[0] = books[0] + plain
        elif plain:
            books = [plain]
        begin, count = RT.shard_range(n_main, chunk)
        n = max(count, 1)
        n_chunks = (n + chunk - 1) // chunk
        n_expo = len(c.exposure_timeline)
        n_params = len(c.model.model_params)
        accum = torch.zeros(n, dtype=torch.float64, device=dev)
        accum_e = torch.zeros((n_expo, n), dtype=torch.float64, device=dev)
        accum_t = torch.zeros((n_expo, self.A, self.nt, n), dtype=torch.float64, device=dev)
        grad, numtan = np.zeros(n_params), 0.0
        for book in books:
            desc, keep, info = self.lower([si], subset=sorted(book, key=lambda p: order[id(p)]))
            plan = C.c_void_p()
            B.check(L.mcre_eq_create(C.byref(desc), C.byref(plan)))
            try:
                slots = L.mcre_eq_slots(plan)
                acc = torch.zeros(slots, dtype=torch.float64, device=dev)
                shift = torch.zeros(slots, dtype=torch.float64, device=dev)
                partial = torch.empty(n_chunks * slots + 1, dtype=torch.float64, device=dev)
                B.check(L.mcre_eq_set_pv_accumulator(plan, accum.data_ptr()))
                B.check(L.mcre_eq_set_exposure_accumulator(plan, accum_e.data_ptr()))
                B.check(L.mcre_eq_set_exposure_tangent_accumulator(plan, accum_t.data_ptr()))
                self._set_coef_tangents(plan, info)
                keep_bridge = self._set_bridge_uniforms(plan, info, "main", n_main, dev)
                rng = self._rng(43, n_main)
                sh = B.Shard(begin, count, chunk)
                B.check(L.mcre_eq_mainsim(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), acc.data_ptr(),
                                          shift.data_ptr(), None, RT.stream_ptr()))
                if credit_out is not None and "w_tan" not in credit_out:
                    # (the credit factor depends on the grid and the joint draw alone: any launch's plan will do)
                    credit_out["w_tan"] = self._credit_weight_tangents(plan, info, rng, sh, n, dev)
                acc_h = RT.all_reduce_tree(acc).cpu().numpy()
                tang = acc_h[3:3 + self.A * self.nt].reshape(self.A, 1, self.nt)
                for a, asset in enumerate(self.assets):
                    for k, g in enumerate(asset.gmap):
                        grad[g] += tang[a, 0, k] / n_main
                numtan += acc_h[2] / n_main
                grad += self._control_variate_gradient(info["owners"], info["recs"], 0, n_params)
            finally:
                L.mcre_eq_destroy(plan)
        grad[self.num_rate_global] += numtan
        return accum_t, grad

    def run(self):
        c = self.c
        dev = RT.compute_device()
        L = B.lib()
        n_main = c.num_paths_mainsim
        n_sets = len(c.netting_sets)
        n_params = len(c.model.model_params)
        t0 = time.perf_counter()
        self.presim_exercise_all([p for p in c.products if is_equity_exercise(p)], dev)
        if c.risk_metrics.requires_exposure_profiles():
            reg = [p for p in c.products if not c._can_use_analytic_exposure_for_product(p) and not is_equity_exercise(p)]
            if reg:
                self.presim_regression(reg, dev)
        t_pre = time.perf_counter() - t0
        results = [None] * n_sets
        group = EQ_MAX_SETS if self.nt == 0 else 2
        # launch groups: up to `group` netting sets and eq_ntrk(nt) path-dependent / exercise products each;
        # a netting set with more tracked products than one launch holds is split over several launches
        ntrk = eq_ntrk(self.nt)
        oversized = [si for si, ns in enumerate(c.netting_sets) if sum(_is_path_dependent(p) for p in ns.products) > ntrk]
        if oversized and self.second:
            raise NotImplementedError(f"second-order sensitivities: at most {ntrk} path-dependent products per netting set")
        for si in oversized:
            results[si] = self._run_split_book(si, dev, n_main, n_params)
        groups, cur, cur_trk = [], [], 0
        for si, ns in enumerate(c.netting_sets):
            if si in oversized:
                continue
            trk = sum(_is_path_dependent(p) for p in ns.products)
            if cur and (len(cur) >= group or cur_trk + trk > ntrk):
                groups.append(cur)
                cur, cur_trk = [], 0
            cur.append(si)
            cur_trk += trk
        if cur:
            groups.append(cur)
        for idxs in groups:
            desc, keep, info = self.lower(idxs)
            plan = C.c_void_p()
            B.check(L.mcre_eq_create(C.byref(desc), C.byref(plan)))
            try:
                cva_metric = self._set_credit(plan, info)
                slots = L.mcre_eq_slots(plan)
                chunk = main_chunk(n_main)
                begin, count = RT.shard_range(n_main, chunk)
                n_chunks = max((count + chunk - 1) // chunk, 1)
                acc = torch.zeros(slots, dtype=torch.float64, device=dev)
                shift = torch.zeros(slots, dtype=torch.float64, device=dev)
                partial = torch.empty(n_chunks * slots + 1, dtype=torch.float64, device=dev)
                rng = self._rng(43, n_main)
                keep_bridge = self._set_bridge_uniforms(plan, info, "main", n_main, dev)
                if self.nt:
                    self._set_coef_tangents(plan, info)
                sh = B.Shard(begin, count, chunk)
                n_metric = info["n_metric"]
                spill = None
                if info["acc"] & B.ACC_SPILL:
                    spill = torch.empty((len(idxs), n_metric, max(count, 1)), dtype=torch.float64, device=dev)
                B.check(L.mcre_eq_mainsim(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), acc.data_ptr(),
                                          shift.data_ptr(), spill.data_ptr() if spill is not None else None,
                                          RT.stream_ptr()))
                acc = RT.all_reduce_tree(acc)
                acc_h, shift_h = acc.cpu().numpy(), shift.cpu().numpy()
                quant = None
                if spill is not None:
                    from mcre.select import order_statistics
                    quant = order_statistics(c, spill, count, n_main)
            finally:
                L.mcre_eq_destroy(plan)
            ns_t = 1 if len(idxs) <= 1 else (2 if len(idxs) <= 2 else 4)
            head = acc_h[:ns_t * 3].reshape(ns_t, 3)
            expo_base = ns_t * 3 + self.A * ns_t * self.nt
            tang = acc_h[ns_t * 3:expo_base].reshape(self.A, ns_t, self.nt) if self.nt else None
            xt_base = expo_base + n_metric * ns_t * 4
            xacc = acc_h[expo_base:xt_base].reshape(n_metric, ns_t, 4)
            xshift = shift_h[expo_base:xt_base].reshape(n_metric, ns_t, 4)
            # exposure tangents [metric date][asset][set][pos / neg][lane-local parameter] (Black-Scholes builds)
            xtan = None
            if self.nt and n_metric and self.kind in (EQ_BS, EQ_HESTON) and not self.second:
                xtan = acc_h[xt_base:].reshape(n_metric, self.A, ns_t, 2, self.nt)
            cva_acc = cva_shift = None
            if cva_metric is not None:
                cva_acc, cva_shift = acc_h[-ns_t * 2:].reshape(ns_t, 2), shift_h[-ns_t * 2:].reshape(ns_t, 2)

            def expo_grads(r, which):
                if xtan is None:
                    return [None] * n_metric
                out = []
                for m in range(n_metric):
                    g = np.zeros(n_params)
                    for a, asset in enumerate(self.assets):
                        for k, gi in enumerate(asset.gmap):
                            g[gi] += xtan[m, a, r, which, k] / n_main
                    out.append(g)
                return out
            for r, si in enumerate(idxs):
                pv = mean_and_error(head[r, 0], head[r, 1], shift_h[r], n_main)
                grad = None
                if self.nt:
                    grad = np.zeros(n_params)
                    for a, asset in enumerate(self.assets):
                        for k, g in enumerate(asset.gmap):
                            grad[g] += tang[a, r, k] / n_main
                    grad[self.num_rate_global] += head[r, 2] / n_main
                    grad += self._control_variate_gradient(info["owners"], info["recs"], r, n_params)
                res = {"pv": (pv, grad), "param_used": self._param_used}
                if self.second:
                    # lane-local upper triangles (00 01 02 11 12 22 behind the 3 first derivatives) -> the model's
                    # parameter order; entries across assets are structurally zero (single-asset products)
                    hess = np.zeros((n_params, n_params))
                    for a, asset in enumerate(self.assets):
                        k = 3
                        for i in range(3):
                            for j in range(i, 3):
                                gi, gj = asset.gmap[i], asset.gmap[j]
                                hess[gi, gj] += tang[a, r, k] / n_main
                                if gi != gj:
                                    hess[gj, gi] += tang[a, r, k] / n_main
                                k += 1
                    res["pv_hess"] = hess
                if info["acc"] & B.ACC_POS:
                    res["pos"] = ([mean_and_error(xacc[m, r, 0], xacc[m, r, 1], xshift[m, r, 0], n_main) for m in range(n_metric)],
                                  expo_grads(r, 0))
                if info["acc"] & B.ACC_NEG:
                    res["neg"] = ([mean_and_error(xacc[m, r, 2], xacc[m, r, 3], xshift[m, r, 2], n_main) for m in range(n_metric)],
                                  expo_grads(r, 1))
                if quant is not None:
                    res["pfe"] = quant[r]
                if cva_acc is not None:
                    res["cva"] = (mean_and_error(cva_acc[r, 0], cva_acc[r, 1], cva_shift[r, 0], n_main), None)
                results[si] = res
        torch.cuda.synchronize(dev)
        timings = {"preprocessing": t_pre, "path_generation": time.perf_counter() - t0 - t_pre, "request_resolution": 0.0}
        return results, timings
