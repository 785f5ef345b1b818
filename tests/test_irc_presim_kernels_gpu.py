"""The interest-rate pre-simulation kernels through the C ABI, against exact references, at the shapes where they go
wrong: mcre_irc_presim (forward spill, value and tangent moments, csrc/irc.cu and csrc/irc_tan.cu),
mcre_irc_lsm_forward (Bermudan units), mcre_irc_solve_coefficients and mcre_irc_set_coefficients_device
(csrc/irc_solve.cu), with multi-GPU sharding emulated in one process.

Plans are lowered the way production lowers them (IrcBackend.lower on tests/cases.py-style books); the references read
the lowered mcre_irc_desc tables (dual tables have stride 1 + nt) rather than re-deriving them: the goldens pin the
lowering.  Output buffers are pre-filled with NaN, so that a slot or entry the kernel forgets shows up.

References
----------
* Forward spill: a numpy restatement of the documented recurrence, in forward-mode duals [value, tangents] when the
  plan carries tangents.  Short rate: ANALYTICAL theta + (r - theta) decay + std z, EULER r + a (theta_t - r) dt +
  sigma sqrt(dt) (row of L) z; left-Riemann logB (or ext_rate dt), N = exp(logB); LIBOR from exp(B r - alpha); the
  float32 window chain W <- fp32(fp64(W) + cf / N), reset at every regression date (cashflows at or before the first
  regression date are dropped, a cashflow on date k closes window k - 1), the last window stored after the loop.
  Draws: injected normals indexed by global path, z[(is n_total + gpath) dim + j] (with |z| up to 8, so that rates go
  negative), or native Philox from oracle/philox.py (pinned to Random123 by tests/test_philox_host.py).
* Moments: computed from the kernel's OWN spilled x, N, W (read back from the scratch), so the check is exact and
  independent of the forward pass: S = fp32(W_k + S) (numpy float32 reproduces it), u = (x - shift) scale, Y = N S,
  every slot a math.fsum.  Tangent moments likewise, with the float64 tangent suffix dS.
* Solve: mpmath at 50 digits on full-rank dates, the host rule mcre/lsm.py:solve_normal_equations_batch everywhere.
  coef_sum: the unit-order sum from +0.0 of the units whose set is in range.
* Patch: the host patch mcre_irc_set_coefficients on a twin plan, both followed by the same mcre_irc_mainsim.

Tolerance model
---------------
* Moments, value and tangent, from the kernel's own spill: |got - fsum| <= 1e-13 * fsum(|terms|) per slot, for the
  totals and for every chunk row of d_partial (a path counted in the wrong chunk cancels in the total).  Slots of
  unused units are exactly zero, and d_partial past the shard's n_chunks rows stays untouched (NaN).  The tangent
  moments' own chunk rows, [chunk][unit][parameter][n_reg][9], are not observable through the entry: the value
  moments reuse d_partial after them, so the tangent moments are checked through their totals.
* x: 1e-13 absolute with injected draws; under Philox 1e-12 * sum_steps sigma sqrt(dt) (Box-Muller on the device
  against host libm differ by <= 1e-12 per normal, as in tests/test_paths_gpu.py).  A lost, doubled or mis-paired
  step moves x by sigma sqrt(dt) |z|.
* N and imm: 1e-13 relative to the magnitude of the terms (the table-driven exp is <= 2 ulp, tests/test_fastmath_*).
  Under Philox N carries the error of x through logB = sum r dt: 1e-13 + T tol_x, T the simulated horizon.
* W (float32), injected draws: bit-identical, except on windows where the reference's float64 pre-rounding value at
  some step lay within 1e-12 relative of a float32 rounding midpoint: one float32 ulp per such step.  Philox: one
  float32 ulp per cashflow date in the window.
* Tangent spills: 1e-12 relative to each array's largest magnitude.
* Solve: coefficients 1e-12 relative to mpmath on well-conditioned full-rank dates; fitted values on the sample
  support within 1e-12 of the largest fitted value against the host rule.  Two dates sit on either side of the 1e-10
  rank cut (rank measure 3e-10 and 3e-11, asserted).  Above it (condition ~3e9) fits agree to 1e-6 with the host
  rule and with mpmath, below it to 1e-9 with the host rule; there the rank-3 and rank-2 fits differ by more than 100
  times the tolerance, so a cut moved past either date fails.
  coef_sum, patch and sharding: bit-identical.

The largest allocation is about 120 MB (the scratch of the 3300-date tangent plan); the module stays below 1 GB."""
import ctypes as C
import math
import os
import subprocess
import sys

import mpmath
import numpy as np
import pytest
import torch

import cases
from mcre import binding as B
from mcre import runtime as RT
from mcre.irc import IrcBackend
from mcre.lsm import solve_normal_equations_batch
from oracle import philox

pytestmark = pytest.mark.gpu

SUM_RTOL = 1e-13
TM_NV = 9
PARTIAL_PAD = 64            # doubles past what the entry may write to d_partial: they must stay NaN


# ---- books and plans ------------------------------------------------------------------------------------------------
def _vasicek(ns, hw=False, sigma=0.02):
    if hw:
        return ns.HullWhiteModel(0., 0.03, 0.05, 0.1, sigma, asset_id="irs", mean_times=[0.3, 0.7, 1.2],
                                 mean_levels=[0.01, 0.06, -0.01])
    return ns.VasicekModel(0., 0.03, 0.05, 0.1, sigma, asset_id="irs")


def _model(ns, kind):
    """kind: vas | hw | vas_cir (rate on noise column 0) | cir_vas (rate on column 1) | vas_cir_det."""
    if kind in ("vas", "hw"):
        return _vasicek(ns, hw=kind == "hw")
    cir = ns.CIRPPModel(0., "GM", cases.HAZARDS, 0.1, 0.01, 0.02, 0.0001, deterministic=kind == "vas_cir_det")
    vas = _vasicek(ns)
    if kind == "cir_vas":
        return ns.ModelConfig([cir, vas], numeraire_model_idx=1, discount_model_idx=1,
                              inter_asset_correlation_matrix=np.array([0.6]))
    return ns.ModelConfig([vas, cir], inter_asset_correlation_matrix=np.array([-0.4]))


def _units(ns, n_units, maturity):
    """Payer and receiver swaps and a coupon bond, all paying inside, before and after the regression grid."""
    out = []
    for u in range(n_units):
        if u == 2:
            out.append(ns.Bond(0.0, maturity * 1.1, 1.0, 0.25, fixed_rate=0.02, asset_id="irs"))
        else:
            kind = ns.IRSType.PAYER if u % 2 == 0 else ns.IRSType.RECEIVER
            out.append(ns.InterestRateSwap(0.0, maturity * (1.0 + 0.15 * u), 1.0 + u, 0.03, 0.25, 0.25, kind,
                                           asset_id="irs"))
    return out


def _controller(kind="vas", n_units=1, tl=None, scheme="EULER", differentiate=False, num_steps=1, maturity=2.0):
    ns = cases.Namespace()
    model = _model(ns, kind)
    units = _units(ns, n_units, maturity)
    tl = np.linspace(0.0, maturity, 9) if tl is None else np.asarray(tl, dtype=np.float64)
    rm = ns.RiskMetrics([ns.EPEMetric()], exposure_timeline=tl)
    sets = [ns.NettingSet(name="s", products=units)]
    sc = ns.SimulationController(sets, model, rm, 256, 256, num_steps, getattr(ns.SimulationScheme, scheme),
                                 differentiate)
    return ns, sc, units


class Plan:
    def __init__(self, desc):
        self.p = C.c_void_p()
        B.check(B.lib().mcre_irc_create(C.byref(desc), C.byref(self.p)))

    def __enter__(self):
        return self.p

    def __exit__(self, *a):
        B.lib().mcre_irc_destroy(self.p)


def _presim_plan(kind="vas", n_units=1, **kw):
    ns, sc, units = _controller(kind, n_units, **kw)
    be = IrcBackend(sc)
    desc, keep, info = be.lower([], units)
    return be, desc, keep, info


def _tables(desc, keep):
    """The descriptor tables the kernels read (numpy views of the lowered host arrays)."""
    t = {k: np.asarray(v) for k, v in keep.items()}
    t.update(nt=desc.nt, w=1 + desc.nt, n_sub=desc.n_sub, n_pre=desc.n_pre_dates, n_reg=desc.n_reg,
             n_units=desc.n_units, n_dates=desc.n_dates, has_cir=desc.has_cir, vas_noise=desc.vas_noise,
             analytical=desc.scheme == B.SCHEME_ANALYTICAL, ext=desc.ext_numeraire, ext_rate=desc.ext_rate)
    return t


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _smem_optin():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _nan(n):
    return torch.full((max(int(n), 1),), float("nan"), dtype=torch.float64, device="cuda")


def _rng(mode, n_total, z=None, seed=42, stream=0):
    r = B.Rng()
    r.mode, r.seed, r.stream, r.n_paths_total = mode, seed, stream, n_total
    if z is not None:
        r.d_z = z.data_ptr()
    return r


def _normals(n_sub, n_total, dim, seed):
    g = np.random.default_rng(seed)
    z = g.standard_normal((n_sub, n_total, dim))
    hot = g.choice(z.size, size=max(1, z.size // 200), replace=False)
    z.flat[hot] = np.where(g.random(hot.size) < 0.5, -8.0, 8.0)
    return z


def _run_presim(plan, desc, n, chunk, rng, begin=0, scratch_fill=float("nan")):
    L = B.lib()
    scratch = torch.full((L.mcre_irc_presim_scratch_bytes(plan, max(n, 1)) // 8 + 1,), scratch_fill,
                         dtype=torch.float64, device="cuda")
    written = L.mcre_irc_partial_bytes(plan, max(n, 1), chunk, 1) // 8
    partial = _nan(written + PARTIAL_PAD)
    mom = _nan(L.mcre_irc_presim_slots(plan))
    tslots = L.mcre_irc_presim_tangent_slots(plan)
    tmom = _nan(tslots) if desc.nt else None
    sh = B.Shard(begin, n, chunk)
    rc = L.mcre_irc_presim(plan, C.byref(rng), C.byref(sh), scratch.data_ptr(), partial.data_ptr(), mom.data_ptr(),
                           tmom.data_ptr() if tmom is not None else None, RT.stream_ptr())
    torch.cuda.synchronize()
    # rows past the shard's n_chunks (past its n_chunks tangent rows on tangent plans) are left untouched
    assert torch.isnan(partial[written:]).all(), "d_partial written past its n_chunks rows"
    return rc, scratch, partial, mom, tmom


def _spill(scratch, t, n):
    """x [n_reg][n], N [n_reg][n], W [n_units][n_reg][n] f32 (+ dx, dN [n_reg][nt][n], dW [n_units][n_reg][nt][n])."""
    R, U, nt = t["n_reg"], t["n_units"], t["nt"]
    raw = scratch.cpu().numpy()
    x = raw[:R * n].reshape(R, n)
    N = raw[R * n:2 * R * n].reshape(R, n)
    wcount = U * R * n
    W = raw[2 * R * n:].view(np.float32)[:wcount].reshape(U, R, n)
    out = dict(x=x, N=N, W=W)
    if nt:
        off = 2 * R * n + (wcount + 1) // 2
        out["dx"] = raw[off:off + R * nt * n].reshape(R, nt, n)
        out["dN"] = raw[off + R * nt * n:off + 2 * R * nt * n].reshape(R, nt, n)
        out["dW"] = raw[off + 2 * R * nt * n:off + (2 * R + U * R) * nt * n].reshape(U, R, nt, n)
    return out


# ---- 1. the forward restatement (forward-mode duals: row 0 value, rows 1.. tangents) ----------------------------------
def _d(table, i, w):
    return np.asarray(table[i * w:(i + 1) * w], dtype=np.float64)[:, None]


def _mul(a, b):
    out = np.empty(np.broadcast_shapes(a.shape, b.shape))
    out[0] = a[0] * b[0]
    out[1:] = a[0] * b[1:] + a[1:] * b[0]
    return out


def _exp(a):
    e = np.exp(a[0])
    return np.concatenate([e[None], e * a[1:]])


def _draws(t, n, begin, inject_z, philox_seed):
    dim = 2 if t["has_cir"] else 1
    if inject_z is not None:
        return inject_z[:, begin:begin + n, :]
    return philox.normals(np.arange(begin, begin + n, dtype=np.uint64), t["n_sub"], dim, philox_seed, 0)


def _forward_ref(t, n, z, berm=False):
    """Restated pre-simulation of one shard -> dict of x, N [n_reg][w][n], W [n_units][n_reg][w][n] (value rounded
    through float32 as the kernel does), W_mid [n_units][n_reg][n] (steps near a float32 midpoint), W_cf (cashflow
    dates per window); Bermudan plans: imm [n_ex][w][n]."""
    w, R, U = t["w"], t["n_reg"], t["n_units"]
    vas, chol = t["vas"], t["chol"]
    r = np.repeat(_d(vas, 0, w), n, axis=1)
    sigma, theta, a = _d(vas, 1, w), _d(vas, 2, w), _d(vas, 3, w)
    second = t["has_cir"] and t["vas_noise"] == 1
    l0 = _d(chol, 2 if second else 0, w)
    l1 = _d(chol, 3, w) if second else np.zeros((w, 1))
    logB = np.zeros((w, n))
    Wv = [np.zeros((w, n)) for _ in range(U)]
    mid = [np.zeros(n, dtype=np.int64) for _ in range(U)]
    ncf = [0] * U
    out = dict(x=np.full((R, w, n), np.nan), N=np.full((R, w, n), np.nan),
               W=np.full((U, R, w, n), np.nan), W_mid=np.zeros((U, R, n), dtype=np.int64),
               W_cf=np.zeros((U, R), dtype=np.int64))
    if berm:
        n_ex = int(t["ex_off"][-1])
        out["imm"] = np.full((n_ex, w, n), np.nan)
        out["imm_raw"] = np.full((n_ex, n), np.nan)
    flags, date_reg, foff = t["flags"], t["date_reg"], t["float_off"]

    def store(u, k):
        out["W"][u, k], out["W_mid"][u, k], out["W_cf"][u, k] = Wv[u], mid[u], ncf[u]

    def eval_date(di):
        f = int(flags[di])
        if berm:
            if f & B.DATE_HAS_REGRESSION:
                k = int(date_reg[di])
                out["x"][k], out["N"][k] = r, _exp(logB)
            if f & B.DATE_HAS_EXERCISE:
                for xi in range(int(t["ex_off"][di]), int(t["ex_off"][di + 1])):
                    U_ = np.zeros((w, n))
                    U_[0] = t["ex_const"][xi]
                    for j in range(int(t["ex_term_off"][xi]), int(t["ex_term_off"][xi + 1])):
                        al, Bc = _d(t["term_coef"], 2 * j, w), _d(t["term_coef"], 2 * j + 1, w)
                        U_ = U_ + _exp(al - _mul(Bc, r)) * t["term_w"][j]
                    b = int(t["ex_unit"][xi])
                    v = (U_ - t["berm_strike"][b]) * t["berm_sign"][b]
                    out["imm"][xi] = np.where((v[0] >= 0.0)[None], v, 0.0)
                    out["imm_raw"][xi] = v[0]
            return
        if not f & (B.DATE_HAS_CASHFLOW | B.DATE_HAS_REGRESSION):
            return
        num = _exp(logB)
        if f & B.DATE_HAS_CASHFLOW:
            inv = np.concatenate([1.0 / num[0:1], -num[1:] / num[0:1] ** 2])
            for u in range(U):
                cf = np.zeros((w, n))
                cf[0] = t["unit_fix"][u, di]
                for j in range(int(foff[di]), int(foff[di + 1])):
                    al, Bc = _d(t["float_coef"], 2 * j, w), _d(t["float_coef"], 2 * j + 1, w)
                    e = _exp(_mul(Bc, r) - al)
                    e[0] -= 1.0
                    cf = cf + e * t["float_inv_tau"][j] * t["unit_float"][u, j]
                pre = Wv[u] + _mul(cf, inv)
                v32 = pre[0].astype(np.float32)
                half = np.spacing(np.abs(v32)).astype(np.float64) / 2.0
                dist = np.abs(np.abs(pre[0] - v32.astype(np.float64)) - half)
                mid[u] = mid[u] + (dist <= 1e-12 * np.abs(pre[0]))
                ncf[u] += 1
                pre[0] = v32.astype(np.float64)
                Wv[u] = pre
        if f & B.DATE_HAS_REGRESSION:
            k = int(date_reg[di])
            out["x"][k], out["N"][k] = r, num
            for u in range(U):
                if k > 0:
                    store(u, k - 1)
                Wv[u], mid[u], ncf[u] = np.zeros((w, n)), np.zeros(n, dtype=np.int64), 0

    for di in range(t["n_pre"]):
        eval_date(di)
    for s in range(t["n_sub"]):
        dt = float(t["step_dt"][s])
        z0 = z[s, :, 0]
        z1 = z[s, :, 1] if z.shape[2] > 1 else np.zeros(n)
        if t["ext"]:
            logB = logB + np.concatenate([np.full((1, n), t["ext_rate"] * dt), np.zeros((w - 1, n))])
        else:
            logB = logB + r * dt
        sv0, sv1 = _d(t["step_vas"], 2 * s, w), _d(t["step_vas"], 2 * s + 1, w)
        if t["analytical"]:
            r = theta + _mul(r - theta, sv0) + sv1 * z0
        else:
            wv = l0 * z0 + l1 * z1
            r = r + _mul(a, sv0 - r) * dt + _mul(sigma, wv) * math.sqrt(dt)
        di = int(t["step_date"][s])
        if di >= 0:
            eval_date(di)
    if not berm and R > 0:
        for u in range(U):
            store(u, R - 1)
    return out


def _sigma_path(t):
    """sum over steps of sigma sqrt(dt) (the Philox tolerance unit of x)."""
    return float(np.sum(t["vas"][1 * t["w"]] * np.sqrt(np.asarray(t["step_dt"], dtype=np.float64))))


def _check_forward(t, got, ref, philox_draws, what):
    w = t["w"]
    tol_x = 1e-12 * _sigma_path(t) if philox_draws else 1e-13
    assert np.all(np.isfinite(got["x"])), what
    assert np.max(np.abs(got["x"] - ref["x"][:, 0])) <= tol_x, f"{what}: x off by {np.max(np.abs(got['x'] - ref['x'][:, 0]))}"
    if not philox_draws:
        assert (ref["x"][:, 0] < 0).any(), f"{what}: no negative rates reached"
    relN = np.abs(got["N"] - ref["N"][:, 0]) / np.abs(ref["N"][:, 0])
    # under Philox logB = sum r dt inherits the error of x: |d logB| <= T tol_x over the simulated horizon T
    tol_N = 1e-13 + (float(np.sum(t["step_dt"])) * tol_x if philox_draws else 0.0)
    assert relN.max() <= tol_N, f"{what}: N {relN.max()} (tolerance {tol_N})"
    if t["n_units"]:
        Wg, Wr = got["W"].astype(np.float64), ref["W"][:, :, 0]
        ulp = np.spacing(np.abs(ref["W"][:, :, 0]).astype(np.float32)).astype(np.float64)
        if philox_draws:
            allow = ref["W_cf"][:, :, None] * ulp
        else:
            allow = ref["W_mid"] * ulp
        bad = np.abs(Wg - Wr) > allow
        assert not bad.any(), f"{what}: W differs at {np.argwhere(bad)[:5].tolist()} ({Wg[bad][:5]} vs {Wr[bad][:5]})"
        if not philox_draws:
            print(f"{what}: {int((ref['W_mid'] > 0).sum())} windows within 1e-12 of a float32 midpoint")
    if w > 1:
        for name, tname in (("x", "dx"), ("N", "dN")):
            refd = np.transpose(ref[name][:, 1:], (0, 1, 2))
            scale = max(np.abs(refd).max(), 1e-300)
            assert np.max(np.abs(got[tname] - refd)) <= 1e-12 * scale, f"{what}: {tname}"
        if t["n_units"]:
            refd = ref["W"][:, :, 1:]
            scale = max(np.abs(refd).max(), 1e-300)
            assert np.max(np.abs(got["dW"] - refd)) <= 1e-12 * scale, f"{what}: dW"


FORWARD_CASES = [
    # (model, scheme, n_units, num_steps, draws, ext_numeraire)
    ("vas", "ANALYTICAL", 1, 3, "inject", False),
    ("vas", "EULER", 2, 3, "inject", False),
    ("hw", "EULER", 3, 3, "inject", False),
    ("vas_cir", "EULER", 4, 2, "inject", False),
    ("cir_vas", "EULER", 2, 2, "inject", False),
    ("vas_cir_det", "EULER", 1, 2, "inject", False),
    ("vas", "EULER", 2, 3, "inject", True),
    ("vas", "EULER", 1, 3, "philox", False),
    ("hw", "ANALYTICAL", 2, 3, "philox", False),
    ("cir_vas", "EULER", 3, 2, "philox", False),
]


def _forward_plan(kind, scheme, n_units, num_steps, differentiate=False, tl=None):
    # regression grid 0.25 .. 1.75 (t = 0 not a regression date here) on a 2y book: cashflows before the first date,
    # on regression dates (quarterly coupons) and after the last one
    tl = np.array([0.25, 0.5, 0.6, 1.0, 1.25, 1.75]) if tl is None else tl
    return _presim_plan(kind, n_units, tl=tl, scheme=scheme, num_steps=num_steps, differentiate=differentiate,
                        maturity=2.0)


@pytest.mark.parametrize("kind,scheme,n_units,num_steps,draws,ext", FORWARD_CASES)
def test_presim_forward_spill_matches_restatement(kind, scheme, n_units, num_steps, draws, ext):
    be, desc, keep, info = _forward_plan(kind, scheme, n_units, num_steps)
    if ext:
        desc = B.IrcDesc.from_buffer_copy(desc)      # (the lowered descriptor may be shared through the plan cache)
        desc.ext_numeraire, desc.ext_rate = 1, 0.021
    t = _tables(desc, keep)
    n, begin, n_total = 1100, 0, 1100        # two full 512-path blocks and a ragged tail
    dim = 2 if t["has_cir"] else 1
    z = _normals(t["n_sub"], n_total, dim, 5) if draws == "inject" else None
    zt = torch.from_numpy(z.ravel()).cuda() if z is not None else None
    rng = _rng(B.RNG_INJECT if z is not None else B.RNG_PHILOX, n_total, zt, seed=42)
    with Plan(desc) as plan:
        rc, scratch, _, _, _ = _run_presim(plan, desc, n, 256, rng)
    B.check(rc)
    got = _spill(scratch, t, n)
    ref = _forward_ref(t, n, _draws(t, n, begin, z, 42))
    _check_forward(t, got, ref, draws == "philox", f"{kind}/{scheme}/{n_units}/{draws}/ext={ext}")


def test_presim_forward_odd_substeps_philox_regression_date_at_zero_and_one_date():
    """Vasicek-only Philox (one Box-Muller pair serves two sub-steps) with an odd n_sub, n_reg = 1 at t = 0 (every
    cashflow lands in the one window after it) and a t = 0 date on a longer grid."""
    odd = False
    for tl, steps in ((np.array([0.0]), 1), (np.array([0.0, 0.1, 0.35, 1.1]), 1), (np.array([0.0, 0.1, 0.35, 1.1]), 3)):
        be, desc, keep, info = _forward_plan("vas", "EULER", 2, steps, tl=tl)
        t = _tables(desc, keep)
        odd = odd or t["n_sub"] % 2 == 1
        n = 700
        with Plan(desc) as plan:
            rc, scratch, _, _, _ = _run_presim(plan, desc, n, 256, _rng(B.RNG_PHILOX, n, seed=7))
        B.check(rc)
        ref = _forward_ref(t, n, _draws(t, n, 0, None, 7))
        _check_forward(t, _spill(scratch, t, n), ref, True, f"tl={tl.tolist()} n_sub={t['n_sub']}")
    assert odd, "no case with an odd number of sub-steps"


# ---- 2. value moments from the kernel's own spill ---------------------------------------------------------------------
def _value_terms(sp, t, k, lo, hi):
    """Per-path terms of the value slots of date k over paths [lo, hi) -> list of arrays [5 + 3 NU]."""
    bs, bc = t["reg_basis"].reshape(-1, 2)[k]
    uu = (sp["x"][k, lo:hi] - bs) * bc
    u2 = uu * uu
    terms = [np.ones_like(uu), uu, u2, u2 * uu, u2 * uu * uu]
    for u in range(t["n_units"]):
        Y = sp["N"][k, lo:hi] * sp["S"][u][k][lo:hi].astype(np.float64)
        terms += [Y, Y * uu, Y * uu * uu]
    return terms


def _suffixes(sp, t):
    """S[u][k] = fp32(W_k + S_{k+1}), numpy float32 (correctly rounded, like the kernel's float add)."""
    R = t["n_reg"]
    S = []
    for u in range(t["n_units"]):
        acc = np.zeros(sp["W"].shape[2], dtype=np.float32)
        per = [None] * R
        for k in range(R - 1, -1, -1):
            acc = sp["W"][u, k] + acc
            per[k] = acc
        S.append(per)
    return S


def _assert_slot(got, terms, what):
    ref, mag = math.fsum(terms), math.fsum(np.abs(terms))
    assert abs(got - ref) <= SUM_RTOL * mag, f"{what}: {got!r} vs fsum {ref!r} (sum |t| {mag:.3e})"


def _check_value_moments(sp, t, n, chunk, mom, partial, nu, chunk_rows=True):
    nv = 5 + 3 * nu
    R = t["n_reg"]
    sp["S"] = _suffixes(sp, t)
    mom = mom.reshape(R, nv)
    n_chunks = (n + chunk - 1) // chunk
    for k in range(R):
        terms = _value_terms(sp, t, k, 0, n)
        for j, tj in enumerate(terms):
            _assert_slot(mom[k, j], tj, f"moment date {k} slot {j}")
        assert np.all(mom[k, len(terms):] == 0.0), f"date {k}: unused unit slots {mom[k, len(terms):]}"
    if not chunk_rows:
        return
    rows = partial[:n_chunks * R * nv].reshape(n_chunks, R, nv)
    for c in range(n_chunks):
        lo, hi = c * chunk, min(n, (c + 1) * chunk)
        for k in range(R):
            terms = _value_terms(sp, t, k, lo, hi)
            for j, tj in enumerate(terms):
                _assert_slot(rows[c, k, j], tj, f"chunk {c} date {k} slot {j}")
            assert np.all(rows[c, k, len(terms):] == 0.0)


@pytest.mark.parametrize("chunk", [256, 768, 4096])
@pytest.mark.parametrize("n_units", [1, 2, 3])
def test_presim_value_moments_match_fsum_of_own_spill(chunk, n_units):
    be, desc, keep, info = _forward_plan("vas", "EULER", n_units, 2)
    t = _tables(desc, keep)
    nu = 1 if n_units <= 1 else (2 if n_units <= 2 else 4)
    with Plan(desc) as plan:
        for n in (1, 127, 128, 511, 512, 513, 4095, 4096, 4097):
            rng = _rng(B.RNG_PHILOX, 5000, seed=3)
            rc, scratch, partial, mom, _ = _run_presim(plan, desc, n, chunk, rng)
            B.check(rc)
            sp = _spill(scratch, t, n)
            _check_value_moments(sp, t, n, chunk, mom.cpu().numpy(), partial.cpu().numpy(), nu)


def test_presim_value_moments_past_the_grid_cap():
    """sm_count * 8 + 1 chunks of 256 paths: more chunks than any occupancy-derived grid, so the chunk loop strides."""
    be, desc, keep, info = _forward_plan("vas", "EULER", 1, 1, tl=np.array([0.5, 1.5]))
    t = _tables(desc, keep)
    n = (_sm_count() * 8 + 1) * 256 - 77
    with Plan(desc) as plan:
        rc, scratch, partial, mom, _ = _run_presim(plan, desc, n, 256, _rng(B.RNG_PHILOX, n, seed=9))
    B.check(rc)
    _check_value_moments(_spill(scratch, t, n), t, n, 256, mom.cpu().numpy(), partial.cpu().numpy(), 1)


def _many_dates_plan(n_reg, n_units, differentiate=False):
    tl = np.linspace(0.0, 2.0, n_reg)
    return _presim_plan("vas", n_units, tl=tl, num_steps=1, differentiate=differentiate, maturity=2.0)


@pytest.mark.parametrize("n_units,n_reg", [(1, 496), (1, 497), (1, 498), (4, 224), (4, 225), (4, 226)])
def test_presim_value_moments_across_the_shared_memory_switch(n_units, n_reg):
    """(n_reg (5 + 3 NU) + 16 (5 + 3 NU)) doubles of shared memory: 32 KB is crossed at 497 dates (NU = 1) and 225
    (NU = 4); above it the launch requests the opt-in."""
    be, desc, keep, info = _many_dates_plan(n_reg, n_units)
    t = _tables(desc, keep)
    assert t["n_reg"] == n_reg
    nu = 1 if n_units == 1 else 4
    n = 300
    with Plan(desc) as plan:
        rc, scratch, partial, mom, _ = _run_presim(plan, desc, n, 256, _rng(B.RNG_PHILOX, n, seed=4))
    B.check(rc)
    _check_value_moments(_spill(scratch, t, n), t, n, 256, mom.cpu().numpy(), partial.cpu().numpy(), nu)


# ---- 3. tangent pre-simulation ------------------------------------------------------------------------------------------
def _check_tangent_moments(sp, t, n, tmom):
    nt, R, U = t["nt"], t["n_reg"], t["n_units"]
    tmom = tmom.reshape(U, nt, R, TM_NV)
    bsc = t["reg_basis"].reshape(-1, 2)
    for u in range(U):
        S = np.zeros(n, dtype=np.float32)
        dS = np.zeros((nt, n))
        for k in range(R - 1, -1, -1):
            S = sp["W"][u, k] + S
            dS = dS + sp["dW"][u, k]
            bs, bc = bsc[k]
            uu = (sp["x"][k] - bs) * bc
            Y = sp["N"][k] * S.astype(np.float64)
            for ip in range(nt):
                du = sp["dx"][k, ip] * bc
                dY = sp["dN"][k, ip] * S.astype(np.float64) + sp["N"][k] * dS[ip]
                u2 = uu * uu
                terms = [du, uu * du, u2 * du, u2 * uu * du, dY, uu * dY, u2 * dY, du * Y, 2.0 * uu * du * Y]
                for j, tj in enumerate(terms):
                    _assert_slot(tmom[u, ip, k, j], tj, f"tangent moment unit {u} param {ip} date {k} slot {j}")


@pytest.mark.parametrize("kind,scheme,n_units,draws", [("vas", "EULER", 1, "inject"), ("hw", "ANALYTICAL", 2, "philox"),
                                                       ("vas_cir", "EULER", 3, "inject"), ("cir_vas", "EULER", 2, "philox")])
def test_presim_tangents_match_dual_restatement_and_fsum(kind, scheme, n_units, draws):
    """nt = 4 (Vasicek) and nt = 8 (Vasicek + CIR++) plans: the spilled dx, dN, dW against the dual restatement,
    the tangent moments [n_units][nt][n_reg][9] and the value moments against fsum over the kernel's own spill."""
    be, desc, keep, info = _forward_plan(kind, scheme, n_units, 2, differentiate=True)
    t = _tables(desc, keep)
    assert t["nt"] in (4, 8)
    n = 1300
    dim = 2 if t["has_cir"] else 1
    z = _normals(t["n_sub"], n, dim, 12) if draws == "inject" else None
    zt = torch.from_numpy(z.ravel()).cuda() if z is not None else None
    rng = _rng(B.RNG_INJECT if z is not None else B.RNG_PHILOX, n, zt, seed=42)
    with Plan(desc) as plan:
        rc, scratch, partial, mom, tmom = _run_presim(plan, desc, n, 256, rng)
    B.check(rc)
    sp = _spill(scratch, t, n)
    ref = _forward_ref(t, n, _draws(t, n, 0, z, 42))
    _check_forward(t, sp, ref, draws == "philox", f"tangent {kind}/{scheme}/{n_units}/{draws}")
    nu = 1 if n_units <= 1 else (2 if n_units <= 2 else 4)
    _check_value_moments(sp, t, n, 256, mom.cpu().numpy(), partial.cpu().numpy(), nu)
    _check_tangent_moments(sp, t, n, tmom.cpu().numpy())


@pytest.mark.parametrize("n_reg", [439, 440, 441])
def test_presim_tangent_moments_across_the_shared_memory_switch(n_reg):
    be, desc, keep, info = _many_dates_plan(n_reg, 1, differentiate=True)
    t = _tables(desc, keep)
    n = 260
    with Plan(desc) as plan:
        rc, scratch, partial, mom, tmom = _run_presim(plan, desc, n, 256, _rng(B.RNG_PHILOX, n, seed=4))
    B.check(rc)
    sp = _spill(scratch, t, n)
    _check_tangent_moments(sp, t, n, tmom.cpu().numpy())


# ---- 4. Bermudan forward -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("differentiate", [False, True])
@pytest.mark.parametrize("payer", [True, False])
def test_lsm_forward_matches_restatement(payer, differentiate):
    ns = cases.Namespace()
    model = _vasicek(ns, hw=True)
    kind = ns.IRSType.PAYER if payer else ns.IRSType.RECEIVER
    swap = ns.InterestRateSwap(0.0, 3.0, 1.0, 0.03, 0.25, 0.25, kind)
    ex = [0.25 * (i + 1) for i in range(8)]
    opt = ns.BermudanOption(swap, ex, 0.0, ns.OptionType.CALL if payer else ns.OptionType.PUT)
    tl = np.array([0.25 * i for i in range(9)])
    rm = ns.RiskMetrics([ns.EPEMetric()], exposure_timeline=tl)
    sc = ns.SimulationController([ns.NettingSet(name="b", products=[opt])], model, rm, 256, 256, 2,
                                 ns.SimulationScheme.EULER, differentiate)
    be = IrcBackend(sc)
    reg_times = sorted(set(opt.regression_timeline.tolist()) | set(tl.tolist()))
    desc, keep, info = be.lower([], [], berm_units=[(opt, 0)], reg_times=reg_times)
    t = _tables(desc, keep)
    w, R, n_ex = t["w"], t["n_reg"], info["n_ex"]
    n = 1100
    z = _normals(t["n_sub"], n, 1, 21)
    zt = torch.from_numpy(z.ravel()).cuda()
    L = B.lib()
    with Plan(desc) as plan:
        scratch = torch.full((L.mcre_irc_lsm_scratch_bytes(plan, n) // 8,), float("nan"), dtype=torch.float64,
                             device="cuda")
        B.check(L.mcre_irc_lsm_forward(plan, C.byref(_rng(B.RNG_INJECT, n, zt)), C.byref(B.Shard(0, n, 256)),
                                       scratch.data_ptr(), RT.stream_ptr()))
        torch.cuda.synchronize()
    raw = scratch.cpu().numpy()
    x, N, imm = raw[:R * n].reshape(R, n), raw[R * n:2 * R * n].reshape(R, n), raw[2 * R * n:(2 * R + n_ex) * n].reshape(n_ex, n)
    ref = _forward_ref(t, n, z, berm=True)
    assert np.max(np.abs(x - ref["x"][:, 0])) <= 1e-13
    assert np.max(np.abs(N - ref["N"][:, 0]) / ref["N"][:, 0]) <= 1e-13
    rimm = ref["imm"][:, 0]
    mag = np.abs(t["ex_const"])[:, None] + 10.0           # |U| + K: the terms of sign (U - K) are O(notional)
    assert np.all(np.abs(imm - rimm) <= 1e-13 * mag), np.max(np.abs(imm - rimm))
    # where sign (U - K) is clearly negative the immediate value is exactly +0.0
    clear = ref["imm_raw"] < -1e-9
    assert clear.any() and (ref["imm_raw"] > 1e-9).any()
    assert np.all(imm[clear] == 0.0) and not np.signbit(imm[clear]).any()
    if differentiate:
        off = (2 * R + n_ex) * n
        nt = t["nt"]
        dx = raw[off:off + R * nt * n].reshape(R, nt, n)
        dN = raw[off + R * nt * n:off + 2 * R * nt * n].reshape(R, nt, n)
        dimm = raw[off + 2 * R * nt * n:off + (2 * R + n_ex) * nt * n].reshape(n_ex, nt, n)
        for got, want, what in ((dx, ref["x"][:, 1:], "dx"), (dN, ref["N"][:, 1:], "dN"), (dimm, ref["imm"][:, 1:], "dimm")):
            ok = np.abs(got - want) <= 1e-12 * max(np.abs(want).max(), 1e-300)
            if what == "dimm":      # at the kink the two sides may pick different branches
                ok |= (np.abs(ref["imm_raw"]) <= 1e-12)[:, None, :]
            assert ok.all(), what
        # out of the money the tangent of max(sign (U - K), 0) is exactly zero
        assert np.all(dimm.transpose(0, 2, 1)[clear] == 0.0)


# ---- 5. sharding -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("draws", ["inject", "philox"])
@pytest.mark.parametrize("n_units", [1, 3])
def test_presim_shards_are_bit_identical_to_the_full_run(draws, n_units):
    """Chunk-aligned shards [b, b + m) give the full run's scratch columns and d_partial rows bit for bit, and shards
    of power-of-two chunk counts combined by RT.tree_sum give its total moments bit for bit (the layout
    IrcBackend.presim_coefficients relies on when it calls the entry at begin + b0)."""
    be, desc, keep, info = _forward_plan("vas_cir", "EULER", n_units, 2)
    t = _tables(desc, keep)
    chunk = 256
    n = 8 * chunk - 100
    z = _normals(t["n_sub"], n, 2, 31) if draws == "inject" else None
    zt = torch.from_numpy(z.ravel()).cuda() if z is not None else None
    mode = B.RNG_INJECT if z is not None else B.RNG_PHILOX
    with Plan(desc) as plan:
        slots = B.lib().mcre_irc_presim_slots(plan)
        rc, s_full, p_full, m_full, _ = _run_presim(plan, desc, n, chunk, _rng(mode, n, zt))
        B.check(rc)
        full = _spill(s_full, t, n)
        pf = p_full.cpu().numpy()
        parts = []
        for b, m in ((0, 4 * chunk), (4 * chunk, n - 4 * chunk), (0, 2 * chunk), (2 * chunk, 2 * chunk)):
            rc, s, p, mo, _ = _run_presim(plan, desc, m, chunk, _rng(mode, n, zt), begin=b)
            B.check(rc)
            sp = _spill(s, t, m)
            for key in ("x", "N", "W"):
                assert np.array_equal(sp[key], full[key][..., b:b + m]), f"shard [{b}, {b + m}) {key}"
            c0, nc = b // chunk, (m + chunk - 1) // chunk
            assert np.array_equal(p.cpu().numpy()[:nc * slots], pf[c0 * slots:(c0 + nc) * slots]), f"partial [{b}, {b + m})"
            parts.append(mo.cpu().numpy())
    m_full = m_full.cpu().numpy()
    assert np.array_equal(RT.tree_sum(parts[:2]), m_full)
    assert np.array_equal(RT.tree_sum([parts[2], parts[3], parts[1]]), m_full)


# ---- 6. device solve and patch -------------------------------------------------------------------------------------------
def _moments_from_samples(u, Y, nu):
    """Moment row [5 + 3 nu] of samples u [m] with right-hand sides Y [n_units][m], in float64 via fsum."""
    row = np.zeros(5 + 3 * nu)
    for p in range(5):
        row[p] = math.fsum(u ** p)
    for j, y in enumerate(Y):
        for i in range(3):
            row[5 + 3 * j + i] = math.fsum(y * u ** i)
    return row


def _mp_solve(row, j):
    mpmath.mp.dps = 50
    G = mpmath.matrix([[mpmath.mpf(row[a + b]) for b in range(3)] for a in range(3)])
    rhs = mpmath.matrix([mpmath.mpf(row[5 + 3 * j + i]) for i in range(3)])
    return np.array([float(c) for c in mpmath.lu_solve(G, rhs)])


def _gram(row):
    return np.array([[row[a + b] for b in range(3)] for a in range(3)])


def _cut_ratio(row):
    """The host rule's rank measure (mcre/lsm.py:solve_normal_equations): smallest over largest singular value of the
    Gram matrix equilibrated by its diagonal.  Full rank when it exceeds 1e-10."""
    G = _gram(row)
    d = np.sqrt(np.diag(G))
    sv = np.linalg.svd(G / np.outer(d, d), compute_uv=False)
    return sv[2] / sv[0]


def _truncated(row, j):
    """Minimum-norm solution with the smallest singular direction of the Gram matrix dropped (the rank-2 branch)."""
    u, sv, vt = np.linalg.svd(_gram(row))
    return (vt[:2].T * (1.0 / sv[:2])) @ (u[:, :2].T @ row[5 + 3 * j:8 + 3 * j])


def _near_cut_samples(g, m, target):
    """u = 1 + eps {-1, 0, 1}: three clusters whose equilibrated Gram matrix has a rank measure ~ eps^4; eps is tuned
    until the measure is target."""
    pattern = g.choice([-1.0, 0.0, 1.0], m)
    pattern[:3] = [-1.0, 0.0, 1.0]
    eps = 1e-2
    for _ in range(6):
        u = 1.0 + eps * pattern
        eps *= (target / _cut_ratio(_moments_from_samples(u, [], 1))) ** 0.25
    return 1.0 + eps * pattern


# unit -> netting-set row layouts of the coef_sum check (n_sets = 3): sets holding two and three units (so that the
# order and the accumulation of the sum matter), an empty set, a unit outside every set (-1) and one past n_sets
SET_LAYOUTS = {1: [[2], [-1]], 2: [[2, 2], [0, -1]], 3: [[2, 2, 2], [2, -1, 2], [0, 5, 0]],
               4: [[2, 2, 2, 5], [0, -1, 0, 5], [2, 0, 2, 2]]}
# fits on the near-cut dates, relative to the largest fitted value.  Above the cut the elimination solves a system of
# condition ~3e9: coefficients carry ~eps * 3e9 ~ 7e-7 of relative error, and the host's own fit is up to 1.2e-7 away
# from mpmath on these samples.  Below it the pseudo-inverse drops an eigenvalue ~3e-11 of the largest and the kept
# ones are well separated.  A branch switch moves the fit by more than 6e-4 (asserted with a margin of 100).
FIT_TOL = {"near_cut_above": 1e-6, "near_cut_below": 1e-9}


@pytest.mark.parametrize("n_units", [1, 2, 3, 4])
@pytest.mark.parametrize("n_reg", [1, 64, 65, 200])
def test_irc_solve_matches_mpmath_and_host_rule(n_units, n_reg):
    """Dates: rank 1 (t = 0: every u equal), well-conditioned full rank, full rank with a rank measure of 3e-10 (just
    above the 1e-10 cut: the elimination branch on an ill-conditioned system), rank measure 3e-11 (just below: the
    pseudo-inverse branch), and u scaled by 1e-6 and 1e6.  On both near-cut dates the rank-3 and the rank-2 fits differ
    by far more than the tolerance, so a cut moved past either date fails."""
    be, desc, keep, info = _many_dates_plan(n_reg, n_units)
    nu = 1 if n_units <= 1 else (2 if n_units <= 2 else 4)
    g = np.random.default_rng(n_reg * 10 + n_units)
    kinds_all = ("rank1", "full", "near_cut_below", "near_cut_above", "scale_small", "scale_big")
    rows, kinds, supports = [], [], []
    for k in range(n_reg):
        kind = kinds_all[k % 6] if n_reg > 1 else "rank1"
        m = 64
        if kind == "rank1":
            u = np.zeros(m)
        elif kind == "near_cut_below":
            u = _near_cut_samples(g, m, 3e-11)
        elif kind == "near_cut_above":
            u = _near_cut_samples(g, m, 3e-10)
        else:
            u = g.standard_normal(m) * {"full": 1.0, "scale_small": 1e-6, "scale_big": 1e6}[kind]
        Y = [np.sin(3.0 * u / (np.abs(u).max() + 1e-300)) * (j + 1) + 0.5 * g.standard_normal(m) for j in range(n_units)]
        row = _moments_from_samples(u, Y, nu)
        if kind == "near_cut_below":
            assert 1e-11 <= _cut_ratio(row) <= 6e-11, _cut_ratio(row)
        elif kind == "near_cut_above":
            assert 1.5e-10 <= _cut_ratio(row) <= 1e-9, _cut_ratio(row)
        rows.append(row)
        kinds.append(kind)
        supports.append(np.unique(u))
    mom = np.array(rows)
    d_mom = torch.from_numpy(mom.ravel()).cuda()
    n_sets = 3
    results = []
    with Plan(desc) as plan:
        for layout in SET_LAYOUTS[n_units]:
            cu = _nan(n_units * n_reg * 3)
            cs = _nan(n_reg * n_sets * 3)
            s_arr, s_ptr = B.as_ip(np.array(layout, dtype=np.int32))
            B.check(B.lib().mcre_irc_solve_coefficients(plan, d_mom.data_ptr(), s_ptr, n_sets, cu.data_ptr(),
                                                        cs.data_ptr(), RT.stream_ptr()))
            torch.cuda.synchronize()
            results.append((layout, cu.cpu().numpy().reshape(n_units, n_reg, 3), cs.cpu().numpy().reshape(n_reg, n_sets, 3)))
    cu = results[0][1]
    G = mom[:, [[0, 1, 2], [1, 2, 3], [2, 3, 4]]]
    for j in range(n_units):
        host = solve_normal_equations_batch(G, mom[:, 5 + 3 * j:8 + 3 * j])
        for k in range(n_reg):
            sup = supports[k]

            def fit(c):
                return c[0] + sup * (c[1] + sup * c[2])
            fit_d, fit_h = fit(cu[j, k]), fit(host[k])
            scale = np.abs(fit_h).max() + 1e-300
            tol = FIT_TOL.get(kinds[k], 1e-12)
            assert np.abs(fit_d - fit_h).max() <= tol * scale, (j, k, kinds[k], cu[j, k], host[k])
            if kinds[k] in ("full", "near_cut_above"):
                want = _mp_solve(mom[k], j)
                if kinds[k] == "full":
                    assert np.all(np.abs(cu[j, k] - want) <= 1e-12 * np.abs(want).max()), (j, k, cu[j, k], want)
                else:
                    assert np.abs(fit_d - fit(want)).max() <= tol * scale, (j, k, cu[j, k], want)
            if kinds[k].startswith("near_cut"):
                gap = np.abs(fit(_mp_solve(mom[k], j)) - fit(_truncated(mom[k], j))).max()
                assert gap > 100.0 * FIT_TOL[kinds[k]] * scale, (j, k, kinds[k], gap)
    for layout, cu_l, cs in results:
        assert np.array_equal(cu_l, cu), layout
        want = np.zeros((n_reg, n_sets, 3))           # unit order, from +0.0, units outside [0, n_sets) skipped
        for j in range(n_units):
            if 0 <= layout[j] < n_sets:
                want[:, layout[j]] = want[:, layout[j]] + cu[j]
        assert np.array_equal(cs, want), layout
        for r in range(n_sets):
            if r not in layout:
                assert np.all(cs[:, r] == 0.0) and not np.signbit(cs[:, r]).any(), (layout, r)


def _main_book(n_sets, cva_only=False, bermudan=False):
    ns = cases.Namespace()
    tl = np.linspace(0.0, 2.0, 9)
    if cva_only:
        vas = _vasicek(ns, sigma=0.02)
        cir = ns.CIRPPModel(0., "GM", cases.HAZARDS, 0.1, 0.01, 0.02, 0.0001)
        model = ns.ModelConfig([vas, cir], inter_asset_correlation_matrix=np.array([0.3]))
        sets = [ns.NettingSet(name="s0", products=_units(ns, 1, 2.0), counterparty_id="GM")]
        metrics = [ns.CVAMetric("GM", 0.4)]
    else:
        model = _vasicek(ns)
        sets = []
        for s in range(n_sets):
            prods = _units(ns, 2, 2.0 + 0.5 * s)[s % 2:s % 2 + 1]
            if bermudan and s == 0:
                swap = ns.InterestRateSwap(0.0, 2.5, 1.0, 0.03, 0.25, 0.25, ns.IRSType.PAYER, asset_id="irs")
                prods = prods + [ns.BermudanOption(swap, [0.5, 1.0, 1.5], 0.0, ns.OptionType.CALL)]
            sets.append(ns.NettingSet(name=f"s{s}", products=prods))
        metrics = [ns.PVMetric(), ns.EPEMetric(), ns.ENEMetric()]
    rm = ns.RiskMetrics(metrics, exposure_timeline=tl)
    sc = ns.SimulationController(sets, model, rm, 256, 256, 2, ns.SimulationScheme.EULER)
    return sc


@pytest.mark.parametrize("case", ["value_1", "value_2", "value_3", "general_bermudan", "general_forced", "cva_only"])
def test_device_patch_is_bit_identical_to_host_patch(case):
    """mcre_irc_set_coefficients_device against mcre_irc_set_coefficients: the same random nonzero coefficients on
    every exposure date (the last included) patched both ways into twin plans; one mcre_irc_mainsim each with the
    same draws must give bit-identical accumulators and shifts.  Covers the lean value kernel (1 - 3 sets), the
    general template with exercise units (a set with a Bermudan option), the general template without them and the
    CVA-only kernel's raw-basis event records.  Value-only plans of linear products reach the general template only
    under MCRE_IRC_GENERIC=1, which the library reads once per process, so that case runs in a child process."""
    if case == "general_forced":
        here = os.path.dirname(os.path.abspath(__file__))
        code = ("import importlib, sys; sys.path[:0] = [%r, %r]; importlib.import_module('montecarlo-risk-engine_b200'); "
                "import test_irc_presim_kernels_gpu as T; T._patch_check('value_2')" % (here, os.path.dirname(here)))
        out = subprocess.run([sys.executable, "-s", "-c", code], env=dict(os.environ, MCRE_IRC_GENERIC="1"),
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
        return
    _patch_check(case)


def _patch_check(case):
    n_sets = int(case.split("_")[1]) if case.startswith("value") else 1
    sc = _main_book(n_sets, cva_only=case == "cva_only", bermudan=case == "general_bermudan")
    be = IrcBackend(sc)
    idxs = list(range(len(sc.netting_sets)))
    desc, keep, info = be.lower(idxs, [])
    n_expo, ns_ = info["n_expo"], len(idxs)
    g = np.random.default_rng(17 + n_sets)
    coef = g.standard_normal((n_expo, ns_, 3)) * np.array([1e-2, 5e-3, 1e-3]) + 1e-4
    n = 2000
    L = B.lib()
    outs = []
    for how in ("host", "device"):
        with Plan(desc) as plan:
            if how == "host":
                arr, ptr = B.as_dp(coef)
                B.check(L.mcre_irc_set_coefficients(plan, ptr, RT.stream_ptr()))
            else:
                d_coef = torch.from_numpy(coef.ravel().copy()).cuda()
                B.check(L.mcre_irc_set_coefficients_device(plan, d_coef.data_ptr(), RT.stream_ptr()))
            slots = L.mcre_irc_main_slots(plan)
            acc, shift = _nan(slots), _nan(slots)
            partial = _nan(L.mcre_irc_partial_bytes(plan, n, 256, 0) // 8 + 1)
            spill = _nan(max(ns_ * info["n_metric"] * n, 1))
            B.check(L.mcre_irc_mainsim(plan, C.byref(_rng(B.RNG_PHILOX, n, seed=43)), C.byref(B.Shard(0, n, 256)),
                                       partial.data_ptr(), acc.data_ptr(), shift.data_ptr(), spill.data_ptr(),
                                       RT.stream_ptr()))
            torch.cuda.synchronize()
            outs.append((acc.cpu().numpy(), shift.cpu().numpy()))
    (a_h, s_h), (a_d, s_d) = outs
    assert np.any(a_h != 0.0) and np.all(np.isfinite(a_h))
    assert np.array_equal(a_h, a_d, equal_nan=True), np.argwhere(a_h != a_d)[:5]
    assert np.array_equal(s_h, s_d, equal_nan=True)


# ---- 7. empty shards and plans that do not fit ---------------------------------------------------------------------------
@pytest.mark.parametrize("differentiate", [False, True])
def test_presim_empty_shard_writes_zero_moments(differentiate):
    """A rank without pre-simulation paths contributes zero moments (like the csrc/lsm.cu moment entries): callers
    need not pre-zero the buffers they all-reduce."""
    be, desc, keep, info = _forward_plan("vas", "EULER", 2, 2, differentiate=differentiate)
    with Plan(desc) as plan:
        rc, scratch, partial, mom, tmom = _run_presim(plan, desc, 0, 256, _rng(B.RNG_PHILOX, 1024), begin=1024)
        B.check(rc)
        assert mom.numel() == B.lib().mcre_irc_presim_slots(plan) and np.all(mom.cpu().numpy() == 0.0)
        if differentiate:
            assert tmom.numel() == B.lib().mcre_irc_presim_tangent_slots(plan) and np.all(tmom.cpu().numpy() == 0.0)


@pytest.mark.parametrize("n_units,differentiate", [(4, False), (1, True)])
def test_presim_refuses_a_plan_with_too_many_regression_dates(n_units, differentiate):
    """Value moments at NU = 4 need (17 n_reg + 272) doubles of shared memory, tangent moments (9 n_reg + 144): 20 dates
    past the device's per-block opt-in limit (about 1,700 and 3,200 dates at 227 KB) the entry must return -3 naming
    the regression dates, before any kernel is launched, and leave no error behind for the next call.  (The tangent
    plan's value moments, 8 n_reg + 128 doubles at NU = 1, still fit: the refusal comes from the tangent kernel.)"""
    per_date, fixed = (9, 144) if differentiate else (17, 272)
    n_reg = (_smem_optin() // 8 - fixed) // per_date + 20
    smem = (per_date * n_reg + fixed) * 8
    assert smem > _smem_optin()
    if differentiate:
        assert (8 * n_reg + 128) * 8 <= _smem_optin()
    be, desc, keep, info = _many_dates_plan(n_reg, n_units, differentiate=differentiate)
    L = B.lib()
    n = 300
    with Plan(desc) as plan:
        before = B.launch_count()
        rc, scratch, partial, mom, tmom = _run_presim(plan, desc, n, 256, _rng(B.RNG_PHILOX, n))
        msg = L.mcre_last_error().decode()
        assert rc == -3, (rc, msg)
        assert "regression dates" in msg, msg
        assert B.launch_count() == before
        assert torch.isnan(scratch).all() and torch.isnan(mom).all()
    # the next, valid call and the next torch operation succeed
    be, desc, keep, info = _forward_plan("vas", "EULER", 1, 1)
    with Plan(desc) as plan:
        rc, scratch, partial, mom, _ = _run_presim(plan, desc, 300, 256, _rng(B.RNG_PHILOX, 300))
    assert rc == 0, L.mcre_last_error().decode()
    assert np.all(np.isfinite(mom.cpu().numpy()))
    assert float(torch.ones(4, device="cuda").sum().item()) == 4.0
