"""Sensitivities of exposure metrics (CVA, EPE, ENE, CE, EEPE, PFE) of netting sets with equity exercise products:
AmericanOption, BermudanOption and FlexiCall on Black-Scholes (single and multi-asset) and Heston.

The exposure of an exercise product is its continuation value (c0 + u (c1 + u c2)) / N(t) for the state (rights left)
the path is in.  Its pathwise tangents need the tangents of the regression coefficients: a tangent pre-simulation spill
(mcre_eq_presim_tangents -> mcre_lsm_prepare_equity_tangents), the tangent backward induction for 1..6 rights
(mcre_lsm_step_states_tangents + regression_tangents per state) and the dual branch of exposure type 3 in the fused
kernel (mcre_eq_set_exercise_exposure_coef_tangents).

There are no reference goldens of these sensitivities.  The arbiter is the oracle's forward-mode duals (oracle/risk.py:
lstsq_dual per state, hard exercise decisions on values, state-selected dual coefficients), which are pinned to the
reference's autograd on the neighbouring cases bs_proxy_greeks_mixed, equity_cva_greeks, heston_exposure_greeks_* and
the rate Bermudan's tangent pass.  The values of the cases with a golden are checked against the reference's outputs."""
import numpy as np
import pytest
import torch

import cases
import parity_helpers as helpers

pytestmark = pytest.mark.gpu


# ---- scenarios without a golden (run through the helpers by a temporary GOLDEN_CASES entry) -------------------------
def bs_american_bermudan(ns_module):
    """An American put and a Bermudan call on one Black-Scholes asset in a thresholded and an MPoR-collateralised
    netting set, every exposure metric with a fused tangent sum (one launch)."""
    m = ns_module
    model = m.BlackScholesModel(0.0, 100.0, 0.03, 0.25)
    put = m.AmericanOption(m.Equity("id"), 1.5, 12, 100.0, m.OptionType.PUT)
    call = m.BermudanOption(m.Equity("id"), [0.25, 0.5, 0.75, 1.0, 1.25], 95.0, m.OptionType.CALL)
    sets = [m.NettingSet(name="thresholded", products=[put], threshold=1.0),
            m.NettingSet(name="collateralised", products=[call], margin_period_of_risk=0.25, threshold=0.5)]
    return model, sets, [m.CEMetric(), m.EPEMetric(), m.ENEMetric(), m.EEPEMetric()], np.linspace(0.0, 1.5, 7)


def heston_american(ns_module):
    """An American put under Heston: exposure tangents with respect to all seven model parameters."""
    m = ns_module
    model = m.HestonModel(0.0, 100.0, 0.03, 0.4, -0.7, 2.0, 0.04, 0.04)
    put = m.AmericanOption(m.Equity("id"), 1.0, 8, 105.0, m.OptionType.PUT)
    return model, [m.NettingSet(name="heston_put", products=[put])], [m.EPEMetric(), m.ENEMetric()], np.linspace(0.0, 1.0, 5)


def hybrid_american(ns_module):
    """Three-model hybrid (Black-Scholes numeraire, Vasicek, CIR++ counterparty) with an American option next to a bond
    and a swap in one netting set: CVA + EPE through HybridBackend."""
    m = ns_module
    cp = "cp"
    eq = m.BlackScholesModel(calibration_date=0.0, spot=100.0, rate=0.03, sigma=0.22, asset_id="equity")
    rates = m.VasicekModel(calibration_date=0.0, rate=0.03, mean=0.03, mean_reversion_speed=1.0, volatility=0.01,
                           asset_id="rates")
    credit = m.CIRPPModel(calibration_date=0.0, asset_id=cp, hazard_rates=cases.HAZARDS, kappa=0.10, theta=0.01,
                          volatility=0.02, y0=0.0001, deterministic=True)
    model = m.ModelConfig(models=[eq, rates, credit], inter_asset_correlation_matrix=[np.array([r]) for r in (0.25, 0.0, 0.0)])
    prods = [m.AmericanOption(underlying=m.Equity("equity"), maturity=1.5, num_exercise_dates=6, strike=100.0,
                              option_type=m.OptionType.PUT, asset_id="equity"),
             m.Bond(startdate=0.0, maturity=2.0, notional=2.0, tenor=0.5, pays_notional=True, fixed_rate=0.025,
                    asset_id="rates"),
             m.InterestRateSwap(startdate=0.0, enddate=2.0, notional=25.0, fixed_rate=0.03, tenor_fixed=0.5,
                                tenor_float=0.25, irs_type=m.IRSType.PAYER, asset_id="rates")]
    sets = [m.NettingSet(name="hybrid_ns", products=prods, counterparty_id=cp)]
    return model, sets, [m.CVAMetric(counterparty_id=cp, recovery_rate=0.4), m.EPEMetric()], np.linspace(0.0, 2.0, 9)


NEW_CASES = {
    "bs_american_bermudan": (bs_american_bermudan, dict(), dict(n_main=2048, n_pre=2048, num_steps=1, scheme="ANALYTICAL",
                                                               differentiate=True)),
    "heston_american_qe": (heston_american, dict(), dict(n_main=2048, n_pre=2048, num_steps=3, scheme="QE", differentiate=True)),
    "heston_american_euler": (heston_american, dict(), dict(n_main=2048, n_pre=2048, num_steps=3, scheme="EULER",
                                                            differentiate=True)),
    "hybrid_american": (hybrid_american, dict(), dict(n_main=1024, n_pre=1024, num_steps=4, scheme="EULER", differentiate=True)),
}
#: cases with a reference golden (values), all on the EquityCreditGreeks route (per-path duals: PFE, a credit model or
#: a book split over launches); its value run splits the book, the value-only run may evaluate it in one launch
GOLDEN = ["flexicall_exposure", "flexicall_6_rights", "mixed_book_exposure", "equity_cva_exercise"]


@pytest.fixture
def register(monkeypatch):
    def add(name):
        if name in NEW_CASES:
            monkeypatch.setitem(cases.GOLDEN_CASES, name, NEW_CASES[name])
    return add


def _close_values(flat, ref, rtol, what, err_rtol=1e-7):
    for key, (va, ea) in flat.items():
        vb, eb = ref[key]
        scale = max(1.0, float(np.nanmax(np.abs(vb))))
        helpers.assert_close(va, vb, rtol, rtol * scale, f"{what} {key} value")
        helpers.assert_close(ea, eb, err_rtol, 1e-11 * scale, f"{what} {key} mc error")


def _greeks_match_oracle(res, out, what):
    """Every derivative of every metric and evaluation against the oracle's out["grads"] at rtol 1e-6, atol 1e-6 max|want|;
    parameters the oracle does not connect (None) compare as 0.0 (None or 0.0 here, the route's convention)."""
    for si, s in enumerate(res.get_netting_set_names()):
        for mi, m in enumerate(res.get_metric_names()):
            got_rows = res.get_derivatives(s, m)
            for ev, want in enumerate(out["grads"][si][mi]):
                got = np.array([0.0 if g is None else float(g) for g in got_rows[ev]])
                want = np.zeros(len(got)) if want is None else np.array([0.0 if w is None else float(w) for w in want])
                helpers.assert_close(got, want, 1e-6, 1e-6 * max(1.0, float(np.max(np.abs(want)))), f"{what} {s}|{m}[{ev}]")


def _exercise_coefficients(sc):
    prods = [p for ns in sc.netting_sets for p in ns.products if hasattr(p, "num_exercise_rights")]
    return [p.regression_coeffs.clone() for p in prods], [rc.clone() for rc in sc.regression_coeffs]


@pytest.mark.parametrize("name", GOLDEN + list(NEW_CASES))
def test_exercise_exposure_greeks_match_oracle(name, register):
    register(name)
    # injected reference draws: values against the golden (values do not move when sensitivities are asked for)
    res, sc = helpers.run_cuda(name, draws="torch", differentiate=True)
    flat = helpers.flatten_results(res)
    if name in GOLDEN:
        gold = helpers.load_golden(name)
        assert res.get_netting_set_names() == gold["sets"] and res.get_metric_names() == gold["metrics"]
        _close_values(flat, {k: (np.array(v), np.array(gold["errors"][k])) for k, v in gold["values"].items()}, 1e-9, name)
    # values and regression coefficients of the value-only run
    res0, sc0 = helpers.run_cuda(name, draws="torch", differentiate=False)
    flat0 = helpers.flatten_results(res0)
    for key, (v, e) in flat0.items():
        scale = max(1e-300, float(np.max(np.abs(v))))
        helpers.assert_close(flat[key][0], v, 1e-12, 1e-12 * scale, f"{name} {key} value with / without sensitivities")
        helpers.assert_close(flat[key][1], e, 1e-12, 1e-12 * scale, f"{name} {key} mc error with / without sensitivities")
    (pc, sc_c), (pc0, sc_c0) = _exercise_coefficients(sc), _exercise_coefficients(sc0)
    assert pc and all(torch.equal(a, b) for a, b in zip(pc, pc0)), f"{name}: exercise coefficients differ"
    assert all(torch.equal(a, b) for a, b in zip(sc_c, sc_c0)), f"{name}: exposure coefficients differ"
    # sensitivities against the oracle's forward-mode duals on the same draws
    out, _ = helpers.run_oracle(name, draws="torch", differentiate=True)
    _close_values(flat, helpers.oracle_flat(out, res.get_netting_set_names(), res.get_metric_names()), 1e-8,
                  name + " oracle", err_rtol=1e-6)
    _greeks_match_oracle(res, out, name)
    # native Philox
    res, _ = helpers.run_cuda(name, draws="philox", differentiate=True)
    out, _ = helpers.run_oracle(name, draws="philox", differentiate=True)
    _close_values(helpers.flatten_results(res), helpers.oracle_flat(out, res.get_netting_set_names(), res.get_metric_names()),
                  1e-8, name + " philox", err_rtol=1e-6)
    _greeks_match_oracle(res, out, name + " philox")


def _step_inputs(R, nt, n, seed):
    g = torch.Generator().manual_seed(seed)

    def r(*shape, lo=-1.0, hi=1.0):
        return (lo + (hi - lo) * torch.rand(*shape, generator=g, dtype=torch.float64)).cuda()
    d = dict(xk=r(n, lo=60.0, hi=140.0), nk=r(n, lo=1.0, hi=1.1), dxk=r(nt, n), dnk=r(nt, n),
             xi=r(n, lo=60.0, hi=140.0), ni=r(n, lo=1.0, hi=1.1), imm=torch.clamp(r(n, lo=-20.0, hi=30.0), min=0.0),
             dni=r(nt, n), dimm=r(nt, n), value=r(R, n, lo=0.0, hi=20.0).float(), dvalue=r(R, nt, n))
    coef = np.random.default_rng(seed).uniform(-1.0, 1.0, (R, 3)) * np.array([8.0, 3.0, 1.0])
    coef[:, 0] += 6.0 * np.arange(1, R + 1)       # continuation values grow with the rights left
    return d, coef


def _tangent_step(L, R, nt, d, coef, value, dvalue, chunk, entry="states"):
    from mcre import binding as B
    n = d["xk"].shape[0]
    n_chunks = (n + chunk - 1) // chunk
    nv = 4 + 5 * R
    partial = torch.empty(n_chunks * nt * nv + 1, dtype=torch.float64, device="cuda")
    tm = torch.zeros(nt * nv, dtype=torch.float64, device="cuda")
    keep, cptr = B.as_dp(coef.reshape(-1))
    args = (d["xk"].data_ptr(), d["nk"].data_ptr(), d["dxk"].data_ptr(), d["dnk"].data_ptr(), 100.0, 0.05,
            d["xi"].data_ptr(), d["ni"].data_ptr(), d["imm"].data_ptr(), d["dni"].data_ptr(), d["dimm"].data_ptr(), cptr,
            100.0, 0.05, value.data_ptr(), dvalue.data_ptr(), n, chunk, partial.data_ptr(), tm.data_ptr(), 0)
    if entry == "states":
        B.check(L.mcre_lsm_step_states_tangents(R, nt, *args))
    else:
        B.check(L.mcre_lsm_step_tangents(nt, *args))
    torch.cuda.synchronize()
    return tm.cpu().numpy().reshape(nt, nv)


@pytest.mark.parametrize("R", [1, 2, 6])
def test_multi_right_tangent_step_matches_numpy(R):
    """mcre_lsm_step_states_tangents on random inputs after the value step of the same date: the running tangents and
    the tangent moments against a numpy restatement of the update (decisions from the value step's expressions) and of
    the sums at 1e-12; one right is mcre_lsm_step_tangents bit for bit.  9000 paths in 4096-path chunks, and more
    256-path chunks than the kernel's grid cap of sm_count * 4 blocks, so that blocks loop over several chunks."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    for n, chunk in ((9000, 4096), ((4 * sm + 3) * 256 + 17, 256)):
        _check_tangent_step(R, 3, n, chunk)


def _check_tangent_step(R, nt, n, chunk):
    from mcre import binding as B
    L = B.lib()
    d, coef = _step_inputs(R, nt, n, 11 + R)
    value = d["value"].clone()
    n_chunks = (n + chunk - 1) // chunk
    partial = torch.empty(n_chunks * (5 + 3 * R) + 1, dtype=torch.float64, device="cuda")
    mom = torch.zeros(5 + 3 * R, dtype=torch.float64, device="cuda")
    keep, cptr = B.as_dp(coef.reshape(-1))
    B.check(L.mcre_lsm_step_states(R, d["xk"].data_ptr(), d["nk"].data_ptr(), 100.0, 0.05, d["xi"].data_ptr(),
                                   d["ni"].data_ptr(), d["imm"].data_ptr(), cptr, 100.0, 0.05, value.data_ptr(), n, chunk,
                                   partial.data_ptr(), mom.data_ptr(), 0))
    dvalue = d["dvalue"].clone()
    tm = _tangent_step(L, R, nt, d, coef, value, dvalue, chunk)

    h = {k: v.cpu().numpy().astype(np.float64) for k, v in d.items()}
    V = value.cpu().numpy().astype(np.float64)
    ui = (h["xi"] - 100.0) * 0.05
    cont = np.zeros((R + 1, n))
    for s in range(R):
        cont[s + 1] = coef[s, 0] + ui * (coef[s, 1] + ui * coef[s, 2])
    dpay = (h["dimm"] - h["imm"] / h["ni"] * h["dni"]) / h["ni"]               # [nt, n]
    dv_old, dv = h["dvalue"], np.empty_like(h["dvalue"])
    for s in range(R):
        ex = h["imm"] + cont[s] > cont[s + 1]
        prev = dv_old[s - 1] if s > 0 else 0.0
        dv[s] = np.where(ex[None, :], dpay + prev, dv_old[s])
    np.testing.assert_allclose(dvalue.cpu().numpy(), dv, rtol=1e-12, atol=1e-12)
    u = (h["xk"] - 100.0) * 0.05
    du = h["dxk"] * 0.05
    want = np.zeros((nt, 4 + 5 * R))
    for p in range(nt):
        want[p, :4] = [np.sum(u ** m * du[p]) for m in range(4)]
        for s in range(R):
            Y = h["nk"] * V[s]
            dY = h["dnk"][p] * V[s] + h["nk"] * dv[s, p]
            want[p, 4 + 5 * s:9 + 5 * s] = [dY.sum(), (u * dY).sum(), (u * u * dY).sum(), (du[p] * Y).sum(),
                                            (2.0 * u * du[p] * Y).sum()]
    np.testing.assert_allclose(tm, want, rtol=1e-12, atol=1e-12 * np.max(np.abs(want)))
    if R == 1:
        dvalue1 = d["dvalue"].clone()
        tm1 = _tangent_step(L, R, nt, d, coef, value, dvalue1, chunk, entry="single")
        assert np.array_equal(tm1, tm) and torch.equal(dvalue1, dvalue)


def test_basket_exposure_sensitivities_still_raise():
    """Exposure sensitivities of baskets (regression proxies on several assets) are not implemented: they raise."""
    ns = cases.Namespace()
    ids = ["a", "b"]
    model = ns.BlackScholesMulti(calibration_date=0.0, rate=0.03, asset_ids=ids, spots=[100.0, 105.0],
                                 volatilities=[0.2, 0.24], correlation_matrix=np.array([[1.0, 0.35], [0.35, 1.0]]))
    basket = ns.BasketOption(1.0, ids, [0.5, 0.5], 100.0, ns.OptionType.CALL, ns.BasketOptionType.ARITHMETIC, False)
    sc = ns.SimulationController([ns.NettingSet(name="basket", products=[basket])], model,
                                 ns.RiskMetrics([ns.EPEMetric()], exposure_timeline=np.linspace(0.0, 1.0, 5)), 1024, 1024, 1,
                                 ns.SimulationScheme.ANALYTICAL, True)
    with pytest.raises(NotImplementedError):
        sc.run_simulation()
