"""PV sensitivities of gas storages on multi-asset Black-Scholes models, under EULER, and netted with equity products
(mcre/storage.py through csrc/storage.cu:storage_main_kernel<NT> with the storage's own tangent slots, and the equity
launches with tangents for the other products of a set).

There are no reference goldens of these sensitivities.  The arbiter is the oracle's forward-mode duals (oracle/risk.py,
oracle/storage.py: hard decisions on values, cashflows differentiated through the spot and the numeraire), anchored once
to the reference's autograd: a one-asset BlackScholesMulti carrying the storage_bs_greeks contract reproduces that golden.
The oracle values a set of storages next to other products only without sensitivities; the gradient of such a set is the
sum of the gradients of its storages and of its other products on the same paths, which the oracle gives in two runs
(_oracle_reference).  Values must not move when sensitivities are asked for."""
import ctypes as C

import numpy as np
import pytest
import torch

import cases
import parity_helpers as helpers

pytestmark = pytest.mark.gpu


# ---- scenarios without a golden (run through the helpers by a temporary GOLDEN_CASES entry) -------------------------
def storage_on_multi(ns_module):
    """A storage on the second asset of the three-asset Black-Scholes model of storage_mixed_book: its row of the joint
    Cholesky factor has off-diagonal entries."""
    m = ns_module
    model, _, _, _ = cases.storage_mixed_book(ns_module)
    st = cases.book_storage(m, 0, "asset_1", 0.5, 18.0, 0.05, 6, 2.0, 0.10, 0.08)
    st.name = "storage"
    return model, [m.NettingSet(name="storage", products=[st])], [m.PVMetric()], None


def storage_on_config(ns_module):
    """A ModelConfig of two Black-Scholes models with different rates, the storage on the one that is not the
    numeraire: the discount factors carry the other model's rate."""
    m = ns_module
    power = m.BlackScholesModel(0.0, 100.0, 0.03, 0.2, asset_id="power")
    gas = m.BlackScholesModel(0.0, 24.0, 0.05, 0.35, asset_id="gas")
    model = m.ModelConfig(models=[power, gas], inter_asset_correlation_matrix=[np.full((1, 1), 0.4)])
    st = cases.book_storage(m, 0, "gas", 0.5, 18.0, 0.05, 6, 2.0, 0.10, 0.08)
    st.name = "storage"
    return model, [m.NettingSet(name="storage", products=[st])], [m.PVMetric()], None


def storage_bs_as_multi(ns_module):
    """The storage_bs_greeks contract on a one-asset BlackScholesMulti: parameters (spot, volatility, rate) in the
    reference's order of the BlackScholesModel of that golden."""
    m = ns_module
    _, sets, metrics, _ = cases.storage_small(ns_module)
    model = m.BlackScholesMulti(calibration_date=0.0, rate=0.03, asset_ids=["gas"], spots=[100.0], volatilities=[0.2],
                                correlation_matrix=np.array([[1.0]]))
    return model, sets, metrics, None


def storage_mixed_book_split(ns_module):
    """storage_mixed_book with a second American and a second Asian option: four path-dependent products, more than one
    launch with tangents tracks (mcre/equity.py:eq_ntrk), so the equity part of the set is split over launches."""
    m = ns_module
    model, sets, metrics, _ = cases.storage_mixed_book(ns_module)
    extra = [m.AmericanOption(underlying=m.Equity("asset_0"), maturity=1.0, num_exercise_dates=4, strike=100.0,
                              option_type=m.OptionType.PUT, asset_id="asset_0"),
             m.AsianOption(0.0, 1.0, 110.0, 4, m.OptionType.CALL, asset_id="asset_2")]
    return model, [m.NettingSet(name="split_book", products=sets[0].products + extra)], metrics, None


_SMALL = dict(n_main=1024, n_pre=1024, differentiate=True)
NEW_CASES = {
    "storage_bsm_greeks": (storage_on_multi, dict(), dict(_SMALL, num_steps=1, scheme="ANALYTICAL")),
    "storage_bsm_greeks_euler": (storage_on_multi, dict(), dict(_SMALL, num_steps=2, scheme="EULER")),
    "storage_bs_greeks_euler": (cases.storage_small, dict(), dict(n_main=256, n_pre=256, num_steps=2, scheme="EULER",
                                                                  differentiate=True)),
    "storage_config_greeks": (storage_on_config, dict(), dict(_SMALL, num_steps=1, scheme="ANALYTICAL")),
    "storage_config_greeks_euler": (storage_on_config, dict(), dict(_SMALL, num_steps=2, scheme="EULER")),
    "storage_bs_as_multi_greeks": (storage_bs_as_multi, dict(), dict(n_main=256, n_pre=256, num_steps=1,
                                                                     scheme="ANALYTICAL", differentiate=True)),
    "storage_mixed_book_split": (storage_mixed_book_split, dict(), dict(n_main=1000, n_pre=1000, num_steps=1,
                                                                        scheme="ANALYTICAL", differentiate=True)),
}
ORACLE_CASES = ["storage_bsm_greeks", "storage_bsm_greeks_euler", "storage_bs_greeks_euler", "storage_config_greeks",
                "storage_config_greeks_euler", "storage_mixed_book", "storage_mixed_book_split"]


@pytest.fixture
def register(monkeypatch):
    def add(name):
        if name in NEW_CASES:
            monkeypatch.setitem(cases.GOLDEN_CASES, name, NEW_CASES[name])
    return add


def _grads(res, s, m):
    return np.array([0.0 if g is None else float(g) for g in res.get_derivatives(s, m)[0]])


def _as_array(row):
    return np.array([0.0 if w is None else float(w) for w in row])


def _oracle_reference(name, draws):
    """-> [set][metric] (value, mc error, gradient [P]) of the oracle with sensitivities.  A book of storages alone is one
    oracle run.  A set that nets storages with other products is valued by one run without sensitivities; its gradient
    (PV is linear in the per-path cashflows) is the sum of two runs with sensitivities, one on the storages and one on the
    other products, on the paths of the whole book: each run gets the other part's modelling dates as (PV-only, hence
    inert) exposure dates, so that both simulate the whole book's timeline with the same draws.  Their values must add
    up to the whole book's, which the caller checks."""
    from oracle import risk
    ns, model, sets, metrics, tl, rkw = helpers.build(name, differentiate=True)
    pre = main = None
    if draws == "torch":
        pre, main = helpers.reference_draws(model, sets, tl, metrics, rkw)
    kw = dict(draws_pre=pre, draws_main=main, degree=rkw.get("degree", 2) + 1)
    args = (rkw["n_main"], rkw["n_pre"], rkw["num_steps"], rkw["scheme"])
    prods = [p for s in sets for p in s.products]
    storage = [risk.kind(p) == "Storage" for p in prods]
    if all(storage):
        out = risk.run(model, sets, metrics, tl, *args, differentiate=True, **kw)
        return [[(*r[mi][0], _as_array(gs[mi][0])) for mi in range(len(r))]
                for r, gs in zip(out["results"], out["grads"])], None
    whole = risk.run(model, sets, metrics, tl, *args, differentiate=False, **kw)
    parts = []
    for keep in (lambda p: risk.kind(p) == "Storage", lambda p: risk.kind(p) != "Storage"):
        sub = [ns.NettingSet(name=s.name, products=[p for p in s.products if keep(p)]) for s in sets]
        dates = sorted({float(t) for p in prods if not keep(p) for t in risk.modeling_timeline(p)})
        parts.append(risk.run(model, sub, metrics, dates, *args, differentiate=True, **kw))
    ref = [[(*r[mi][0], sum(_as_array(part["grads"][si][mi][0]) for part in parts)) for mi in range(len(r))]
           for si, r in enumerate(whole["results"])]
    part_values = [[sum(part["results"][si][mi][0][0] for part in parts) for mi in range(len(r))]
                   for si, r in enumerate(whole["results"])]
    return ref, part_values


@pytest.mark.parametrize("draws", ["torch", "philox"])
@pytest.mark.parametrize("name", ORACLE_CASES)
def test_storage_greeks_match_oracle_duals_and_values_do_not_move(name, draws, register):
    register(name)
    res, _ = helpers.run_cuda(name, draws=draws, differentiate=True)
    res0, _ = helpers.run_cuda(name, draws=draws, differentiate=False)
    flat, flat0 = helpers.flatten_results(res), helpers.flatten_results(res0)
    for key, (v, e) in flat0.items():
        helpers.assert_close(flat[key][0], v, 1e-12, 0.0, f"{name} {draws} {key} value with / without sensitivities")
        helpers.assert_close(flat[key][1], e, 1e-12, 0.0, f"{name} {draws} {key} mc error with / without sensitivities")
    if name == "storage_mixed_book" and draws == "torch":
        gold = helpers.load_golden(name)
        for key, v in gold["values"].items():
            helpers.assert_close(flat[key][0], v, 1e-9, 1e-9, f"{name} {key} against the reference")
    ref, part_values = _oracle_reference(name, draws)
    for si, s in enumerate(res.get_netting_set_names()):
        for mi, m in enumerate(res.get_metric_names()):
            v, e, want = ref[si][mi]
            if part_values is not None:      # the two partial runs simulated the whole book's paths
                helpers.assert_close([part_values[si][mi]], [v], 1e-12, 0.0, f"{name} {draws} {s}|{m} sum of the parts")
            got_v, got_e = flat[f"{s}|{m}"]
            helpers.assert_close(got_v, [v], 1e-8, 0.0, f"{name} {draws} {s}|{m} value against the oracle")
            # (a nearly deterministic PV has a standard error of rounding size: 1e-12 of the value on top)
            helpers.assert_close(got_e, [e], 1e-8, 1e-12 * abs(v), f"{name} {draws} {s}|{m} mc error against the oracle")
            assert np.any(want != 0.0)
            helpers.assert_close(_grads(res, s, m), want, 1e-8, 1e-8 * float(np.max(np.abs(want))),
                                 f"{name} {draws} {s}|{m} sensitivities against the oracle")


def test_one_asset_multi_model_reproduces_the_reference_storage_greeks(register):
    """storage_bs_greeks (the reference's autograd) on a one-asset BlackScholesMulti with the reference's draws.  The
    multi-asset step rounds (r - sigma^2 / 2) dt where the single-asset one rounds r dt - sigma^2 dt / 2: 1e-8."""
    register("storage_bs_as_multi_greeks")
    gold = helpers.load_golden("storage_bs_greeks")
    res, _ = helpers.run_cuda("storage_bs_as_multi_greeks", draws="torch")
    flat = helpers.flatten_results(res)
    helpers.assert_close(flat["storage|pv"][0], gold["values"]["storage|pv"], 1e-8, 0.0, "pv")
    helpers.assert_close(flat["storage|pv"][1], gold["errors"]["storage|pv"], 1e-8, 0.0, "pv error")
    want = np.array(gold["derivatives"]["storage|pv"][0], dtype=float)
    helpers.assert_close(_grads(res, "storage", "pv"), want, 1e-8, 1e-8 * float(np.max(np.abs(want))), "derivatives")


def test_sharded_tangents_are_bit_identical_to_one_full_range(register, monkeypatch):
    """mcre_storage_mainsim with tangents on the path ranges [0, n/2) and [n/2, n) of one GPU: the concatenated per-path
    cashflows and tangents are bit-identical to those of one full-range call, and so is the PV gradient of their
    fixed-order chunk sums to the run's."""
    from mcre import binding as B
    from mcre.storage import tangent_slots
    name = "storage_bsm_greeks"
    register(name)
    L = B.lib()
    orig = L.mcre_storage_mainsim
    seen = {}

    def wrapped(plan, rng, shard, coef, init, cfs, final, tan, coef_e, expo, stream):
        rc = orig(plan, rng, shard, coef, init, cfs, final, tan, coef_e, expo, stream)
        sh = shard._obj
        n, half, nt = sh.n_paths, sh.n_paths // 2, 3
        outs = []
        for begin, count in ((sh.path_begin, n), (sh.path_begin, half), (sh.path_begin + half, n - half)):
            c = torch.zeros(count, dtype=torch.float64, device="cuda")
            t = torch.zeros((nt, count), dtype=torch.float64, device="cuda")
            B.check(orig(plan, rng, C.byref(B.Shard(begin, count, sh.chunk_paths)), coef, init, c.data_ptr(), None,
                         t.data_ptr(), None, None, stream))
            outs.append((c, t))
        torch.cuda.synchronize()
        seen.update(full=outs[0], halves=outs[1:], chunk=sh.chunk_paths)
        return rc
    monkeypatch.setattr(L, "mcre_storage_mainsim", wrapped)
    res, sc = helpers.run_cuda(name, draws="philox")
    (c, t), ((ca, ta), (cb, tb)) = seen["full"], seen["halves"]
    assert torch.equal(torch.cat([ca, cb]), c) and torch.equal(torch.cat([ta, tb], dim=1), t)
    n = c.shape[0]
    chunk = seen["chunk"]
    n_chunks = (n + chunk - 1) // chunk
    partial = torch.empty(n_chunks * 6 + 1, dtype=torch.float64, device="cuda")
    out_t = torch.zeros(6, dtype=torch.float64, device="cuda")
    zero = torch.zeros(3, dtype=torch.float64, device="cuda")
    B.check(L.mcre_sum_stats(torch.cat([ta, tb], dim=1).contiguous().data_ptr(), n, 3, chunk, zero.data_ptr(), 0,
                             partial.data_ptr(), out_t.data_ptr(), 0))
    sums = out_t.cpu().numpy().reshape(3, 2)[:, 0] / n
    slots, _ = tangent_slots(sc.model, "asset_1")
    got = _grads(res, "storage", "pv")
    assert list(got[slots]) == list(sums)
    assert np.all(np.delete(got, slots) == 0.0)


def test_pathwise_greeks_agree_with_central_differences(register):
    """BlackScholesMulti / ANALYTICAL, native Philox, 2^16 paths in both passes: d/d spot of the storage's asset and
    d/d rate against central differences of the PV on the same streams (the policy re-fitted on the bumped
    pre-simulation), at relative bumps of 1e-4 and 1e-3: 1e-2 relative.  (Measured on a B200: spot to 1e-12, rate to
    2e-7; at a bump of 1e-2 the rate difference picks up decision flips and changes sign.)
    The volatility is not compared: its differences are dominated by the decision flips that the pathwise tangent leaves
    out by design, and do not converge.  Measured on a B200 for this case: pathwise 0.2811, central differences 1.0438,
    0.8788 and 0.3446 at relative bumps of 1e-4, 1e-3 and 1e-2."""
    name = "storage_bsm_greeks"
    register(name)
    n = 1 << 16
    res, sc = helpers.run_cuda(name, draws="philox", n_main=n, n_pre=n)
    got = _grads(res, "storage", "pv")

    def pv(k, v):
        ns, model, sets, metrics, tl, rkw = helpers.build(name, n_main=n, n_pre=n, differentiate=False)
        model.model_params[k] = torch.tensor(v, dtype=torch.float64)
        sc = ns.SimulationController(sets, model, ns.RiskMetrics(metrics), n, n, rkw["num_steps"],
                                     getattr(ns.SimulationScheme, rkw["scheme"]), False)
        return float(sc.run_simulation().get_results("storage", "pv")[0])
    for k, label in ((1, "spot"), (6, "rate")):
        v0 = float(sc.model.model_params[k])
        for rel in (1e-4, 1e-3):
            h = rel * abs(v0)
            fd = (pv(k, v0 + h) - pv(k, v0 - h)) / (2 * h)
            assert abs(got[k] - fd) <= 1e-2 * abs(fd), f"d/d {label}: pathwise {got[k]} vs central difference {fd} (h {h})"
