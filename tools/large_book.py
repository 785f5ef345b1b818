#!/usr/bin/env python
"""Products-per-second of one large mixed netting set on BlackScholesMulti (SURVEY §8f item 2): the shape of the
reference's tests/pv_tests/pv_performance_large_netting_set.py (Europeans, binaries, baskets, Asians, barriers,
Americans, FlexiCalls and gas storages in ONE netting set, PV metric, 1000 paths).
The path-dependent / exercise products exceed what one launch tracks, so the book is split over launches
(mcre/equity.py:_run_split_book).

    python tools/large_book.py [--scale 1.0] [--paths 1000] [--differentiate]
"""
import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402


def build_book(ns, ids, counts):
    cyc = lambda seq, i: seq[i % len(seq)]   # noqa: E731
    prods = []
    for i in range(counts["european"]):
        a = cyc(ids, i)
        prods.append(ns.EuropeanOption(ns.Equity(a), cyc([0.25, 0.5, 0.75, 1.0, 1.5, 2.0, 2.5, 3.0], i),
                                       cyc([80.0, 90.0, 100.0, 110.0, 120.0], i),
                                       ns.OptionType.CALL if i % 2 == 0 else ns.OptionType.PUT, asset_id=a))
    for i in range(counts["binary"]):
        prods.append(ns.BinaryOption(cyc([0.5, 1.0, 1.5, 2.0], i), cyc([90.0, 100.0, 110.0], i), 8.0 + 2.0 * (i % 4),
                                     ns.OptionType.CALL if i % 2 == 0 else ns.OptionType.PUT, asset_id=cyc(ids, i)))
    for i in range(counts["basket"]):
        k = 2 + i % 3
        w = np.array(cyc([[0.5, 0.3, 0.2, 0.0], [0.25, 0.25, 0.25, 0.25], [0.4, 0.35, 0.15, 0.10]], i)[:k])
        prods.append(ns.BasketOption(cyc([0.75, 1.25, 2.0, 2.5], i), ids[:k], list(w / w.sum()), 95.0 + 5.0 * (i % 5),
                                     ns.OptionType.CALL if i % 2 == 0 else ns.OptionType.PUT,
                                     ns.BasketOptionType.ARITHMETIC if i % 3 else ns.BasketOptionType.GEOMETRIC, False))
    for i in range(counts["asian"]):
        prods.append(ns.AsianOption(0.0, cyc([0.5, 0.75, 1.0, 1.5, 2.0], i), 88.0 + 6.0 * (i % 6), cyc([8, 12, 18, 24], i),
                                    ns.OptionType.CALL if i % 2 == 0 else ns.OptionType.PUT,
                                    ns.AsianAveragingType.ARITHMETIC if i % 3 else ns.AsianAveragingType.GEOMETRIC,
                                    asset_id=cyc(ids, i)))
    for i in range(counts["barrier"]):
        prods.append(ns.BarrierOption(startdate=0.0, maturity=cyc([0.5, 0.75, 1.25, 1.75, 2.5, 3.0], i), strike=85.0 + 7.5 * (i % 6),
                                      num_observation_timepoints=cyc([8, 12, 18, 24, 36], i),
                                      option_type=ns.OptionType.CALL if i % 3 else ns.OptionType.PUT,
                                      barrier1=cyc([118.0, 125.0, 132.0, 140.0], i) + 2.0 * (i % 2),
                                      barrier_option_type1=ns.BarrierOptionType.UPANDOUT, asset_id=cyc(ids, i)))
    for i in range(counts["american"]):
        a = cyc(ids, i)
        prods.append(ns.AmericanOption(underlying=ns.Equity(a), maturity=cyc([0.75, 1.0, 1.5, 2.0, 2.5, 3.0], i),
                                       num_exercise_dates=cyc([8, 12, 18, 24, 36, 48], i),
                                       strike=cyc([80.0, 92.5, 100.0, 107.5, 120.0], i),
                                       option_type=ns.OptionType.PUT if i % 2 == 0 else ns.OptionType.CALL, asset_id=a))
    for i in range(counts["flexicall"]):
        a, mat, m = cyc(ids, i), cyc([1.0, 1.5, 2.0, 2.5], i), cyc([3, 4, 5], i)
        unders = [ns.EuropeanOption(ns.Equity(a), float(t), 92.0 + 4.0 * j, ns.OptionType.CALL, asset_id=a)
                  for j, t in enumerate(np.linspace(mat / m, mat, m))]
        prods.append(ns.FlexiCall(underlyings=unders, num_exercise_rights=min(2, m - 1), asset_id=a))
    import cases
    for i in range(counts.get("storage", 0)):       # pv_performance_large_netting_set.py:235-251
        prods.append(cases.book_storage(ns, i, cyc(ids, i), cyc([1.0, 1.5, 2.0, 2.5], i), cyc([18.0, 26.0, 34.0, 42.0], i),
                                        cyc([0.05, 0.10, 0.125], i), 6 + i % 5, 2.0 + 0.5 * (i % 5), 0.10 + 0.02 * (i % 4),
                                        0.08 + 0.015 * (i % 4)))
    return prods


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--paths", type=int, default=1000)
    ap.add_argument("--exposure-points", type=int, default=0,
                    help="> 0: EPE + PFE(0.95) on that many exposure dates over 2.5y "
                         "(tests/exposure_tests/ee_performance_large_netting_set.py) instead of PV")
    ap.add_argument("--cva", action="store_true",
                    help="CVA of the book against a counterparty with a CIR++ intensity, 80 exposure dates over the book's "
                         "horizon, MPoR 10 days, EULER (tests/exposure_tests/cva_perfprmance_large_netting_set.py:69-193)")
    ap.add_argument("--differentiate", action="store_true",
                    help="PV with first-order pathwise sensitivities to every model parameter; also prints the norm of the "
                         "gradient and the number of derivatives that are not None")
    args = ap.parse_args()
    if args.differentiate and (args.cva or args.exposure_points > 0):
        ap.error("--differentiate runs the PV book")
    importlib.import_module("montecarlo-risk-engine_b200")
    import torch
    import cases
    from mcre import binding as B
    ns = cases.Namespace()
    base = dict(european=39400, binary=1000, basket=1000, asian=2000, barrier=4000, american=1800, flexicall=700)
    # the reference's PV book carries 100 gas storages, its exposure and CVA books 10 of their 5000 products
    # (ee_performance_large_netting_set.py:36, cva_perfprmance_large_netting_set.py:78)
    base["storage"] = 100
    counts = {k: max(1, int(round(v * args.scale))) for k, v in base.items()}
    ids = [f"asset_{i}" for i in range(4)]
    corr = np.full((4, 4), 0.35) + 0.65 * np.eye(4)
    model = ns.BlackScholesMulti(calibration_date=0.0, rate=0.03, asset_ids=ids, spots=[95.0 + 7.5 * i for i in range(4)],
                                 volatilities=[0.18 + 0.03 * i for i in range(4)], correlation_matrix=corr)
    prods = build_book(ns, ids, counts)
    nset = ns.NettingSet(name="mixed_state_dependent_book", products=prods)
    scheme = ns.SimulationScheme.ANALYTICAL
    if args.cva:
        credit = ns.CIRPPModel(calibration_date=0.0, asset_id="cp", hazard_rates=cases.HAZARDS, kappa=0.10, theta=0.01,
                               volatility=0.02, y0=0.0001)
        market = model
        model = ns.ModelConfig(models=[market, credit], inter_asset_correlation_matrix=[np.full((4, 1), 0.2, dtype=float)])
        horizon = max(float(p.modeling_timeline[-1]) for p in prods)
        nset = ns.NettingSet(name="mixed_state_dependent_book_cva", products=prods, counterparty_id="cp",
                             margin_period_of_risk=10 / 252)
        rm = ns.RiskMetrics([ns.CVAMetric("cp", 0.4)], exposure_timeline=np.linspace(0.0, horizon, args.exposure_points or 80))
        scheme = ns.SimulationScheme.EULER
    elif args.exposure_points > 0:
        rm = ns.RiskMetrics([ns.EPEMetric(), ns.PFEMetric(0.95)], exposure_timeline=np.linspace(0.0, 2.5, args.exposure_points))
    else:
        rm = ns.RiskMetrics([ns.PVMetric()])
    sc = ns.SimulationController([nset], model, rm, args.paths, args.paths, 1, scheme, args.differentiate)
    # warm-up on a tiny book of the same kinds: CUDA module loading and allocator growth are not product work
    warm = build_book(ns, ids, {k: 2 for k in base})
    ns.SimulationController([ns.NettingSet(name="warm", products=warm)], model, ns.RiskMetrics([ns.PVMetric()]), args.paths,
                            args.paths, 1, scheme, args.differentiate).run_simulation()
    torch.cuda.synchronize()
    l0 = B.launch_count()
    t0 = time.perf_counter()
    res = sc.run_simulation()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if args.cva:
        shown = {"exposure_points": args.exposure_points or 80,
                 "cva": float(res.get_results(nset.get_name(), "cva[cp]", evaluation_idx=0)),
                 "mc_error": float(res.get_mc_error(nset.get_name(), "cva[cp]", evaluation_idx=0))}
    elif args.exposure_points > 0:
        epe = np.asarray(res.get_results(nset.get_name(), "epe"))
        shown = {"exposure_points": args.exposure_points, "epe_mean": float(epe.mean()), "epe_max": float(epe.max()),
                 "pfe_max": float(np.asarray(res.get_results(nset.get_name(), "pfe[0.95]")).max())}
    else:
        shown = {"pv": float(res.get_results(nset.get_name(), "pv", evaluation_idx=0)),
                 "mc_error": float(res.get_mc_error(nset.get_name(), "pv", evaluation_idx=0))}
        if args.differentiate:
            grad = [g for g in res.get_derivatives(nset.get_name(), "pv")[0] if g is not None]
            shown.update(gradient_norm=float(np.linalg.norm([float(g) for g in grad])), derivatives_not_none=len(grad))
    print(json.dumps({"num_products": len(prods), **counts, "paths": args.paths, "timeline_size": int(sc.simulation_timeline.numel()),
                      **shown,
                      "total_seconds": dt, "products_per_second": len(prods) / dt, "kernel_launches": B.launch_count() - l0,
                      "timings": {k: round(v, 4) for k, v in sc.last_timings.items()}}))


if __name__ == "__main__":
    main()
