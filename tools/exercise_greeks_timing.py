#!/usr/bin/env python
"""Cost of the sensitivities of exposure metrics of an exercise product: an American put on one Black-Scholes asset
(50 exercise dates, 25 exposure dates, EPE + ENE + PFE, ANALYTICAL), 2^20 main and 2^18 pre-simulation paths, value only
against differentiate=True end to end, and where the time of the sensitivity run goes:
  pre-simulation  = paths + value induction (the value-only run's pre-simulation), the tangent spill
                    (presim_tangent_spill) and the tangent induction (the rest of the sensitivity run's pre-simulation:
                    tangent gather, tangent steps, per-date tangent moment read-back and regression_tangents)
  main pass       = everything after the pre-simulation.
Every timer ends in a device synchronise; best of --repeat runs.  Writes the JSON to --out and prints it.
python tools/exercise_greeks_timing.py [--out profiles/exercise_greeks_timing.json]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
importlib.import_module("montecarlo-risk-engine_b200")
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--main-log2", type=int, default=20)
    ap.add_argument("--pre-log2", type=int, default=18)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exercise_greeks_timing.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    import cases
    from mcre.equity import EquityBackend
    ns = cases.Namespace()
    n_main, n_pre = 1 << args.main_log2, 1 << args.pre_log2
    timers = {}

    def timed(name, fn):
        def wrapper(*a, **k):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn(*a, **k)
            torch.cuda.synchronize()
            timers[name] = timers.get(name, 0.0) + time.perf_counter() - t0
            return r
        return wrapper
    EquityBackend.presim_exercise_all = timed("presim", EquityBackend.presim_exercise_all)
    EquityBackend.presim_tangent_spill = timed("spill", EquityBackend.presim_tangent_spill)

    def run(diff):
        model = ns.BlackScholesModel(0.0, 100.0, 0.03, 0.25)
        put = ns.AmericanOption(ns.Equity("id"), 1.0, 50, 100.0, ns.OptionType.PUT)
        metrics = [ns.EPEMetric(), ns.ENEMetric(), ns.PFEMetric(0.95)]
        sc = ns.SimulationController([ns.NettingSet(name="put", products=[put])], model,
                                     ns.RiskMetrics(metrics, exposure_timeline=np.linspace(0.0, 1.0, 25)), n_main, n_pre, 1,
                                     ns.SimulationScheme.ANALYTICAL, diff)
        timers.clear()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sc.run_simulation()
        torch.cuda.synchronize()
        return dict(timers, total=time.perf_counter() - t0)

    out = {"book": "AmericanOption put on one BlackScholesModel, 50 exercise dates, 25 exposure dates, EPE + ENE + PFE, "
                   "ANALYTICAL", "main_paths": n_main, "presim_paths": n_pre}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        out["gpu"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out["gpu"] = torch.cuda.get_device_name()
    run(False)      # warm-up: module load, allocator
    run(True)
    best = {}
    for _ in range(args.repeat):
        for label, diff in (("value", False), ("greeks", True)):
            t = run(diff)
            if label not in best or t["total"] < best[label]["total"]:
                best[label] = t
    v, g = best["value"], best["greeks"]
    out["seconds"] = {
        "value_only_end_to_end": v["total"],
        "greeks_end_to_end": g["total"],
        "presim_paths_and_value_induction": v["presim"],
        "presim_tangent_spill": g.get("spill", 0.0),
        "presim_tangent_induction": g["presim"] - v["presim"] - g.get("spill", 0.0),
        "main_pass_value_only": v["total"] - v["presim"],
        "main_pass_greeks": g["total"] - g["presim"],
    }
    # HBM traffic of the tangent induction kernels (R = 1, nt = 3: per path, date and parameter the step reads x_k, N_k,
    # x_i, N_i, imm_i, dx_k, dN_k, dN_i, dimm_i and the f32 value, reads and writes dV)
    n_dates = 50 + 25
    out["tangent_step_bytes"] = n_dates * 3 * n_pre * (9 * 8 + 4 + 16)
    print(json.dumps(out))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
