#!/usr/bin/env python
"""Headline benchmark: correlated path-steps/s of the Vasicek + CIR++ wrong-way-risk CVA
config (BASELINE.json configs[2]: payer swap 10y quarterly, 240 exposure steps, 2^24 paths
per GPU-job, rho sweep), on N B200s, next to the reference's own CPU implementation timed on the host cores.

    python bench.py --gpus N --steps K --warmup W            # this implementation
    python bench.py --impl reference --steps K --warmup W     # the UNMODIFIED reference (oracle/_ref, see oracle/make_ref.py)
    python bench.py --impl port --steps K --warmup W          # the oracle port (numpy restatement) on all host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also writes the last timed step's outputs

`--dump-outputs DIR` writes what the last timed step returned, so that two builds can be compared output for
output (same arguments -> same plans, coefficients and Philox streams): DIR/acc.npy and DIR/shift.npy, the
all-reduced accumulator of mcre_irc_mainsim and its pilot shifts (float64, one entry per slot), and DIR/cva.npy,
[CVA, Monte Carlo error] finished from them the way SimulationController.run_simulation() does.

A "step" is one full main-simulation pass (all paths x 240 sub-steps, one rho of the sweep)
with the plan and regression coefficients resident in HBM.  `e2e` times the public API
call (SimulationController.run_simulation(): plan lowering, pre-simulation regression,
H2D of the plan tables, main pass, D2H of the accumulators) from host objects.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "path-steps/sec (paths×steps) for Vasicek+CIR++ CVA"
UNIT = "path-steps/s"
N_STEPS_SIM = 240
FLOP_PER_PATH_STEP = 225.0  # SURVEY §8(d) algorithmic FP64 flop model for config 3
# what irc_cva_kernel executes per path-step: 45 DFMA + 13 DMUL + 6 DADD (profiles/r02_cva_kernel.md)
EXECUTED_FLOP_PER_PATH_STEP = 45 * 2 + 13 + 6
NCU_FP64_PIPE_PCT = 52.9          # sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active, final build
NCU_DRAM_BYTES_PER_LAUNCH = 101.6  # dram__bytes_read.sum + dram__bytes_write.sum of one launch: the state lives in registers
RHOS = np.linspace(-0.9, 0.9, 19)


def build_case(ns, rho):
    import cases
    vas = ns.VasicekModel(0., 0.03, 0.05, 0.02, 0.2, asset_id="irs")
    cir = ns.CIRPPModel(0., "GM", cases.HAZARDS, 0.1, 0.01, 0.02, 0.0001)
    model = ns.ModelConfig([vas, cir], inter_asset_correlation_matrix=np.array([rho]))
    irs = ns.InterestRateSwap(0.0, 10.0, 1.0, 0.03, 0.25, 0.25, ns.IRSType.PAYER, asset_id="irs")
    sets = [ns.NettingSet(name="irs", products=[irs], counterparty_id="GM")]
    metrics = [ns.CVAMetric("GM", 0.4)]
    return model, sets, metrics, np.arange(N_STEPS_SIM + 1) / 24.0


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.reasons, self.stop_flag, self.max_mhz = gpu_index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nme, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def cpu_port_rate(n_paths, repeats=1, rho=0.3, n_pre=2048):
    """Times the oracle (numpy restatement of the reference) on a bounded sample of the same
    workload: main-simulation phase only (paths + cashflows + exposure + CVA), coefficients fixed."""
    import cases
    from oracle import engine, risk
    ns = cases.Namespace()
    model, sets, metrics, tl = build_case(ns, rho)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        pre = engine.torch_reference_draws(42, n_pre, N_STEPS_SIM, 2)
        t_draw0 = time.perf_counter()
        # the reference's own draw procedure: one torch.randn(N, d, float64) per sub-step (model.py:47)
        main = engine.torch_reference_draws(43, n_paths, N_STEPS_SIM, 2)
        t_draw = time.perf_counter() - t_draw0
        t1 = time.perf_counter()
        out = risk.run(model, sets, metrics, tl, n_paths, n_pre, 1, "EULER", draws_pre=pre, draws_main=main)
        t2 = time.perf_counter()
        # main-sim share: total minus a pre-simulation of n_pre paths, plus drawing the normals
        dt = (t2 - t1) * n_paths / (n_paths + n_pre) + t_draw
        best = dt if best is None else min(best, dt)
    return n_paths * N_STEPS_SIM / best, best


def _cpu_worker(task):
    """One host core's share of a CPU step (runs in a spawned worker process)."""
    n_paths, rho = task
    import torch
    torch.set_num_threads(1)
    importlib.import_module("montecarlo-risk-engine_b200")
    if n_paths == 0:
        return 0.0          # warm-up task: imports only
    return cpu_port_rate(n_paths, rho=rho, n_pre=256)[1]   # tiny pre-simulation: the step is the main pass


class CpuPool:
    """The oracle port on ALL host cores: the path range of a CPU step is split over one
    single-threaded worker process per core (paths are independent, exactly like the GPU
    sharding); a step's time is the wall clock around the whole map."""

    def __init__(self, workers=None):
        import concurrent.futures as cf
        import multiprocessing as mp
        self.workers = workers or max(1, min(os.cpu_count() or 1, 64))
        self.pool = cf.ProcessPoolExecutor(self.workers, mp_context=mp.get_context("spawn"))
        list(self.pool.map(_cpu_worker, [(0, 0.0)] * self.workers))   # import everything once per worker

    def step(self, paths_per_worker, rho):
        t0 = time.perf_counter()
        list(self.pool.map(_cpu_worker, [(paths_per_worker, rho)] * self.workers))
        dt = time.perf_counter() - t0
        return self.workers * paths_per_worker * N_STEPS_SIM / dt, dt

    def close(self):
        self.pool.shutdown()


REF_SRC = os.path.join(ROOT, "oracle", "_ref", "src")


def reference_available():
    return os.path.isfile(os.path.join(REF_SRC, "controller", "controller.py"))


def run_reference_arm(args):
    """`--impl reference`: the UNMODIFIED reference (oracle/_ref/src, copied from /root/reference/src by
    oracle/make_ref.py) through its own public API: SimulationController(...).run_simulation() of config 3 on all host
    cores (torch intra-op threads), on a bounded sample of the paths.  `value` follows SURVEY 8d: main-simulation
    pipeline (the controller's own phase log: path_generation + request_resolution + valuation); `e2e` is the whole
    call including the pre-simulation, whose path count keeps the 1/16 ratio of the GPU arm.
    Falls back to the oracle port (kind "port") only when oracle/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not reference_available():
        return run_port_arm(args)
    import logging
    import types
    import torch
    # the reference's module names (controller, models, ...) are the ones this repo's package uses too: this process
    # imports the reference only
    sys.path.insert(0, REF_SRC)
    _helpers = types.ModuleType("helpers")          # namespace package in the reference; tests/helpers.py would win
    _helpers.__path__ = [os.path.join(REF_SRC, "helpers")]
    sys.modules["helpers"] = _helpers
    import cases
    ns = cases.Namespace()
    assert os.path.realpath(sys.modules["controller.controller"].__file__).startswith(os.path.realpath(REF_SRC))
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_main = 1 << args.ref_paths_log2
    n_pre = max(n_main >> 4, 1024)

    class Grab(logging.Handler):
        def __init__(self):
            super().__init__()
            self.phases = None

        def emit(self, record):
            if isinstance(record.args, tuple) and len(record.args) == 7:
                self.phases = dict(zip(("preprocessing", "path_generation", "request_resolution", "valuation", "total"),
                                       (float(x) for x in record.args[2:])))

    grab = Grab()
    lg = logging.getLogger("controller.controller")
    lg.setLevel(logging.INFO)
    lg.addHandler(grab)
    main_t, total_t, phases, cva = [], [], None, None
    for i in range(args.warmup + args.steps):
        model, sets, metrics, tl = build_case(ns, float(RHOS[i % len(RHOS)]))
        rm = ns.RiskMetrics(metrics, exposure_timeline=tl)
        t0 = time.perf_counter()
        sc = ns.SimulationController(sets, model, rm, n_main, n_pre, 1, ns.SimulationScheme.EULER)
        res = sc.run_simulation()
        wall = time.perf_counter() - t0
        ph = grab.phases
        if i >= args.warmup:
            main_t.append(ph["path_generation"] + ph["request_resolution"] + ph["valuation"])
            total_t.append(wall)
            phases = ph
            cva = float(res.get_results("irs", "cva[GM]")[0])
    ms = 1e3 * float(np.mean(main_t))
    value = n_main * N_STEPS_SIM / (ms * 1e-3)
    e2e_value = n_main * N_STEPS_SIM / float(np.mean(total_t))
    sample = (f"{n_main} main + {n_pre} pre-simulation paths x {N_STEPS_SIM} steps per step, unmodified reference "
              f"(oracle/_ref/src = /root/reference/src) SimulationController.run_simulation(), torch {torch.__version__} CPU, "
              f"{cores} intra-op threads; value = path_generation + request_resolution + valuation of its phase log")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[2]: Vasicek+CIR++ WWR CVA payer swap, 2^24 paths x 240 steps (bounded CPU sample)",
                       "paths_per_step": n_main, "presim_paths": n_pre, "sub_steps": N_STEPS_SIM},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "phases_last_step_s": phases, "cva_last_step": cva}
    print(json.dumps(line))


def run_port_arm(args):
    """The oracle port (numpy restatement) on all host cores: one single-threaded worker process per core."""
    pool = CpuPool()
    per_worker = (1 << 15) if pool.workers <= 32 else (1 << 14)   # ~0.8 GB of path tensor per worker
    n = per_worker * pool.workers
    times = []
    for i in range(args.warmup + args.steps):
        rate, dt = pool.step(per_worker, float(RHOS[i % len(RHOS)]))
        if i >= args.warmup:
            times.append(dt)
    pool.close()
    ms = 1e3 * float(np.mean(times))
    value = n * N_STEPS_SIM / (ms * 1e-3)
    sample = (f"{n} paths x {N_STEPS_SIM} steps per step ({per_worker} per worker process, {pool.workers} workers = host cores), "
              "main simulation incl. normal generation: torch.randn draws + numpy FP64 restatement of the reference")
    line = {"impl": "reference" if args.impl == "reference" else "port", "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[2]: Vasicek+CIR++ WWR CVA payer swap, 2^24 paths x 240 steps (bounded CPU sample)",
                       "paths_per_step": n, "sub_steps": N_STEPS_SIM},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": pool.workers, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--paths-log2", type=int, default=24, help="paths per GPU (weak scaling) / in total (strong scaling)")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: 2^paths-log2 paths per GPU (default, what the driver's scaling run uses); strong: "
                         "2^paths-log2 paths in total = BASELINE's 2^24-path config split over the GPUs")
    ap.add_argument("--presim-log2", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="kernel tuning runs: skip the end-to-end leg")
    ap.add_argument("--ref-paths-log2", type=int, default=17, help="main-simulation paths per step of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.impl == "port":
        return run_port_arm(args) if int(os.environ.get("RANK", "0")) == 0 else None

    import torch
    import torch.distributed as dist
    importlib.import_module("montecarlo-risk-engine_b200")
    import cases
    from mcre import binding as B
    from mcre import runtime as RT
    from mcre.irc import CHUNK_PATHS, IrcBackend

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = RT.compute_device()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ns = cases.Namespace()
    strong = args.scaling == "strong"
    n_total = (1 << args.paths_log2) if strong else (1 << args.paths_log2) * world
    n_per_gpu = n_total // world
    n_pre = 1 << args.presim_log2
    L = B.lib()

    # ---- resident plans: one per rho of the sweep actually visited ---------------------
    n_iter = args.warmup + args.steps
    plans = []
    for i in range(min(n_iter, len(RHOS))):
        model, sets, metrics, tl = build_case(ns, float(RHOS[i]))
        rm = ns.RiskMetrics(metrics, exposure_timeline=tl)
        sc = ns.SimulationController(sets, model, rm, n_total, n_pre, 1, ns.SimulationScheme.EULER)
        sc.rng_stream = i
        be = IrcBackend(sc)
        coefs = be.presim_coefficients(sc.products, dev)            # pre-simulation (untimed here)
        desc, keep, info = be.lower([0], [])
        plan = C.c_void_p()
        B.check(L.mcre_irc_create(C.byref(desc), C.byref(plan)))
        coef = np.zeros((info["n_expo"], 1, 3, 1))
        coef[:, 0, :, 0] = coefs[id(sc.products[0])][0]
        arr, ptr = B.as_dp(coef)
        B.check(L.mcre_irc_set_coefficients(plan, ptr, RT.stream_ptr()))
        torch.cuda.synchronize()
        plans.append((plan, keep, sc, info))
    begin, count = RT.shard_range(n_total, CHUNK_PATHS)
    slots = L.mcre_irc_main_slots(plans[0][0])
    acc = torch.zeros(slots, dtype=torch.float64, device=dev)
    shift = torch.zeros(slots, dtype=torch.float64, device=dev)
    partial = torch.empty(L.mcre_irc_partial_bytes(plans[0][0], count, CHUNK_PATHS, 0) // 8 + 1, dtype=torch.float64, device=dev)

    def step(i):
        plan = plans[i % len(plans)][0]
        rng = B.Rng()
        rng.mode, rng.seed, rng.stream, rng.n_paths_total = B.RNG_PHILOX, 43, i % len(plans), n_total
        sh = B.Shard(begin, count, CHUNK_PATHS)
        B.check(L.mcre_irc_mainsim(plan, C.byref(rng), C.byref(sh), partial.data_ptr(), acc.data_ptr(),
                                   shift.data_ptr(), None, RT.stream_ptr()))
        return RT.all_reduce_tree(acc)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
    launches0 = B.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        total = step(args.warmup + i)
        ev[i + 1].record()
    barrier()
    launches = B.launch_count() - launches0
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        from mcre.finish import irc_raw_to_neutral
        info = plans[(args.warmup + args.steps - 1) % len(plans)][3]
        acc_h, shift_h = total.cpu().numpy(), shift.cpu().numpy()
        rows = info["n_metric"] + 1
        res = irc_raw_to_neutral(acc_h.reshape(rows, -1), shift_h.reshape(rows, -1), n_total, 0, info["n_metric"],
                                 info["acc"])
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in (("acc", acc_h), ("shift", shift_h), ("cva", np.array(res["cva"][0], dtype=np.float64))):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    ms_total = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = n_total * N_STEPS_SIM / (ms_step * 1e-3)
    per_gpu = value / world

    # ---- roofline: FP64 pipe (SURVEY §8d) ------------------------------------------------
    peak = C.c_double(0.0)
    B.check(L.mcre_dfma_peak(C.byref(peak), RT.stream_ptr()))
    achieved = per_gpu * FLOP_PER_PATH_STEP * 1e-12
    executed = per_gpu * EXECUTED_FLOP_PER_PATH_STEP * 1e-12
    roofline = {"bound": "fp64", "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s",
                "frac": achieved / peak.value if peak.value > 0 else None,
                # what the hardware counts (profiles/r02_cva_kernel.md, ncu --set full of this build, 2^22 paths x 240 steps):
                "fp64_pipe_pct_ncu": NCU_FP64_PIPE_PCT,
                "executed_fp64_instr_per_path_step": 64, "executed_flop_per_path_step": EXECUTED_FLOP_PER_PATH_STEP,
                "executed_tflops": executed, "executed_frac": executed / peak.value if peak.value > 0 else None,
                "traffic": NCU_DRAM_BYTES_PER_LAUNCH, "traffic_unit": "bytes per launch (ncu, 2^22 paths x 240 steps)",
                "note": "frac: algorithmic 225 FP64 flop/path-step of SURVEY 8d (exp/log/sincos/sqrt/div weighted 20-30 flop) x path-steps/s / "
                        "DFMA peak measured in this run.  The kernel EXECUTES 64 FP64 instructions = 109 flop per path-step "
                        "(executed_frac, equal to ncu's sm__pipe_fp64_cycles_active within a point) next to 79 integer / other "
                        "instructions, 37 of them the ten Philox rounds; an FP64 instruction holds the issue port ~2.2 cycles, so "
                        "the path is issue bound at (2.2 x 64 + 79) slots per path-step, not HBM or tensor-core bound"}

    # ---- end to end through the public API (host objects in, numpy results out) ------------
    e2e_times, h2d, d2h = [], 0, 0
    cva = None
    # one untimed call first (first-use costs: NCCL connections of the moment all-gather, allocator growth), then best of 2
    for i in range(0 if args.no_e2e else 3):
        model, sets, metrics, tl = build_case(ns, float(RHOS[(i + 7) % len(RHOS)]))
        barrier()
        h2d0, d2h0 = B.h2d_bytes(), RT.d2h_bytes
        t0 = time.perf_counter()
        rm = ns.RiskMetrics(metrics, exposure_timeline=tl)
        sc = ns.SimulationController(sets, model, rm, n_total, n_pre, 1, ns.SimulationScheme.EULER)
        sc.rng_stream = 100 + i
        res = sc.run_simulation()
        cva = float(res.get_results("irs", "cva[GM]")[0])
        barrier()
        if i > 0:
            e2e_times.append(time.perf_counter() - t0)
        if os.environ.get("MCRE_BENCH_DEBUG") and e2e_times:
            sys.stderr.write(f"rank {rank} e2e {i}: {e2e_times[-1] * 1e3:.2f} ms {sc.last_timings}\n")
        h2d, d2h = B.h2d_bytes() - h2d0, RT.d2h_bytes - d2h0      # measured: counted where the copies are made
    e2e_dt = min(e2e_times) if e2e_times else float("inf")
    tt = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e = {"value": n_total * N_STEPS_SIM / float(tt.item()), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "includes": f"plan lowering + pre-simulation of 2^{args.presim_log2} paths + main pass; best of 2 calls after one untimed call",
           "cva": cva}

    # ---- parity guard: the same config on a small Philox stream, CUDA vs the oracle (checker only, not timed) ----
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import risk
        n_chk = 1 << 14
        model, sets, metrics, tl = build_case(ns, 0.3)
        rm = ns.RiskMetrics(metrics, exposure_timeline=tl)
        sc = ns.SimulationController(sets, model, rm, n_chk, n_chk, 1, ns.SimulationScheme.EULER)
        res = sc.run_simulation()
        got = float(res.get_results("irs", "cva[GM]")[0])
        out = risk.run(model, sets, metrics, tl, n_chk, n_chk, 1, "EULER")
        want = float(out["results"][0][0][0][0])
        parity = {"paths": n_chk, "rho": 0.3, "cva_cuda": got, "cva_oracle": want, "rel_diff": abs(got - want) / abs(want),
                  "what": "public API on native Philox vs oracle/ (numpy restatement pinned by the reference's goldens) on the same stream"}
        if not parity["rel_diff"] <= 1e-8:
            raise SystemExit(f"bench: CUDA result differs from the oracle on the same Philox stream: {parity}")

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # the reference's own implementation on the host cores (a subprocess: its module names collide with this
            # package's), bounded sample; the oracle port's number beside it
            ref = None
            if reference_available():
                try:
                    outp = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                           "--warmup", "0", "--ref-paths-log2", str(args.ref_paths_log2)],
                                          capture_output=True, text=True, timeout=900)
                    ref = json.loads(outp.stdout.strip().splitlines()[-1])
                except Exception as exc:  # noqa: BLE001
                    ref = None
                    sys.stderr.write(f"reference leg failed: {exc}\n")
            pool = CpuPool()
            per_worker = (1 << 15) if pool.workers <= 32 else (1 << 14)
            pool.step(per_worker, 0.3)
            rate, dt = max((pool.step(per_worker, 0.3) for _ in range(2)), key=lambda r: r[0])
            pool.close()
            port = {"value": rate, "cores": pool.workers,
                    "sample": f"{per_worker * pool.workers} paths x {N_STEPS_SIM} steps ({per_worker} per worker process, "
                              f"{pool.workers} workers = host cores), oracle (torch.randn draws + numpy FP64 restatement "
                              f"of the reference), main simulation, best of 2: {dt:.2f} s"}
            if ref is not None:
                cpu = dict(ref["cpu_baseline"], e2e_value=ref["e2e"]["value"], phases_s=ref.get("phases_last_step_s"), port=port)
            else:
                cpu = {"value": rate, "unit": UNIT, "cores": pool.workers, "kind": "port", "sample": port["sample"]}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": "configs[2]: Vasicek+CIR++ WWR CVA payer swap, rho sweep, 2^%d paths%s x 240 steps"
                                       % (args.paths_log2, " in total" if strong else "/GPU"),
                           "paths_per_gpu": n_per_gpu, "sub_steps": N_STEPS_SIM, "presim_paths": n_pre,
                           "l2": "no HBM-resident inputs: state in registers; each step re-reads only KB-sized plan tables"},
                "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
                "cpu_baseline": cpu, "parity_check": parity}
        print(json.dumps(line))
    for plan, *_ in plans:
        L.mcre_irc_destroy(plan)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
