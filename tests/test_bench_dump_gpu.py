"""bench.py --dump-outputs: the last timed step's outputs are what a caller of the public API receives for the same
rho and Philox stream, and two runs with the same arguments write the same bits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import cases

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PATHS_LOG2, PRESIM_LOG2, WARMUP, STEPS = 16, 14, 1, 2


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(STEPS), "--warmup", str(WARMUP),
           "--paths-log2", str(PATHS_LOG2), "--presim-log2", str(PRESIM_LOG2), "--no-cpu-baseline", "--no-e2e",
           "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_dump_outputs_repeat_and_match_public_api(tmp_path):
    line = _bench(tmp_path / "a")
    assert line["steps"] == STEPS
    _bench(tmp_path / "b")
    dumped = {}
    for name in ("acc", "shift", "cva"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.all(np.isfinite(a)), name
        np.testing.assert_array_equal(a, b, err_msg=name)
        dumped[name] = a
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20

    # the last timed step ran rho RHOS[k] on Philox stream k
    k = WARMUP + STEPS - 1
    ns = cases.Namespace()
    model, sets, metrics, tl = bench.build_case(ns, float(bench.RHOS[k]))
    sc = ns.SimulationController(sets, model, ns.RiskMetrics(metrics, exposure_timeline=tl), 1 << PATHS_LOG2,
                                 1 << PRESIM_LOG2, 1, ns.SimulationScheme.EULER)
    sc.rng_stream = k
    res = sc.run_simulation()
    cva, err = float(res.get_results("irs", "cva[GM]")[0]), float(res.get_mc_error("irs", "cva[GM]")[0])
    assert dumped["cva"][0] == pytest.approx(cva, rel=1e-9)
    assert dumped["cva"][1] == pytest.approx(err, rel=1e-6)
