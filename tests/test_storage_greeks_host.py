"""Host side of the PV sensitivities of gas storages on Black-Scholes models (mcre/storage.py:tangent_slots, step_table
with tangents): a storage on one asset of a BlackScholesMulti or of a ModelConfig of Black-Scholes models, ANALYTICAL and
EULER.  CPU only: the step tangent records against central differences of the value records, the slot map, and the runs
that still raise."""
import numpy as np
import pytest
import torch

import cases


def _two_bs_config(ns):
    """A ModelConfig of two Black-Scholes models with different rates; the numeraire is the first one."""
    a = ns.BlackScholesModel(0.0, 100.0, 0.03, 0.2, asset_id="power")
    b = ns.BlackScholesModel(0.0, 24.0, 0.05, 0.35, asset_id="gas")
    return ns.ModelConfig(models=[a, b], inter_asset_correlation_matrix=[np.full((1, 1), 0.4)])


def _storage(ns, asset, end_day=5.0):
    cfg = ns.StorageConfig()
    cfg.add_volume_constraint(0.0, end_day, 0.0, 6.0, 0.0)
    cfg.add_injection_flexibility(0.0, end_day, 0.0, 2.0)
    cfg.add_withdrawal_flexibility(0.0, end_day, 0.0, 2.0)
    cfg.add_variable_injection_cost(0.0, 0.1)
    cfg.add_variable_withdrawal_cost(0.0, 0.1)
    return ns.Storage(asset_id=asset, start_date=0.0, end_date=end_day, initial_amount=1.0, storage_config=cfg, num_states=4)


def _models(ns):
    """(label, model, asset id) of the new combinations."""
    bsm, _, _, _ = cases.storage_mixed_book(ns)
    bs, _, _, _ = cases.storage_small(ns)
    return [("bsm_asset_1", bsm, "asset_1"), ("bs", bs, "gas"), ("config_gas", _two_bs_config(ns), "gas"),
            ("config_power", _two_bs_config(ns), "power")]


def test_tangent_slots_map_to_the_flattened_parameters():
    from mcre.storage import tangent_slots
    ns = cases.Namespace()
    got = {label: tangent_slots(model, asset) for label, model, asset in _models(ns)}
    # BlackScholesMulti [spots x3, vols x3, rate]: the asset's spot and volatility, the shared rate (also the numeraire's)
    assert got["bsm_asset_1"] == ([1, 4, 6], 2)
    assert got["bs"] == ([0, 1, 2], 2)
    # ModelConfig [power: spot, vol, rate, gas: spot, vol, rate], numeraire = power: its rate is a fourth slot
    assert got["config_gas"] == ([3, 4, 5, 2], 3)
    assert got["config_power"] == ([0, 1, 2], 2)
    s2f, _, _, _ = cases.storage_small(ns, model_kind="s2f")
    assert tangent_slots(s2f, "gas") == (list(range(6)), 0)


@pytest.mark.parametrize("scheme", ["ANALYTICAL", "EULER"])
def test_step_tangents_of_black_scholes_assets_equal_finite_differences(scheme):
    """d(A, B00, M, B10, B11, log F, Bw) per slot against central differences of the value records, for every parameter
    of the joint model.  The draw's coefficients cx bx_j move by dB00 (j = 0) + dBw cx bx_j under ANALYTICAL; under
    EULER the step's m and cx move by dM and dBw and the rows of the correlation factor stay.  Parameters outside the
    storage's slots - the other assets' spots and volatilities - leave the records unchanged."""
    from mcre.storage import STEP, step_table, tangent_slots
    from mcre.timegrid import build_time_grid
    ns = cases.Namespace()
    sch = getattr(ns.SimulationScheme, scheme)
    for label, model, asset in _models(ns):
        st = _storage(ns, asset)
        grid = build_time_grid(0.0, st.product_timeline.tolist(), 2)
        slots, _ = tangent_slots(model, asset)
        base, tan = step_table(model, grid, sch, len(slots), asset_id=asset, kernel_record=True)
        assert tan.shape == (max(grid.n_sub, 1), len(slots), 7)
        assert np.all(base[:, 7] == (1.0 if scheme == "EULER" else 0.0))
        n = grid.n_sub
        flat = [p for p in model.model_params]

        def table(k, v):
            old = float(flat[k])
            _set(model, k, v)
            t, _ = step_table(model, grid, sch, asset_id=asset)
            _set(model, k, old)
            return t[:n]
        for g in range(len(flat)):
            v0 = float(flat[g])
            h = 1e-6 * max(abs(v0), 1e-3)
            fd = (table(g, v0 + h) - table(g, v0 - h)) / (2 * h)
            if g not in slots:
                np.testing.assert_allclose(fd, 0.0, atol=1e-9, err_msg=f"{label} {scheme} parameter {g}")
                continue
            t = tan[:n, slots.index(g), :]
            what = f"{label} {scheme} parameter {g}"
            np.testing.assert_allclose(t[:, 2], fd[:, 3], rtol=2e-6, atol=1e-9, err_msg=what + " dM")
            np.testing.assert_allclose(t[:, 5], fd[:, 6], rtol=2e-6, atol=1e-9, err_msg=what + " d log F")
            if scheme == "EULER":
                np.testing.assert_allclose(t[:, 6], fd[:, 4], rtol=2e-6, atol=1e-9, err_msg=what + " d cx")
                np.testing.assert_allclose(fd[:, 8:8 + 8], 0.0, atol=1e-9, err_msg=what + " correlation rows")
                assert np.all(t[:, [0, 1, 3, 4]] == 0.0)
            else:
                cb = base[:n, 4:5] * base[:n, 8:16]
                want = t[:, 6:7] * cb
                want[:, 0] += t[:, 1]
                np.testing.assert_allclose(want, fd[:, 4:5] * base[:n, 8:16] + base[:n, 4:5] * fd[:, 8:16], rtol=2e-6,
                                           atol=1e-9, err_msg=what + " d(cx bx)")
                assert np.all(t[:, [0, 3, 4]] == 0.0)
        assert STEP == base.shape[1]


def _set(model, k, v):
    """Set flattened parameter k of a (possibly composite) model in place."""
    from models.model_config import ModelConfig
    if isinstance(model, ModelConfig):
        for m, off in zip(model.models, model.param_offsets()):
            if off <= k < off + len(m.model_params):
                m.model_params[k - off] = torch.tensor(v, dtype=torch.float64)
        model.model_params = [p for m in model.models for p in m.get_model_params()]
    else:
        model.model_params[k] = torch.tensor(v, dtype=torch.float64)


def test_new_sensitivity_runs_are_accepted_and_the_others_still_raise():
    from mcre.storage import StorageBackend
    ns = cases.Namespace()

    def ctrl(model, sets, metrics=None, scheme="ANALYTICAL", tl=None, **kw):
        rm = ns.RiskMetrics(metrics or [ns.PVMetric()], exposure_timeline=tl) if tl is not None else \
            ns.RiskMetrics(metrics or [ns.PVMetric()])
        return ns.SimulationController(sets, model, rm, 256, 256, 1, getattr(ns.SimulationScheme, scheme), True, **kw)
    model, sets, _, _ = cases.storage_mixed_book(ns)
    for scheme in ("ANALYTICAL", "EULER"):
        be = StorageBackend(ctrl(model, sets, scheme=scheme))
        assert be.mixed and be.nt == 3
    cfg = _two_bs_config(ns)
    be = StorageBackend(ctrl(cfg, [ns.NettingSet(name="s", products=[_storage(ns, "gas")])]))
    assert be.nt == 4 and be.slots["gas"] == ([3, 4, 5, 2], 3)
    bs, bs_sets, _, _ = cases.storage_small(ns)
    assert StorageBackend(ctrl(bs, bs_sets, scheme="EULER")).nt == 3
    # exposure metrics and CVA with sensitivities: still raise
    with pytest.raises(NotImplementedError, match="exposure"):
        StorageBackend(ctrl(model, sets, metrics=[ns.EPEMetric()], tl=[0.0, 0.5, 1.0]))
    cva_model, cva_sets, cva_metrics, tl = cases.storage_cva_mixed(ns)
    with pytest.raises(NotImplementedError):
        StorageBackend(ctrl(cva_model, cva_sets, metrics=cva_metrics, tl=tl, scheme="EULER"))
    # a storage in a ModelConfig with a credit model, PV only: still raises
    with pytest.raises(NotImplementedError, match="credit"):
        StorageBackend(ctrl(cva_model, cva_sets, scheme="EULER"))
