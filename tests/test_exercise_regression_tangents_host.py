"""Differentiated normal equations of exercise products with several rights, on the host: per state s (rights left),
mcre.lsm.regression_tangents on that state's right-hand side, coefficients and tangent moments - split out of the
multi-state layout of mcre_lsm_step_states_tangents by state_tangent_moments - against the oracle's lstsq_dual (forward
mode through the least-squares solution, oracle/risk.py) on the same random paths and tangents.  Moments in numpy, no
GPU: one full-rank date and the rank-deficient t = 0 date (every path has the same explanatory value)."""
import numpy as np
import pytest

from mcre.lsm import regression_tangents, solve_normal_equations, state_tangent_moments
from oracle import ad
from oracle.risk import lstsq_dual


def _paths(rng, n, R, nt, degenerate):
    u = np.zeros(n) if degenerate else rng.standard_normal(n)
    du = rng.standard_normal((nt, n)) * 0.3
    Y = np.abs(rng.standard_normal((R, n))) * np.linspace(1.0, 2.0, R)[:, None]
    dY = rng.standard_normal((R, nt, n))
    return u, du, Y, dY


def _multi_state_moments(u, du, Y, dY):
    """[nt, 4 + 5 R] in the kernel's order: sum u^m du (m = 0..3), then per state sum dY, u dY, u^2 dY, du Y, 2 u du Y."""
    R, nt = Y.shape[0], du.shape[0]
    tm = np.zeros((nt, 4 + 5 * R))
    for p in range(nt):
        tm[p, :4] = [np.sum(u ** m * du[p]) for m in range(4)]
        for s in range(R):
            tm[p, 4 + 5 * s:9 + 5 * s] = [np.sum(dY[s, p]), np.sum(u * dY[s, p]), np.sum(u * u * dY[s, p]),
                                          np.sum(du[p] * Y[s]), np.sum(2.0 * u * du[p] * Y[s])]
    return tm


@pytest.mark.parametrize("degenerate", [False, True], ids=["full_rank", "t0_rank_deficient"])
@pytest.mark.parametrize("R", [1, 2, 6])
def test_per_state_regression_tangents_match_oracle_lstsq_dual(R, degenerate):
    rng = np.random.default_rng(7 + R + 10 * degenerate)
    n, nt = 400, 3
    u, du, Y, dY = _paths(rng, n, R, nt, degenerate)
    A = np.stack([np.ones(n), u, u * u], axis=1)
    G = A.T @ A
    tm = _multi_state_moments(u, du, Y, dY)
    dA = np.zeros((nt, n, 3))
    dA[:, :, 1], dA[:, :, 2] = du, 2.0 * u[None, :] * du
    for s in range(R):
        rhs = A.T @ Y[s]
        coef = solve_normal_equations(G, rhs)
        got = regression_tangents(G, rhs, coef, state_tangent_moments(tm, s))
        want = lstsq_dual(ad.Dual(A, dA), ad.Dual(Y[s][:, None], dY[s][:, :, None]))
        np.testing.assert_allclose(coef, want.v[:, 0], rtol=1e-8, atol=1e-8 * np.max(np.abs(want.v)))
        np.testing.assert_allclose(got, want.t[:, :, 0], rtol=1e-8, atol=1e-8 * np.max(np.abs(want.t)),
                                   err_msg=f"state {s + 1} of {R}")
