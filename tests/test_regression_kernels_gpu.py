"""The regression kernels through the C ABI, against exact references, at the shapes where reductions and grid-stride
loops go wrong: the Longstaff-Schwartz exercise step and its batched forms (csrc/lsm.cu), the 3x3 device solver
(csrc/solve3.cuh), the storage moments, normal-equation solver and backward step (csrc/storage.cu).

References
----------
* Sums: math.fsum of the per-path terms, each term computed in numpy with the kernel's own double expressions.
* Solves: mpmath at 50 digits on the very double moments the kernel reads; minimum-norm solutions from mpmath.eigsy.
* Exercise update: a numpy restatement of the rule of mcre_lsm_step_states (include/mcre.h): decisions in float64,
  the value update rounded through float32 like the kernel.

Tolerance model
---------------
* Moment sums: |got - fsum| <= 1e-13 * fsum(|terms|) per slot.  Losing or double counting one path at the largest
  size moves a sum by about 3e-6 relative, far above this bound.
* Value arrays: bit-identical on every path whose exercise margin |imm + cont[s] - cont[s+1]| exceeds 1e-12 of its
  scale.  The device may contract c0 + u (c1 + u c2) into FMAs, numpy does not; the near-tie paths are counted and the
  count must be small.  Without coefficients every cont is exactly zero, so every path must match, including the
  deliberate ties imm = 0, which must not exercise (the test is a strict >).
* Batched kernels: bit-identical (np.array_equal) to the per-product calls, unused moment slots exactly zero.
* 3x3 solver: the same coefficients as the host rule (mcre/lsm.py:solve_normal_equations) at 1e-12 relative, and both
  within kappa * 1e-15 of mpmath, kappa (at least 10) the ratio of the largest to the smallest kept eigenvalue of the
  system the branch solves (equilibrated on the full-rank branch); where kappa * 1e-15 exceeds 1e-12 (near the rank
  cut-off) the host comparison widens to it.  Coefficients are compared in
  the norm of the equilibrated basis, |(c - ref) * sqrt(diag G)| <= tol * |ref * sqrt(diag G)|.
* Storage solver: fitted values on the support of the samples within (1e-12 + kappa * 1e-14) * max|y| of
  numpy.linalg.lstsq(G, rhs, rcond=1e-12) in exact arithmetic, kappa = largest / smallest kept eigenvalue.  Keeping an
  eigenvalue the rule cuts moves them by O(max|y|).
* Storage backward step: bit-identical on every (path, state) whose best action is clear of the runner-up by 1e-12 of
  their scale (the continuation polynomial may contract into FMAs; the inventory arithmetic is unfused by design);
  bit-identical everywhere on the last date, which has no continuation."""
import ctypes as C
import math

import mpmath
import numpy as np
import pytest
import torch

import cases
from mcre import binding as B
from mcre.lsm import LSM_MAX_NV, LSM_MAX_RIGHTS, STEP_JOB, solve_normal_equations

pytestmark = pytest.mark.gpu

mpmath.mp.dps = 50

SUM_RTOL = 1e-13
MARGIN = 1e-12
SH_K, SC_K = 100.0, 0.05          # standardisation of the regression date's spot
SH_I, SC_I = 95.0, 0.04           # ... and of the product date's (different, so that a swap shows)
MOMENTS_JOB = np.dtype([("x", "u8"), ("v", "u8"), ("nk", "f8"), ("shift", "f8"), ("scale", "f8")])   # mcre_lsm_job
VARIANTS = ["no_imm", "no_coef", "coef"]    # regression date without product date / last product date / with coefficients


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _sizes(chunk, cap_blocks_per_sm=8, cap=True):
    """Path counts across chunk edges, several chunks, and (cap) one count whose chunks outnumber the kernel's grid cap
    of cap_blocks_per_sm * multi_processor_count blocks, so that blocks loop over several chunks."""
    out = [1, 255, 257, 4095, 4097, 3 * 4096 + 17]
    if cap:
        out.append((cap_blocks_per_sm * _sm_count() + 3) * chunk + 17)
    return out


def _nan(*shape):
    """Device buffer pre-filled with NaN: a slot the kernel forgets to write shows."""
    return torch.full(shape, float("nan"), dtype=torch.float64, device="cuda")


def _assert_sums(got, terms, what):
    got = np.asarray(got, dtype=np.float64)
    assert got.shape[0] == len(terms), f"{what}: {got.shape[0]} slots, {len(terms)} expected"
    for i, t in enumerate(terms):
        ref, mag = math.fsum(t), math.fsum(np.abs(t))
        assert abs(got[i] - ref) <= SUM_RTOL * mag, f"{what} slot {i}: {got[i]!r} vs fsum {ref!r} (sum |t| {mag:.3e})"


# ---- A. exercise step ----------------------------------------------------------------------------------------------
def _step_data(R, n, seed):
    rng = np.random.default_rng(seed)
    d = dict(xk=rng.uniform(60.0, 140.0, n), nk=rng.uniform(1.0, 1.1, n), xi=rng.uniform(60.0, 140.0, n),
             ni=rng.uniform(1.0, 1.1, n), imm=np.maximum(rng.uniform(-20.0, 30.0, n), 0.0))   # 40 % exact zeros
    value = rng.uniform(0.0, 20.0, (R, n)).astype(np.float32)
    coef = rng.uniform(-1.0, 1.0, (R, 3)) * np.array([8.0, 3.0, 1.0])
    coef[:, 0] += 6.0 * np.arange(1, R + 1)          # continuation values grow with the rights left
    return d, value, coef


def _step_ref(R, d, value, coef, variant):
    """-> (updated float32 value [R, n], mask of paths whose decisions are clear of a tie, moment terms [5 + 3R])."""
    n = value.shape[1]
    v, clear = value.copy(), np.ones(n, dtype=bool)
    if variant != "no_imm":
        imm = d["imm"]
        cont = [np.zeros(n)] * (R + 1)
        if variant == "coef":
            ui = (d["xi"] - SH_I) * SC_I
            cont = [np.zeros(n)] + [coef[s, 0] + ui * (coef[s, 1] + ui * coef[s, 2]) for s in range(R)]
        pay = imm / d["ni"]
        nv = np.empty_like(v)
        for s in range(R):
            lhs = imm + cont[s]
            ex = lhs > cont[s + 1]
            if variant == "coef":
                scale = np.maximum(np.abs(imm), np.maximum(np.abs(cont[s]), np.abs(cont[s + 1])))
                clear &= np.abs(lhs - cont[s + 1]) > MARGIN * scale
            step = np.where(ex, pay, 0.0).astype(np.float32)
            prev = v[s - 1] if s > 0 else np.zeros(n, dtype=np.float32)
            nv[s] = step + np.where(ex, prev, v[s])
        v = nv
    u = (d["xk"] - SH_K) * SC_K
    u2 = u * u
    terms = [np.ones(n), u, u2, u2 * u, u2 * u2]
    for s in range(R):
        y = d["nk"] * v[s].astype(np.float64)
        terms += [y, y * u, y * u2]
    return v, clear, terms


def _dev(d):
    return {k: torch.from_numpy(np.ascontiguousarray(a)).cuda() for k, a in d.items()}


def _step_states(L, R, dd, coef, variant, value, n, chunk, entry="states"):
    """mcre_lsm_step_states (entry "step": mcre_lsm_step, one right) on device arrays; value (device, float32 [R, n]) is
    updated in place -> moments (host)."""
    nv = 5 + 3 * R
    partial, mom = _nan(max(-(-n // chunk), 1) * nv + 1), _nan(nv)
    keep, cptr = B.as_dp(coef.reshape(-1)) if variant == "coef" else (None, None)
    ex = (None, None, None) if variant == "no_imm" else (dd["xi"].data_ptr(), dd["ni"].data_ptr(), dd["imm"].data_ptr())
    args = (dd["xk"].data_ptr(), dd["nk"].data_ptr(), SH_K, SC_K, *ex, cptr, SH_I, SC_I, value.data_ptr(), n, chunk,
            partial.data_ptr(), mom.data_ptr(), 0)
    B.check(L.mcre_lsm_step(*args) if entry == "step" else L.mcre_lsm_step_states(R, *args))
    torch.cuda.synchronize()
    return mom.cpu().numpy()


def _check_step(L, R, n, chunk, variant, seed):
    d, value, coef = _step_data(R, n, seed)
    dd = _dev(d)
    val = torch.from_numpy(value).cuda()
    mom = _step_states(L, R, dd, coef, variant, val, n, chunk)
    want_v, clear, terms = _step_ref(R, d, value, coef, variant)
    what = f"R={R} n={n} chunk={chunk} {variant}"
    _assert_sums(mom, terms, what)
    got_v = val.cpu().numpy()
    near = int(np.sum(~clear))
    assert near <= 2 + n // 100000, f"{what}: {near} near-tie paths"
    bad = np.nonzero(np.any(got_v[:, clear] != want_v[:, clear], axis=0))[0]
    assert bad.size == 0, f"{what}: value differs on {bad.size} clear paths, first {np.nonzero(clear)[0][bad[0]]}"
    if variant == "no_coef":
        # exact ties imm = 0 against cont = 0: never exercised, the values of those paths are untouched
        ties = d["imm"] == 0.0
        assert ties.any() or n < 8
        assert np.array_equal(got_v[:, ties], value[:, ties]), f"{what}: a path with imm = 0 exercised"


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("R", range(1, LSM_MAX_RIGHTS + 1))
@pytest.mark.parametrize("chunk", [256, 4096])
def test_lsm_step_states_matches_fsum_and_numpy(chunk, R, variant):
    """mcre_lsm_step_states, 1..6 rights, across chunk edges and (chunk 256) past the grid cap of sm_count * 8 blocks:
    moments against fsum, the float32 values against the numpy restatement of the exercise update."""
    L = B.lib()
    for n in _sizes(chunk, cap=chunk == 256):
        _check_step(L, R, n, chunk, variant, seed=1000 * R + n % 997)


def test_lsm_step_states_past_the_grid_cap_at_chunk_4096():
    """The same past the grid cap at the 4096-path chunk of large pre-simulations (about 5e6 paths on a B200)."""
    _check_step(B.lib(), 1, (8 * _sm_count() + 1) * 4096 + 3, 4096, "coef", seed=7)


@pytest.mark.parametrize("R", range(1, LSM_MAX_RIGHTS + 1))
def test_lsm_step_states_without_paths_gives_zero_moments(R):
    L = B.lib()
    dd = _dev(dict(xk=np.zeros(1), nk=np.ones(1), xi=np.zeros(1), ni=np.ones(1), imm=np.ones(1)))
    val = torch.zeros((R, 1), dtype=torch.float32, device="cuda")
    coef = np.ones((R, 3))
    for variant in VARIANTS:
        mom = _step_states(L, R, dd, coef, variant, val, 0, 256)
        assert np.array_equal(mom, np.zeros(5 + 3 * R)), variant
    assert torch.equal(val, torch.zeros_like(val))


# ---- B. batched kernels, bit for bit -------------------------------------------------------------------------------
#: (rights, variant) of the jobs of one mcre_lsm_step_batch launch
JOB_MIX = [(1, "no_imm"), (2, "no_coef"), (3, "coef"), (4, "no_imm"), (5, "coef"), (6, "no_coef"), (6, "coef"),
           (1, "coef"), (2, "coef"), (3, "no_coef"), (4, "coef"), (5, "no_imm"), (1, "no_coef"), (6, "no_imm")]


@pytest.mark.parametrize("chunk", [256, 4096])
def test_lsm_step_batch_is_bit_identical_to_per_product_steps(chunk):
    """mcre_lsm_step_batch with jobs of 1..6 rights, with and without exercise update and coefficients: every job's
    moment row and value array equal those of its own mcre_lsm_step_states call on a fresh copy; the unused tail of each
    23-wide row is exactly zero."""
    L = B.lib()
    for n in [0] + _sizes(chunk, cap=chunk == 256):
        # three input sets shared by the jobs (like products on one asset); values, coefficients per job
        pools = [_dev(_step_data(1, max(n, 1), 31 * q + n % 89)[0]) for q in range(3)]
        rng = np.random.default_rng(n % 1013)
        jobs, singles, batch_vals = np.zeros(len(JOB_MIX), dtype=STEP_JOB), [], []
        for j, (R, variant) in enumerate(JOB_MIX):
            dd = pools[j % 3]
            _, value, coef = _step_data(R, max(n, 1), 7 * j + 1)
            coef = coef + rng.uniform(-1.0, 1.0, coef.shape)
            v_batch = torch.from_numpy(value).cuda()
            v_single = v_batch.clone()
            singles.append((_step_states(L, R, dd, coef, variant, v_single, n, chunk), v_single))
            batch_vals.append(v_batch)
            job = jobs[j]
            job["n_rights"], job["xk"], job["nk"] = R, dd["xk"].data_ptr(), dd["nk"].data_ptr()
            job["shift_k"], job["scale_k"], job["shift_i"], job["scale_i"] = SH_K, SC_K, SH_I, SC_I
            job["value"] = v_batch.data_ptr()
            if variant != "no_imm":
                job["xi"], job["ni"], job["imm"] = dd["xi"].data_ptr(), dd["ni"].data_ptr(), dd["imm"].data_ptr()
            if variant == "coef":
                job["has_coef"] = 1
                job["coef"][:3 * R] = coef.reshape(-1)
        n_chunks = max(-(-n // chunk), 1)
        partial, mom = _nan(n_chunks * len(JOB_MIX) * LSM_MAX_NV + 1), _nan(len(JOB_MIX), LSM_MAX_NV)
        B.check(L.mcre_lsm_step_batch(len(JOB_MIX), jobs.ctypes.data, n, chunk, partial.data_ptr(), mom.data_ptr(), 0))
        torch.cuda.synchronize()
        rows = mom.cpu().numpy()
        for j, (R, variant) in enumerate(JOB_MIX):
            nv, what = 5 + 3 * R, f"n={n} chunk={chunk} job {j} (R={R}, {variant})"
            assert np.array_equal(rows[j, :nv], singles[j][0]), f"{what}: moments differ from the per-product call"
            assert np.array_equal(rows[j, nv:], np.zeros(LSM_MAX_NV - nv)), f"{what}: unused tail not zero"
            assert torch.equal(batch_vals[j], singles[j][1]), f"{what}: values differ from the per-product call"


@pytest.mark.parametrize("chunk", [256, 4096])
def test_lsm_moments_batch_is_bit_identical_and_matches_fsum(chunk):
    """mcre_lsm_moments_batch equals mcre_lsm_step_states(1, ..., imm = NULL) with the numeraire array filled with the
    job's constant, bit for bit, and both match fsum."""
    L = B.lib()
    n_jobs = 9
    for n in [0] + _sizes(chunk, cap=chunk == 256):
        m = max(n, 1)
        rng = np.random.default_rng(n % 1009)
        xs = torch.from_numpy(rng.uniform(60.0, 140.0, (3, m))).cuda()
        vs = torch.from_numpy(rng.uniform(-5.0, 20.0, (n_jobs, m)).astype(np.float32)).cuda()
        jobs = np.zeros(n_jobs, dtype=MOMENTS_JOB)
        jobs["x"] = [xs[j % 3].data_ptr() for j in range(n_jobs)]
        jobs["v"] = [vs[j].data_ptr() for j in range(n_jobs)]
        jobs["nk"] = rng.uniform(0.9, 1.2, n_jobs)
        jobs["shift"] = rng.uniform(90.0, 110.0, n_jobs)
        jobs["scale"] = rng.uniform(0.02, 0.08, n_jobs)
        partial, mom = _nan(max(-(-n // chunk), 1) * n_jobs * 8 + 1), _nan(n_jobs, 8)
        B.check(L.mcre_lsm_moments_batch(n_jobs, jobs.ctypes.data, n, chunk, partial.data_ptr(), mom.data_ptr(), 0))
        torch.cuda.synchronize()
        rows = mom.cpu().numpy()
        xs_h, vs_h = xs.cpu().numpy(), vs.cpu().numpy()
        for j in range(n_jobs):
            what = f"n={n} chunk={chunk} job {j}"
            nk_arr = torch.full((m,), float(jobs["nk"][j]), dtype=torch.float64, device="cuda")
            val = vs[j:j + 1].clone()
            p1, m1 = _nan(max(-(-n // chunk), 1) * 8 + 1), _nan(8)
            B.check(L.mcre_lsm_step_states(1, int(jobs["x"][j]), nk_arr.data_ptr(), float(jobs["shift"][j]),
                                           float(jobs["scale"][j]), None, None, None, None, 0.0, 1.0, val.data_ptr(), n,
                                           chunk, p1.data_ptr(), m1.data_ptr(), 0))
            torch.cuda.synchronize()
            assert np.array_equal(rows[j], m1.cpu().numpy()), f"{what}: differs from mcre_lsm_step_states"
            u = (xs_h[j % 3, :n] - jobs["shift"][j]) * jobs["scale"][j]
            u2 = u * u
            y = jobs["nk"][j] * vs_h[j, :n].astype(np.float64)
            _assert_sums(rows[j], [np.ones(n), u, u2, u2 * u, u2 * u2, y, y * u, y * u2], what)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("chunk", [256, 4096])
def test_lsm_step_dev_and_solve_dev_match_host_path(chunk, variant):
    """mcre_lsm_step_dev (coefficients read from device memory) equals mcre_lsm_step bit for bit, moments and values;
    mcre_lsm_solve_dev on those moments equals mcre/lsm.py:solve_normal_equations at 1e-12."""
    L = B.lib()
    for n in [0] + _sizes(chunk, cap=chunk == 256):
        m = max(n, 1)
        d, value, coef = _step_data(1, m, 17 + n % 991)
        dd = _dev(d)
        v_host, v_dev = torch.from_numpy(value).cuda(), torch.from_numpy(value).cuda()
        mom_host = _step_states(L, 1, dd, coef, variant, v_host, n, chunk, entry="step")
        d_coef = torch.from_numpy(coef.reshape(-1).copy()).cuda()
        ex = (None, None, None) if variant == "no_imm" else (dd["xi"].data_ptr(), dd["ni"].data_ptr(), dd["imm"].data_ptr())
        partial, mom = _nan(max(-(-n // chunk), 1) * 8 + 1), _nan(8)
        B.check(L.mcre_lsm_step_dev(dd["xk"].data_ptr(), dd["nk"].data_ptr(), SH_K, SC_K, *ex,
                                    d_coef.data_ptr() if variant == "coef" else None, SH_I, SC_I, v_dev.data_ptr(), n,
                                    chunk, partial.data_ptr(), mom.data_ptr(), 0))
        out = _nan(3)
        B.check(L.mcre_lsm_solve_dev(mom.data_ptr(), out.data_ptr(), 0))
        torch.cuda.synchronize()
        what = f"n={n} chunk={chunk} {variant}"
        assert np.array_equal(mom.cpu().numpy(), mom_host), f"{what}: moments differ from mcre_lsm_step"
        assert torch.equal(v_dev, v_host), f"{what}: values differ from mcre_lsm_step"
        G, rhs = _gram3(mom_host), mom_host[5:8]
        want = solve_normal_equations(G, rhs)
        _assert_coef(out.cpu().numpy(), want, G, 1e-12, what + " device vs host solve")


# ---- C. 3x3 device solver ------------------------------------------------------------------------------------------
def _gram3(m):
    return np.array([[m[0], m[1], m[2]], [m[1], m[2], m[3]], [m[2], m[3], m[4]]])


def _moments3(u, y):
    """The 8 moments of the step (sum u^0..u^4, sum y u^0..u^2), exactly rounded."""
    u2 = u * u
    return np.array([math.fsum(t) for t in (np.ones_like(u), u, u2, u2 * u, u2 * u2, y, y * u, y * u2)])


def _scale_of(G):
    d = np.sqrt(np.clip(np.diag(G), 0.0, None))
    return np.where(d > 0.0, d, 1.0)


def _assert_coef(got, want, G, rtol, what):
    """|(got - want) * sqrt(diag G)| <= rtol * |want * sqrt(diag G)| (coefficients in the equilibrated basis)."""
    d = _scale_of(G)
    err, ref = np.linalg.norm((got - want) * d), np.linalg.norm(want * d)
    assert np.all(np.isfinite(got)) and err <= rtol * ref, f"{what}: {got} vs {want} (error {err:.3e}, scale {ref:.3e})"


def _mp_eig(G):
    E, Q = mpmath.eigsy(mpmath.matrix(G.tolist()))
    return [E[i] for i in range(G.shape[0])], Q


def _mp_minnorm(G, rhs, rcond):
    """Minimum-norm solution of G c = rhs with the eigenvalues <= rcond * max cut, at 50 digits -> (c, kappa of the kept
    part, number kept)."""
    lam, Q = _mp_eig(G)
    top = max(abs(v) for v in lam)
    k = G.shape[0]
    c = [mpmath.mpf(0)] * k
    kept = [v for v in lam if v > rcond * top]
    for e, v in enumerate(lam):
        if v > rcond * top:
            proj = mpmath.fsum(Q[i, e] * mpmath.mpf(float(rhs[i])) for i in range(k)) / v
            c = [c[i] + Q[i, e] * proj for i in range(k)]
    return np.array([float(x) for x in c]), float(top / min(kept)) if kept else 0.0, len(kept)


def _equilibrated_ratio(G):
    Gs = G / np.outer(_scale_of(G), _scale_of(G))
    lam, _ = _mp_eig(Gs)
    return float(min(abs(v) for v in lam) / max(abs(v) for v in lam))


def _near_degenerate(ratio, seed):
    """Samples u = +-1 + delta z whose equilibrated Gram matrix has its smallest / largest eigenvalue near `ratio`
    (the weak direction is u^2 ~ 1, its eigenvalue ~ delta^2)."""
    rng = np.random.default_rng(seed)
    c, z = rng.choice([-1.0, 1.0], 400), rng.standard_normal(400)
    delta = 1e-3
    for _ in range(4):
        u = c + delta * z
        delta *= math.sqrt(ratio / _equilibrated_ratio(_gram3(_moments3(u, u))))
    return c + delta * z


def _solver_cases():
    rng = np.random.default_rng(5)
    u = rng.standard_normal(1000)
    out = {"random": (u, 3.0 + 2.0 * u - u * u + rng.standard_normal(1000), "full")}
    y = rng.uniform(0.0, 10.0, 300)
    out["u_zero"] = (np.zeros(300), y, "deficient")
    out["u_const"] = (np.full(300, 1.7), y, "deficient")
    out["u_two_values"] = (rng.choice([-0.8, 1.3], 300), y, "deficient")
    for ratio, branch in ((1e-9, "full"), (1e-11, "deficient")):
        u = _near_degenerate(ratio, seed=int(-math.log10(ratio)))
        out[f"ratio_{ratio:g}"] = (u, 2.0 + u + 0.5 * u * u + 0.1 * rng.standard_normal(u.size), branch)
    for s in (1e-6, 1e6):
        u = s * (1.0 + rng.uniform(0.0, 1.0, 500))
        v = u / s
        out[f"scale_{s:g}"] = (u, 1.0 + 2.0 * v - v * v + 0.1 * rng.standard_normal(500), "full")
    out["zero_rhs"] = (u, np.zeros(500), "full")
    return out


SOLVER_CASES = _solver_cases()


def _solve_dev(L, m):
    mom, out = torch.from_numpy(np.asarray(m, dtype=np.float64).copy()).cuda(), _nan(3)
    B.check(L.mcre_lsm_solve_dev(mom.data_ptr(), out.data_ptr(), 0))
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("case", list(SOLVER_CASES))
def test_solve3_dev_matches_host_rule_and_mpmath(case):
    """mcre_lsm_solve_dev on the moments of explicit samples: the host rule's branch, the host's coefficients, and the
    mpmath minimum-norm solution (full rank: the exact solve; rank deficient: the pseudo-inverse of the raw Gram matrix
    with the 1e-10 cut, the gelsy convention of to_raw_basis)."""
    u, y, branch = SOLVER_CASES[case]
    m = _moments3(u, y)
    G, rhs = _gram3(m), m[5:8]
    d = np.sqrt(np.diag(G))
    live = d > 0.0
    host_full = bool(live.all()) and _equilibrated_ratio(G) > 1e-10
    assert host_full == (branch == "full"), f"{case}: the case is not on the {branch} side of the cut"
    got, host = _solve_dev(B.lib(), m), solve_normal_equations(G, rhs)
    if case == "zero_rhs":
        assert np.array_equal(got, np.zeros(3)) and np.array_equal(host, np.zeros(3))
        return
    if branch == "full":
        Gs = G / np.outer(d, d)
        ys, kappa, _ = _mp_minnorm(Gs, rhs / d, 0.0)
        ref = ys / d
    else:
        ref, kappa, kept = _mp_minnorm(G, rhs, 1e-10)
        assert kept < 3
        # the cut matters: the uncut solution is far from the cut one
        full_inv, _, _ = _mp_minnorm(G, rhs, 0.0)
        if case.startswith("ratio"):
            assert np.linalg.norm((full_inv - ref) * _scale_of(G)) > 1e-3 * np.linalg.norm(ref * _scale_of(G))
    tol = max(kappa, 10.0) * 1e-15
    _assert_coef(got, host, G, max(1e-12, tol), f"{case}: device vs host")
    _assert_coef(host, ref, G, tol, f"{case}: host vs mpmath")
    _assert_coef(got, ref, G, tol, f"{case}: device vs mpmath")
    if case == "u_zero":
        assert np.allclose(got, [np.mean(y), 0.0, 0.0], rtol=1e-13, atol=0.0)
    if case == "u_const":
        phi = np.array([1.0, 1.7, 1.7 ** 2])
        _assert_coef(got, np.mean(y) * phi / phi.dot(phi), G, 1e-13, f"{case}: gelsy convention")


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf")])
@pytest.mark.parametrize("slot", range(5))
def test_solve3_dev_non_finite_gram_gives_zeros(slot, bad):
    u, y, _ = SOLVER_CASES["random"]
    m = _moments3(u, y)
    m[slot] = bad
    assert np.array_equal(_solve_dev(B.lib(), m), np.zeros(3))
    assert np.array_equal(solve_normal_equations(_gram3(m), m[5:8]), np.zeros(3))


def test_solve3_dev_rank_without_paths_gives_zeros():
    assert np.array_equal(_solve_dev(B.lib(), np.zeros(8)), np.zeros(3))


# ---- D. storage moments and solver ---------------------------------------------------------------------------------
def _storage_plan(S, NB):
    """A minimal plan: one (last) action date, no sub-steps, one knot per rate curve - enough for the moment and solve
    entry points, which read only the state and basis counts."""
    rec = np.zeros(48)
    rec[1], rec[3], rec[4], rec[8], rec[9], rec[10] = 1.0, float(S - 1), 1.0, 1.0, 1.0, 1.0
    arrays = dict(step=np.zeros(24), step_date=np.full(1, -1, np.int32), date_rec=rec, numeraire=np.ones(1),
                  step_tan=np.zeros(1), dlog_num=np.zeros(1), step_expo=np.full(1, -1, np.int32),
                  expo_numeraire=np.zeros(1))
    d = B.StorageDesc()
    d.n_sub, d.n_dates, d.n_pre_dates, d.n_states, d.n_basis = 0, 1, 0, S, NB
    d.log_spot0, d.noise_dim, d.n_tan, d.n_expo, d.n_pre_expo = math.log(100.0), 1, 0, 0, 0
    keep = []
    for name, a in arrays.items():
        a, ptr = (B.as_ip if a.dtype == np.int32 else B.as_dp)(a)
        keep.append(a)
        setattr(d, name, ptr)
    plan = C.c_void_p()
    B.check(B.lib().mcre_storage_create(C.byref(d), C.byref(plan)))
    return plan


@pytest.fixture
def storage_plan():
    plans = []

    def make(S, NB):
        plans.append(_storage_plan(S, NB))
        return plans[-1]
    yield make
    torch.cuda.synchronize()
    for p in plans:
        B.lib().mcre_storage_destroy(p)


@pytest.mark.parametrize("NB", range(1, 7))
@pytest.mark.parametrize("S", [2, 7, 16])
@pytest.mark.parametrize("chunk", [256, 4096])
def test_storage_moments_match_fsum(storage_plan, chunk, S, NB):
    """mcre_storage_moments against fsum: [s * NB + k] = sum u^k num value[s], then [S * NB + q] = sum u^q, q < 2 NB - 1;
    path counts across chunk edges and past 64 chunks (two levels of the tree reduction)."""
    L = B.lib()
    plan = storage_plan(S, NB)
    slots = L.mcre_storage_moment_slots(plan)
    assert slots == S * NB + 2 * NB - 1
    sizes = [0, 1, 255, 257, 4095, 4097]
    if chunk == 256 or NB in (1, 6):        # (fsum of ~3e5 paths x 100 slots is the slow part of the module)
        sizes.append(65 * chunk + 3)
    num, centre, inv_scale = 1.0372, 97.5, 0.11
    for n in sizes:
        m = max(n, 1)
        rng = np.random.default_rng(S * 100 + NB + n % 983)
        x = rng.uniform(80.0, 115.0, m)
        value = rng.uniform(-2e3, 5e3, (S, m))
        xd, vd = torch.from_numpy(x).cuda(), torch.from_numpy(value).cuda()
        partial, out = _nan(max(-(-n // chunk), 1) * slots + 1), _nan(slots)
        B.check(L.mcre_storage_moments(plan, num, centre, inv_scale, xd.data_ptr(), vd.data_ptr(), n, chunk,
                                       partial.data_ptr(), out.data_ptr(), 0))
        torch.cuda.synchronize()
        u = (x[:n] - centre) * inv_scale
        terms = []
        for s in range(S):
            w = num * value[s, :n]
            for _ in range(NB):
                terms.append(w)
                w = w * u
        w = np.ones(n)
        for _ in range(2 * NB - 1):
            terms.append(w)
            w = w * u
        _assert_sums(out.cpu().numpy(), terms, f"S={S} NB={NB} n={n} chunk={chunk}")


def _cholesky_gate(G):
    """The fast-path condition of storage_solve_kernel before it was made sound: every Cholesky pivot above 1e-8 of the
    largest diagonal entry."""
    nb, dmax = G.shape[0], float(np.max(np.diag(G)))
    Lc = np.zeros_like(G)
    for j in range(nb):
        dj = G[j, j] - Lc[j, :j] @ Lc[j, :j]
        if not dj > 1e-8 * dmax:
            return False
        Lc[j, j] = math.sqrt(dj)
        for i in range(j + 1, nb):
            Lc[i, j] = (G[i, j] - Lc[i, :j] @ Lc[j, :j]) / Lc[j, j]
    return True


def _storage_moments_of(u, counts, ys, NB):
    """Moments of samples with multiplicities: [s * NB + k] = sum count y_s u^k, [S * NB + q] = sum count u^q."""
    rows = [[c * yv * uv ** k for c, yv, uv in zip(counts, y, u)] for y in ys for k in range(NB)]
    rows += [[c * uv ** q for c, uv in zip(counts, u)] for q in range(2 * NB - 1)]
    return np.array([math.fsum(r) for r in rows])


def _ill_conditioned_family(n_cases=5):
    """NB = 6 Hankel moment matrices of discrete distributions with integer path counts that pass the old Cholesky gate
    although their eigenvalue ratio is below the 1e-12 cut, with every eigenvalue at least 10x clear of the cut: the
    example of the finding, then a seeded search."""
    found = [(np.array([5.637, 4.453, -3.436, -5.066, 2.451, -3.045]),
              np.array([24338.0, 382127.0, 157.0, 1095632.0, 380092.0, 8.0]))]
    rng = np.random.default_rng(2024)
    while len(found) < n_cases:
        u = np.round(rng.uniform(-6.0, 6.0, 6), 3)
        counts = np.floor(np.exp(rng.uniform(0.0, math.log(2e6), 6)))
        mom = _storage_moments_of(u, counts, [], 6)
        G = np.array([[mom[a + b] for b in range(6)] for a in range(6)])
        if not _cholesky_gate(G) or np.linalg.eigvalsh(G)[0] > 1e-13 * np.trace(G):
            continue
        lam, _ = _mp_eig(G)
        r = sorted(float(v / max(lam)) for v in lam)
        if r[0] < 1e-13 and not any(1e-13 <= v <= 1e-11 for v in r):
            found.append((u, counts))
    return found


def _storage_solver_cases():
    rng = np.random.default_rng(9)
    out = []
    for NB in range(1, 7):
        u = rng.standard_normal(2000)
        out.append((f"continuous_nb{NB}", NB, u, np.ones(2000)))
        out.append((f"deterministic_nb{NB}", NB, np.full(1, 0.37), np.array([4096.0])))
        for k in range(2, NB):
            out.append((f"rank{k}_nb{NB}", NB, np.linspace(-1.5, 2.0, k), rng.integers(1, 5000, k).astype(float)))
    for i, (u, counts) in enumerate(_ill_conditioned_family()):
        out.append((f"gate_passing_{i}", 6, u, counts))
    return out


STORAGE_SOLVER_CASES = {c[0]: c[1:] for c in _storage_solver_cases()}


@pytest.mark.parametrize("case", list(STORAGE_SOLVER_CASES))
def test_storage_solve_matches_mpmath_lstsq(storage_plan, case):
    """mcre_storage_solve against numpy.linalg.lstsq(G, rhs, rcond=1e-12) in exact arithmetic (the documented rule):
    fitted values on the support of the samples; entries 0..1 of the coefficient row (centre, inverse scale) untouched."""
    NB, u, counts = STORAGE_SOLVER_CASES[case]
    S = 3
    ys = [10.0 * np.sin(3.0 * u + s) + s for s in range(S)]
    mom = _storage_moments_of(u, counts, ys, NB)
    G = np.array([[mom[S * NB + a + b] for b in range(NB)] for a in range(NB)])
    plan = storage_plan(S, NB)
    d_mom = torch.from_numpy(mom).cuda()
    row = torch.full((2 + S * NB,), float("nan"), dtype=torch.float64, device="cuda")
    row[0], row[1] = 97.25, -0.125
    B.check(B.lib().mcre_storage_solve(plan, d_mom.data_ptr(), 1e-12, row.data_ptr(), 0))
    torch.cuda.synchronize()
    got = row.cpu().numpy()
    assert got[0] == 97.25 and got[1] == -0.125, f"{case}: centre / inverse scale overwritten"
    powers = u[:, None] ** np.arange(NB)[None, :]
    ymax = max(float(np.max(np.abs(y))) for y in ys)
    for s in range(S):
        ref, kappa, kept = _mp_minnorm(G, mom[s * NB:(s + 1) * NB], 1e-12)
        if case.startswith("deterministic"):
            assert kept == 1
        elif case.startswith("rank"):
            assert kept == int(case[4:case.index("_")])
        fit, want = powers @ got[2 + s * NB:2 + (s + 1) * NB], powers @ ref
        tol = (1e-12 + kappa * 1e-14) * ymax
        err = float(np.max(np.abs(fit - want)))
        assert err <= tol, f"{case} state {s}: fitted values off by {err:.3e} (tolerance {tol:.3e}, kept {kept} of {NB})"


# ---- E. one storage backward date ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def storage_product():
    from mcre.storage import StorageBackend, step_table
    from mcre.timegrid import build_time_grid
    ns = cases.Namespace()
    model, sets, metrics, _ = cases.storage_s2f(ns, which="storage2", end_day=40, num_states=6)
    sc = ns.SimulationController(sets, model, ns.RiskMetrics(metrics), 1024, 1024, 1, ns.SimulationScheme.ANALYTICAL,
                                 False, regression_function=ns.PolyomialRegression(degree=3))
    be = StorageBackend(sc)
    grid = build_time_grid(be._t0(), sc.simulation_timeline.tolist(), sc.num_steps)
    prod = sc.products[0]
    plan, numeraire, acts, _ = be._create(prod, grid, *step_table(sc.model, grid, sc.simulation_scheme, 0))
    yield prod, plan, numeraire, be.n_basis
    torch.cuda.synchronize()
    B.lib().mcre_storage_destroy(plan)


def _action_values(prod, i, spot, coeffs, NB, std):
    """The three action values of oracle/storage.py:cashflows per (path, state) entering date i, with the payoffs and the
    states the actions lead to -> (values, payoffs, next states), each [n, S, 3]."""
    from oracle import storage as OS
    S, n = prod.num_states, spot.shape[0]
    state = np.tile(np.arange(S, dtype=float), (n, 1))
    date, next_date = float(prod.product_timeline[i]), float(prod.next_action_dates[i])
    cfg = prod.storage_config
    moves = [OS.transition(prod, date, next_date, a, state) for a in ("inj", "no", "wd")]
    sp = spot[:, None]
    ci, cw = cfg.get_variable_injection_cost(date), cfg.get_variable_withdrawal_cost(date)
    pays = [-moves[0][1] * (sp + ci), -moves[1][1] * np.where(moves[1][1] >= 0.0, sp + ci, sp - cw),
            -moves[2][1] * (sp - cw)]
    nstates = np.stack([mv[0] for mv in moves], axis=2)
    if next_date >= prod.end_date - OS.DATE_TOL:
        return np.stack(pays, axis=2), np.stack(pays, axis=2), nstates
    grid = OS.basis((spot - std[0]) * std[1], NB) @ coeffs.T
    return np.stack([p + OS.lookup(grid, mv[0], S) for p, mv in zip(pays, moves)], axis=2), np.stack(pays, axis=2), nstates


@pytest.mark.parametrize("n", [1, 127, 129, 1000])
@pytest.mark.parametrize("which", ["inner", "last"])
def test_storage_backward_matches_oracle(storage_product, which, n):
    """mcre_storage_backward on one inner date (continuation polynomials per state) and on the last date of a real
    storage against oracle/storage.py cashflows + lookup: float32 cashflow over the numeraire plus the float64 tail
    interpolated at the state the best action leads to."""
    from oracle import storage as OS
    prod, plan, numeraire, NB = storage_product
    S = prod.num_states
    i = len(prod.product_timeline) - 1 if which == "last" else len(prod.product_timeline) // 2
    rec = prod.lower()[i]
    assert (rec[10] != 0.0) == (which == "last")
    rng = np.random.default_rng(n)
    spot = 92.0 * np.exp(0.08 * rng.standard_normal(n))
    value_in = rng.uniform(0.0, 5e6, (S, n))
    centre, inv_scale = 92.0, 0.2
    # continuation worth s * (inventory per state) * P(u): injecting pays where P exceeds the spot plus the cost (low
    # spots), withdrawing where it falls below the spot less the cost (spots a little above the centre)
    coeffs = np.array([[92.0, 3.0, 0.5, -0.05]]) * (rec[1] * np.arange(S))[:, None]
    coeffs = coeffs[:, :NB]
    row = np.concatenate([[centre, inv_scale], coeffs.reshape(-1)])
    d_row, d_spot = torch.from_numpy(row).cuda(), torch.from_numpy(spot).cuda()
    d_val = torch.from_numpy(value_in.copy()).cuda()
    B.check(B.lib().mcre_storage_backward(plan, i, d_row.data_ptr(), d_spot.data_ptr(), d_val.data_ptr(), n, 0))
    torch.cuda.synchronize()
    got = d_val.cpu().numpy().T                                                       # [n, S]
    num = np.full(n, numeraire[i])
    state = np.tile(np.arange(S, dtype=float), (n, 1))
    nstate, cf = OS.cashflows(prod, i, spot, num, state, coeffs, NB, (centre, inv_scale))
    want = cf.astype(np.float32).astype(np.float64) + OS.lookup(value_in.T, nstate, S)
    vals, pays, nstates = _action_values(prod, i, spot, coeffs, NB, (centre, inv_scale))
    order = np.argsort(vals, axis=2, kind="stable")
    top = [np.take_along_axis(a, order[..., 2:0:-1], axis=2) for a in (vals, pays, nstates)]    # best, runner-up
    (v1, v2), (p1, p2), (s1, s2) = ((t[..., 0], t[..., 1]) for t in top)
    # clear: the runner-up is 1e-12 of the scale behind, or leads to the same payoff and state (an empty store cannot
    # withdraw: holding and withdrawing are the same move, an exact tie on both sides)
    clear = (v1 - v2 > MARGIN * np.max(np.abs(vals), axis=2)) | ((p1 == p2) & (s1 == s2))
    if which == "last":
        clear[:] = True       # no continuation: the same arithmetic on both sides, ties included
    near = int(np.sum(~clear))
    assert near <= 2, f"{which} n={n}: {near} near-tie (path, state) pairs"
    bad = np.argwhere(clear & (got != want))
    assert bad.size == 0, f"{which} n={n}: {len(bad)} values differ, first (path, state) {tuple(bad[0])}"
    if n == 1000 and which == "inner":
        best = np.argmax(vals, axis=2)
        assert len(np.unique(best)) == 3, f"{which}: the inputs should exercise all three actions"
