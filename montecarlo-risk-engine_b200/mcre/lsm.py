"""Longstaff-Schwartz backward induction driver shared by the model families.

The family-specific forward pass spills, date-major on the device, the explanatory variable
x[k][n] and numeraire N[k][n] per regression date k and the immediate exercise value imm[i][n]
per exercise date i; this module runs the reference's regression schedule
(src/controller/controller.py:294-383) over them with one fused `mcre_lsm_step` launch per
regression date (exercise update of the product date entering the window + 8 moments), an
all-reduce of the moments over the path-sharding ranks and a host solve of the 3x3 normal
equations."""
from __future__ import annotations

from bisect import bisect_left

import numpy as np
import torch

from mcre import binding as B
from mcre import runtime as RT


def solve_normal_equations(G, rhs):
    """Minimum-norm least-squares solution of G c = rhs (G = Gram matrix of the basis).

    The reference solves the tall system with LAPACK gelsy (controller.py:368-374), which
    returns the minimum-norm solution for rank-deficient designs (at t = 0 every path has
    the same explanatory value).  Same convention here via an SVD pseudo-inverse of the
    symmetrically equilibrated Gram matrix."""
    d = np.sqrt(np.clip(np.diag(G), 0.0, None))
    if not np.all(np.isfinite(G)) or d[0] == 0.0:
        return np.zeros(3)
    live = d > 0.0
    scale = np.where(live, d, 1.0)
    Gs = G / np.outer(scale, scale)
    u, s, vt = np.linalg.svd(Gs)
    tol = 1e-10 * s[0]
    rank = int(np.sum(s > tol))
    if rank == 3:
        return np.linalg.solve(Gs, rhs / scale) / scale
    # rank deficient (constant regressor): minimum norm in the unscaled coefficients, like gelsy
    u2, s2, vt2 = np.linalg.svd(G)
    keep = s2 > 1e-10 * s2[0]
    return (vt2[keep].T * (1.0 / s2[keep])) @ (u2[:, keep].T @ rhs)


def solve_normal_equations_batch(G, rhs):
    """solve_normal_equations for a stack of systems: G [n,3,3], rhs [n,3] -> [n,3].  One batched SVD /
    solve for the full-rank dates; rank-deficient ones (t = 0) go through the scalar routine."""
    G, rhs = np.asarray(G, dtype=np.float64), np.asarray(rhs, dtype=np.float64)
    n = G.shape[0]
    out = np.zeros((n, 3))
    if n == 0:
        return out
    d = np.sqrt(np.clip(np.diagonal(G, axis1=1, axis2=2), 0.0, None))
    ok = np.isfinite(G).all(axis=(1, 2)) & (d[:, 0] > 0.0) & (d > 0.0).all(axis=1)
    scale = np.where(d > 0.0, d, 1.0)
    Gs = G / (scale[:, :, None] * scale[:, None, :])
    Gs_safe = np.where(ok[:, None, None], Gs, np.eye(3)[None])
    sv = np.linalg.svd(Gs_safe, compute_uv=False)
    full = ok & (sv[:, 2] > 1e-10 * sv[:, 0])
    if full.any():
        sol = np.linalg.solve(Gs_safe[full], (rhs[full] / scale[full])[:, :, None])[:, :, 0]
        out[full] = sol / scale[full]
    # rank deficient (constant regressor, every exercise product's t = 0 date): minimum norm in the unscaled
    # coefficients like gelsy = the pseudo-inverse of the raw Gram matrix with the scalar routine's cut-off, batched
    # (the scalar routine per system cost 0.17 ms x thousands of products per book)
    usable = np.isfinite(G).all(axis=(1, 2)) & (d[:, 0] > 0.0)       # (the scalar routine returns zeros otherwise)
    todo = ~full & usable & np.any(rhs != 0.0, axis=1)      # a zero right-hand side has the zero solution in every branch
    if todo.any():
        u2, s2, vt2 = np.linalg.svd(G[todo])
        inv = np.where(s2 > 1e-10 * s2[:, :1], 1.0 / np.where(s2 > 0.0, s2, 1.0), 0.0)
        proj = np.einsum("nji,nj->ni", u2, rhs[todo])                  # u^T rhs
        out[todo] = np.einsum("nji,nj->ni", vt2, inv * proj)           # v (s^-1 u^T rhs)
    return out


def gram_pinv(G):
    """Pseudo-inverse of a Gram matrix with the rank decision of solve_normal_equations."""
    d = np.sqrt(np.clip(np.diag(G), 0.0, None))
    if not np.all(np.isfinite(G)) or d[0] == 0.0:
        return np.zeros((3, 3))
    scale = np.where(d > 0.0, d, 1.0)
    Gs = G / np.outer(scale, scale)
    s = np.linalg.svd(Gs, compute_uv=False)
    if s[2] > 1e-10 * s[0]:
        return np.linalg.inv(Gs) / np.outer(scale, scale)
    u2, s2, vt2 = np.linalg.svd(G)
    keep = s2 > 1e-10 * s2[0]
    return (vt2[keep].T * (1.0 / s2[keep])) @ u2[:, keep].T


def regression_tangents(G, rhs, coef, tm):
    """d(coefficients)/d(parameter) of the least-squares fit c = pinv(A) Y from moment sums.

    The reference keeps torch.linalg.lstsq inside the autograd graph (controller.py:368-383), whose
    backward is the derivative of the pseudo-inverse.  With A = [1, u, u^2] per path and everything
    expressed through sums over paths (G = A^T A, G+ = pinv(G), A+ = G+ A^T):
        dc = G+ (A^T dY - A^T dA c) + G+ (dA^T Y - dA^T A c) + (I - G+ G) dA^T A G+ c
    where A^T dA [i][j] = j sum u^(i+j-1) du.  The last term only matters on rank-deficient dates
    (t = 0: every path has the same x).
    G [3,3], rhs [3], coef [3], tm [nt, 9] (mcre_irc_presim tangent moments) -> [nt, 3]."""
    Gp = gram_pinv(G)
    nt = tm.shape[0]
    out = np.zeros((nt, 3))
    proj = np.eye(3) - Gp @ G
    for p in range(nt):
        mu, r, q1, q2 = tm[p, 0:4], tm[p, 4:7], tm[p, 7], tm[p, 8]
        AtdA = np.zeros((3, 3))
        for i in range(3):
            for j in (1, 2):
                AtdA[i, j] = j * mu[i + j - 1]
        dAtY = np.array([0.0, q1, q2])
        out[p] = Gp @ (r - AtdA @ coef) + Gp @ (dAtY - AtdA.T @ coef) + proj @ (AtdA.T @ (Gp @ coef))
    return out


def state_tangent_moments(tm, s):
    """Tangent moments of state s (0-based: s + 1 rights left) in the layout regression_tangents takes, [nt, 9], from
    the multi-state layout of mcre_lsm_step_states_tangents [nt, 4 + 5 R] (sum u^m du shared by the states)."""
    return np.concatenate([tm[:, :4], tm[:, 4 + 5 * s:9 + 5 * s]], axis=1)


LSM_MAX_RIGHTS = 6         # MCRE_LSM_MAX_RIGHTS (include/mcre.h)
LSM_MAX_NV = 5 + 3 * LSM_MAX_RIGHTS   # moments of the widest step


#: mcre_lsm_step_job (include/mcre.h)
STEP_JOB = np.dtype([("n_rights", "i4"), ("has_coef", "i4"), ("xk", "u8"), ("nk", "u8"), ("shift_k", "f8"), ("scale_k", "f8"),
                     ("xi", "u8"), ("ni", "u8"), ("imm", "u8"), ("coef", "f8", (3 * LSM_MAX_RIGHTS,)), ("shift_i", "f8"), ("scale_i", "f8"),
                     ("value", "u8")])
assert STEP_JOB.itemsize == 88 + 24 * LSM_MAX_RIGHTS


class DeferredSteps:
    """What a generator yields in batched mode: the step jobs of its current round (to be run in order) instead of
    launching them itself; the driver runs the j-th jobs of all products in one launch (mcre_lsm_step_batch)."""

    def __init__(self, jobs, count, chunk_paths):
        self.jobs, self.count, self.chunk_paths = jobs, count, chunk_paths


def backward_induction_steps(xs, nums, imm, ptl, reg_times, basis, count, chunk_paths, dev, n_rights=1, tangents=None,
                             batched=False):
    """Generator form of the backward induction: queues the kernels of one regression date, yields the device
    tensor that will hold its moments and expects the solved coefficients of that date back (`send`: [3, 3],
    one row per state, from the driver's all-reduce + batched normal-equation solve).  Returns the
    coefficients (StopIteration.value).  Lets a driver run many products in lock-step with ONE all-reduce and
    ONE device-to-host read per step for all of them (run_backward_inductions).

    xs, nums: device [n_reg, n]; imm: device [n_ex, n] (row i = product date i); ptl: product (exercise)
    dates; reg_times: regression dates (sorted, contain every product date); basis: [n_reg, 2] (shift, scale).
    -> coefficients in the standardised basis: [n_reg, 3] for one exercise right, [n_reg, n_rights, 3]
    (state s = rights left at row s-1) for a FlexiCall.
    tangents: dict(nt, dxs [n_reg, nt, n], dnums [n_reg, nt, n], dimm [n_ex, nt, n]) - the pathwise tangents of the
    spilled arrays; the generator then also returns d(coefficients)/d(parameters) (mcre_lsm_step_states_tangents +
    regression_tangents once per state, with the state's right-hand side, coefficients and tangent moments):
    -> (coef, dcoef), dcoef [n_reg, nt, 3] for one exercise right, [n_reg, n_rights, nt, 3] otherwise.  Tangent
    products step through the per-product launches (the exercise decisions, and so the coefficients, are those of the
    batched launch bit for bit)."""
    L = B.lib()
    stream = RT.stream_ptr()      # once per induction: tens of thousands of steps per book
    n_reg = len(reg_times)
    n = xs.shape[1]
    R = int(n_rights)
    nv = 5 + 3 * R
    reg_idx = {t: k for k, t in enumerate(reg_times)}
    coef = np.zeros((n_reg, R, 3))
    value = torch.zeros((R, n), dtype=torch.float32, device=dev)
    n_chunks = (n + chunk_paths - 1) // chunk_paths
    partial = torch.empty(n_chunks * nv + 1, dtype=torch.float64, device=dev)
    moments = torch.zeros(LSM_MAX_NV, dtype=torch.float64, device=dev)
    keep = {}
    if tangents is not None:
        nt = int(tangents["nt"])
        ntv = 4 + 5 * R       # tangent moments per parameter: sum u^m du, then 5 per state
        dxs, dnums, dimm = tangents["dxs"], tangents["dnums"], tangents["dimm"]
        dvalue = torch.zeros((R, nt, n), dtype=torch.float64, device=dev)
        tpartial = torch.empty(n_chunks * nt * ntv + 1, dtype=torch.float64, device=dev)
        tmoments = torch.zeros(nt * ntv, dtype=torch.float64, device=dev)
        dcoef = np.zeros((n_reg, R, nt, 3))

    batched = batched and tangents is None
    queue = []
    xs_ptr, nums_ptr, imm_ptr, value_ptr, row = xs.data_ptr(), nums.data_ptr(), imm.data_ptr(), value.data_ptr(), n * 8

    def step(k, i):
        """moments of regression date k, after the exercise update at product date i (or None)."""
        if batched:
            # the same call as below, recorded for the driver's batched launch
            job = np.zeros((), dtype=STEP_JOB)
            job["n_rights"], job["xk"], job["nk"] = R, xs_ptr + k * row, nums_ptr + k * row
            job["shift_k"], job["scale_k"], job["scale_i"], job["value"] = basis[k, 0], basis[k, 1], 1.0, value_ptr
            if i is not None:
                ki = reg_idx[ptl[i]]
                job["xi"], job["ni"], job["imm"] = xs_ptr + ki * row, nums_ptr + ki * row, imm_ptr + i * row
                job["shift_i"], job["scale_i"] = basis[ki, 0], basis[ki, 1]
                if i < len(ptl) - 1:
                    job["has_coef"] = 1
                    job["coef"][:3 * R] = coef[ki].reshape(-1)
            queue.append(job)
            return
        args_i = (None, None, None, None, 0.0, 1.0)
        if i is not None:
            ki = reg_idx[ptl[i]]
            cptr = None
            if i < len(ptl) - 1:
                keep["c"], cptr = B.as_dp(coef[ki].reshape(-1))
            args_i = (xs[ki].data_ptr(), nums[ki].data_ptr(), imm[i].data_ptr(), cptr,
                      float(basis[ki, 0]), float(basis[ki, 1]))
        B.check(L.mcre_lsm_step_states(R, xs[k].data_ptr(), nums[k].data_ptr(), float(basis[k, 0]), float(basis[k, 1]),
                                       *args_i, value.data_ptr(), count, chunk_paths, partial.data_ptr(),
                                       moments.data_ptr(), stream))
        if tangents is not None:
            # same exercise decision applied to the running tangents, then the tangent moments of date k
            targs = (None, None, None, None, None, None, 0.0, 1.0)
            if i is not None:
                targs = (args_i[0], args_i[1], args_i[2], dnums[ki].data_ptr(), dimm[i].data_ptr(), args_i[3],
                         args_i[4], args_i[5])
            B.check(L.mcre_lsm_step_states_tangents(R, nt, xs[k].data_ptr(), nums[k].data_ptr(), dxs[k].data_ptr(),
                                                    dnums[k].data_ptr(), float(basis[k, 0]), float(basis[k, 1]), *targs,
                                                    value.data_ptr(), dvalue.data_ptr(), count, chunk_paths,
                                                    tpartial.data_ptr(), tmoments.data_ptr(), stream))

    last = len(ptl)
    for k in range(n_reg - 1, -1, -1):
        t_reg = reg_times[k]
        pidx = bisect_left(ptl, t_reg)
        if pidx >= len(ptl):
            continue      # after the last exercise date: no continuation value (controller.py:303-305)
        t_next = pidx + 1 if ptl[pidx] == t_reg else pidx
        if t_next < last:
            for i in range(last - 1, t_next, -1):   # product dates that are not regression dates
                step(k, i)
            step(k, t_next)
            last = t_next
        else:
            step(k, None)
        if batched:
            jobs = list(queue)
            del queue[:]
            solved, m = yield DeferredSteps(jobs, count, chunk_paths)
        else:
            solved, m = yield moments   # [3 states, 3] from the driver's batched solve of this round, host moments
        coef[k] = solved[:R]
        if tangents is not None:
            tm = RT.all_reduce_tree(tmoments).cpu().numpy().reshape(nt, ntv)
            G = np.array([[m[0], m[1], m[2]], [m[1], m[2], m[3]], [m[2], m[3], m[4]]])
            for s in range(R):
                dcoef[k, s] = regression_tangents(G, m[5 + 3 * s:8 + 3 * s], coef[k, s], state_tangent_moments(tm, s))
    if tangents is not None:
        return (coef[:, 0, :], dcoef[:, 0]) if R == 1 else (coef, dcoef)
    return coef[:, 0, :] if R == 1 else coef


def backward_induction_device(xs, nums, imm, ptl, reg_times, basis, count, chunk_paths, dev):
    """Backward induction of ONE single-right exercise product (value-only) as a stream of kernels: per regression
    date the fused step launch (exercise update + 8 moments, mcre_lsm_step_dev with the continuation coefficients
    read from device memory), the all-reduce of the moments over the ranks (on the stream) and the 3x3 solve on the
    device (mcre_lsm_solve_dev).  Same schedule and arithmetic as backward_induction_steps; the host reads the
    coefficients back once at the end instead of once per date (round 1: 0.7 ms of round trip per exercise date).
    -> coefficients [n_reg, 3] in the standardised basis (numpy)."""
    L = B.lib()
    stream = RT.stream_ptr()
    n_reg = len(reg_times)
    n = xs.shape[1]
    reg_idx = {t: k for k, t in enumerate(reg_times)}
    coef = torch.zeros((n_reg, 3), dtype=torch.float64, device=dev)
    value = torch.zeros((1, n), dtype=torch.float32, device=dev)
    n_chunks = (n + chunk_paths - 1) // chunk_paths
    partial = torch.empty(n_chunks * 8 + 1, dtype=torch.float64, device=dev)
    moments = torch.zeros(8, dtype=torch.float64, device=dev)
    xs_ptr, nums_ptr, imm_ptr, coef_ptr, row = xs.data_ptr(), nums.data_ptr(), imm.data_ptr(), coef.data_ptr(), n * 8
    _, world = RT.dist_info()

    def step(k, i):
        args_i = (None, None, None, None, 0.0, 1.0)
        if i is not None:
            ki = reg_idx[ptl[i]]
            cptr = coef_ptr + ki * 24 if i < len(ptl) - 1 else None
            args_i = (xs_ptr + ki * row, nums_ptr + ki * row, imm_ptr + i * row, cptr, float(basis[ki, 0]), float(basis[ki, 1]))
        B.check(L.mcre_lsm_step_dev(xs_ptr + k * row, nums_ptr + k * row, float(basis[k, 0]), float(basis[k, 1]), *args_i,
                                    value.data_ptr(), count, chunk_paths, partial.data_ptr(), moments.data_ptr(), stream))

    last = len(ptl)
    for k in range(n_reg - 1, -1, -1):
        t_reg = reg_times[k]
        pidx = bisect_left(ptl, t_reg)
        if pidx >= len(ptl):
            continue      # after the last exercise date: no continuation value (controller.py:303-305)
        t_next = pidx + 1 if ptl[pidx] == t_reg else pidx
        if t_next < last:
            for i in range(last - 1, t_next, -1):   # product dates that are not regression dates
                step(k, i)
            step(k, t_next)
            last = t_next
        else:
            step(k, None)
        m = RT.all_reduce_tree(moments) if world > 1 else moments
        B.check(L.mcre_lsm_solve_dev(m.data_ptr(), coef_ptr + k * 24, stream))
    return RT.to_host(coef)


def run_backward_inductions(gens):
    """Drive backward_induction_steps generators in lock-step: per round every live generator queues its next
    step, then the moments of all of them are all-reduced over the ranks and read back together.
    -> list of coefficient arrays in the order of `gens`."""
    results = [None] * len(gens)
    pending = {}
    for i, g in enumerate(gens):
        try:
            pending[i] = next(g)
        except StopIteration as e:
            results[i] = e.value
    L = B.lib()
    while pending:
        keys = list(pending)
        deferred = [k for k in keys if isinstance(pending[k], DeferredSteps)]
        if deferred:
            # wave w = the w-th step of every product of the round, one launch per wave; a product's moments are those
            # of its last step
            dev = RT.compute_device()
            stream = RT.stream_ptr()
            first = pending[deferred[0]]
            n_chunks = max((first.count + first.chunk_paths - 1) // first.chunk_paths, 1)
            out_rows = {}
            w = 0
            while True:
                wave = [k for k in deferred if len(pending[k].jobs) > w]
                if not wave:
                    break
                table = np.array([pending[k].jobs[w] for k in wave], dtype=STEP_JOB)
                mom = torch.zeros((len(wave), LSM_MAX_NV), dtype=torch.float64, device=dev)
                partial = torch.empty(n_chunks * len(wave) * LSM_MAX_NV + 1, dtype=torch.float64, device=dev)
                B.check(L.mcre_lsm_step_batch(len(wave), table.ctypes.data, first.count, first.chunk_paths,
                                              partial.data_ptr(), mom.data_ptr(), stream))
                for j, k in enumerate(wave):
                    out_rows[k] = mom[j]
                w += 1
            for k in deferred:
                pending[k] = out_rows[k]
        m = RT.all_reduce_tree(torch.stack([pending[k] for k in keys])).cpu().numpy()      # [K, LSM_MAX_NV]
        G = m[:, [[0, 1, 2], [1, 2, 3], [2, 3, 4]]]
        # one batched solve per state for all products of the round (states a product does not have carry zeros)
        host = np.stack([solve_normal_equations_batch(G, m[:, 5 + 3 * s:8 + 3 * s]) for s in range(LSM_MAX_RIGHTS)], axis=1)
        for j, (k, row) in enumerate(zip(keys, host)):
            try:
                pending[k] = gens[k].send((row, m[j]))
            except StopIteration as e:
                results[k] = e.value
                del pending[k]
    return results


def backward_induction(xs, nums, imm, ptl, reg_times, basis, count, chunk_paths, dev, n_rights=1, tangents=None):
    """One product: see backward_induction_steps."""
    return run_backward_inductions([backward_induction_steps(xs, nums, imm, ptl, reg_times, basis, count, chunk_paths,
                                                             dev, n_rights=n_rights, tangents=tangents)])[0]


def to_raw_basis(coefs, basis, degenerate=None):
    """Coefficients of [1, u, u^2], u = (x - shift) * scale  ->  coefficients of [1, x, x^2].
    `degenerate[k]`: every path has x = shift at date k (t = calibration date); the reference's
    lstsq then returns the minimum-norm solution in the raw basis: c = f * phi / |phi|^2 with
    phi = [1, x, x^2] and f the fitted constant."""
    sh, sc = basis[:, 0], basis[:, 1]
    c0, c1, c2 = coefs[:, 0], coefs[:, 1], coefs[:, 2]
    out = np.empty_like(coefs)
    out[:, 2] = c2 * sc * sc
    out[:, 1] = c1 * sc - 2.0 * c2 * sc * sc * sh
    out[:, 0] = c0 - c1 * sc * sh + c2 * sc * sc * sh * sh
    if degenerate is not None:
        for k in np.nonzero(np.asarray(degenerate))[0]:
            phi = np.array([1.0, sh[k], sh[k] * sh[k]])
            out[k] = coefs[k, 0] * phi / phi.dot(phi)
    return out
