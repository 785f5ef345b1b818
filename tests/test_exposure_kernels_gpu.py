"""The exposure post-processing kernels through the C ABI, against exact references, at the shapes where reductions,
grid caps and compaction go wrong, and with multi-GPU sharding emulated in one process: the radix select and the path
locator (csrc/select.cu), mcre_sum_stats (csrc/util.cu), the netting-set terms, the per-path CVA integrand and the
exposure tangent sums (csrc/equity.cu), and the joint correlated draw (csrc/paths.cu).

References
----------
* Order statistics: numpy.sort of the row (values), and a sort of the order-preserving 64-bit image of the doubles
  (bits: -0.0 sorts before +0.0, like the kernel's keys).  The path of a statistic: the smallest index whose bits equal
  the target.  NaN is out of contract (exposures are finite) and not tested; +-inf, subnormals and both zeros are.
* Sums: math.fsum of the per-path terms, each term computed in numpy with the kernel's own double expressions.
* Netting-set terms: a numpy restatement of products/netting_set.py (threshold dead band, collateral one margin period
  earlier).  The per-path CVA: its FMA chain evaluated exactly with fractions and rounded once per step, which is what
  a correctly rounded FMA gives.
* Tangent sums: the documented rule of include/mcre.h restated in numpy, summed by fsum; on the edges (exposures at
  exactly +-h, U = 0) the derivative torch.autograd gives the reference's expressions.
* Correlated normals: oracle/philox.py (itself pinned to the Random123 vectors by tests/test_philox_host.py) times the
  Cholesky factor in numpy.
* Sharding: paths split as RT.shard_range deals them out; every rank's kernel runs on a contiguous copy of its columns
  (or, for the select, on a pointer offset into the full row), histograms are added, partial sums combined by
  RT.tree_sum, exactly as over several GPUs.

Tolerance model
---------------
* Order statistics and locate: exact (the selected value bit-identical to the bit-order sort, equal to numpy.sort).
* Sums: |got - fsum| <= 1e-13 * fsum(|terms|) per slot (constant CVA weights: times |w|, per-path weights: times lgd).
  Losing or double counting one term moves a sum by far more than this.
* Sharded sums: bit-identical to the single-shard call when every shard but the last holds a power-of-two number of
  chunks (the layouts RT.shard_range promises GPU-count-independent bits for); other layouts are not asserted.
* Netting-set terms: bit-identical, except that the sign of a zero is not compared (with h = 0 the kernel's dead band
  returns +0.0 where the reference passes -0.0 through).  Per-path CVA: bit-identical to the exactly rounded chain.
* Correlated normals: 1e-12 absolute under Philox (device against host libm in Box-Muller, as tests/test_paths_gpu.py);
  1e-15 * sum_j |L_ij z_j| with injected normals (the device may contract into FMAs).

The largest allocation is about 270 MB (the tangents of the 520k-path sharding case); the module stays below 1 GB."""
import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from mcre import binding as B
from mcre import runtime as RT
from mcre.select import select_rows

pytestmark = pytest.mark.gpu

SUM_RTOL = 1e-13
NOT_HERE = -1                      # index buffers are pre-filled with this: an entry the kernel forgets shows


def _sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float64, device="cuda")


def _shards(n, chunk, world):
    return [RT.shard_range(n, chunk, r, world) for r in range(world)]


def _cols(a, begin, count):
    """Contiguous device copy of the last-axis slice [begin, begin + count) (a rank's own arrays); an empty shard gets a
    one-column buffer, like the product's max(count, 1) allocations."""
    if count == 0:
        return torch.zeros(a.shape[:-1] + (1,), dtype=torch.float64, device="cuda")
    return _dev(a[..., begin:begin + count])


def _assert_sum(got, terms, what, scale=1.0):
    ref, mag = math.fsum(terms), math.fsum(np.abs(terms))
    assert abs(got - scale * ref) <= SUM_RTOL * abs(scale) * mag, \
        f"{what}: {got!r} vs fsum {scale * ref!r} (sum |t| {mag:.3e})"


# ---- 1. radix select and locate ------------------------------------------------------------------------------------
def _sel_lib():
    L = B.lib()
    L.mcre_select_create.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    L.mcre_select_destroy.argtypes = [C.c_void_p]
    L.mcre_select_destroy.restype = None
    L.mcre_select_begin.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]
    L.mcre_select_count.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    L.mcre_select_scan.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    L.mcre_select_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.mcre_select_compact.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p]
    return L


def _key_sorted(row):
    """The row sorted in the order of the kernel's keys (IEEE total order on finite values, infinities and both
    zeros: -0.0 before +0.0)."""
    u = _bits(row).view(np.uint64)
    sign = np.uint64(1) << np.uint64(63)
    key = np.where(u >> np.uint64(63) != 0, ~u, u | sign)
    k = np.sort(key)
    return np.where(k >> np.uint64(63) != 0, k & ~sign, ~k).view(np.float64)


def _assert_selected(got, rows, ranks, what):
    """got [n_rows, R] against numpy.sort (values) and the key-order sort (bits)."""
    for i, row in enumerate(rows):
        want_v = np.sort(row)[ranks[i]]
        want_b = _key_sorted(row)[ranks[i]]
        assert np.array_equal(got[i], want_v), f"{what} row {i}: {got[i]} vs sort {want_v} at ranks {ranks[i]}"
        assert np.array_equal(_bits(got[i]), _bits(want_b)), f"{what} row {i}: bits {got[i]} vs {want_b}"


def _first_index(row, target):
    hit = np.nonzero(_bits(row) == _bits(np.float64(target)))[0]
    return int(hit[0]) if hit.size else None


def _locate(x, offset, row_stride, n_local, targets):
    """mcre_select_locate on rows starting `offset` elements into each row of x -> host int64 [n_rows]."""
    n_rows = len(targets)
    t = _dev(np.asarray(targets, dtype=np.float64))
    idx = torch.full((n_rows,), NOT_HERE, dtype=torch.int64, device="cuda")
    B.check(B.lib().mcre_select_locate(x.data_ptr() + 8 * offset, row_stride, n_local, n_rows, t.data_ptr(),
                                       idx.data_ptr(), RT.stream_ptr()))
    return idx.cpu().numpy()


def _select_sharded(x, n, ranks, parts):
    """The select of mcre/select.py over emulated ranks: each (begin, count) of `parts` gets its own plan and reads its
    slice of every row of x [n_rows][n] by pointer offset (row_stride n); the histograms of a pass are summed over the
    ranks before every plan scans; compaction after pass 1 is local.  -> [rank][n_rows, R]."""
    L = _sel_lib()
    st = RT.stream_ptr()
    rows, R = ranks.shape
    rk = np.ascontiguousarray(ranks, dtype=np.int64)
    plans = []
    try:
        for _ in parts:
            p = C.c_void_p()
            B.check(L.mcre_select_create(rows, R, C.byref(p)))
            plans.append(p)
            B.check(L.mcre_select_begin(p, rk.ctypes.data_as(C.POINTER(C.c_int64)), st))
        hists = [torch.zeros(rows * R * 256, dtype=torch.int64, device="cuda") for _ in parts]
        for ps in range(8):
            for p, h, (b, c) in zip(plans, hists, parts):
                B.check(L.mcre_select_count(p, x.data_ptr() + 8 * b, n, c, ps, h.data_ptr(), st))
            total = torch.stack(hists).sum(dim=0)
            for p in plans:
                B.check(L.mcre_select_scan(p, ps, total.data_ptr(), st))
            if ps == 1:
                for p, (b, c) in zip(plans, parts):
                    B.check(L.mcre_select_compact(p, x.data_ptr() + 8 * b, n, c, 2, st))
            torch.cuda.synchronize()
        outs = []
        for p in plans:
            out = _nan(rows * R)
            B.check(L.mcre_select_finish(p, out.data_ptr(), st))
            outs.append(out.cpu().numpy().reshape(rows, R))
        return outs
    finally:
        for p in plans:
            L.mcre_select_destroy(p)


def _value_rows(n, rng):
    """One row per value class -> [rows, n] float64."""
    z = rng.standard_normal((8, n))
    rows = [
        z[0] * 3.0,                                            # plain
        np.round(z[1] * 4.0) / 4.0,                            # heavy ties
        np.full(n, 3.25),                                      # all equal
        -np.abs(z[2]) * 1e-3 - 1e-300,                         # negatives only
        rng.integers(-3000, 3000, n) * 5e-324,                 # subnormals (and +0.0)
        np.where(rng.random(n) < 0.05, np.where(z[3] > 0, np.inf, -np.inf), z[3] * 1e300),  # +-inf and huge
        np.where(rng.random(n) < 0.5, -0.0, 0.0),              # both zeros only
        np.where(rng.random(n) < 0.4, np.where(rng.random(n) < 0.5, -0.0, 0.0), z[4]),    # zeros in a spread row
    ]
    out = np.stack(rows)
    if n >= 3:
        out[6, 0] = 0.0                                        # +0.0 before the first -0.0: matching by value would
        out[6, 1:3] = -0.0                                     # find path 0 for the target -0.0
        out[7, 0], out[7, 1] = 0.0, -0.0
    return out


def _rank_rows(n, R, n_rows, rng):
    """Per row R ranks (R = 1..4): rank 0, n - 1, repeated ranks, neighbours of a quantile rank."""
    out = []
    for i in range(n_rows):
        k = int(rng.integers(n))
        cand = [[0, n - 1, k, k], [k, k, min(k + 1, n - 1), max(k - 1, 0)], [n - 1, 0, n // 2, n - 1]][i % 3]
        out.append(cand[:R])
    return np.array(out, dtype=np.int64)


def _padded(rows, n, stride, fill):
    """[n_rows, stride] device buffer: rows in [:, :n], the padding behind n_local cycles through `fill` [n_rows, k]."""
    buf = np.empty((rows.shape[0], stride))
    buf[:, :n] = rows
    if stride > n:
        k = fill.shape[1]
        buf[:, n:] = fill[:, np.arange(stride - n) % k]
    return _dev(buf)


ABSENT = 12345.678                 # in the padding of every row, never among its values


@pytest.mark.parametrize("R", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [1, 2, 255, 2049, 65535, 65536, 66536, 100003])
def test_select_matches_sort_on_strided_rows(n, R):
    """Every value class, R = 1..4 ranks per row incl. rank 0, n - 1 and repeated ranks, n_local on both sides of the
    compaction threshold 65536 and not a multiple of 256 or 2048.  Rows are strided, and the padding behind n_local
    holds +-inf, +-huge, +-tiny, the wanted statistics and a value absent from the row: reading it changes answers."""
    rng = np.random.default_rng(n * 7 + R)
    rows = _value_rows(n, rng)
    ranks = _rank_rows(n, R, rows.shape[0], rng)
    want = np.stack([np.sort(r)[k] for r, k in zip(rows, ranks)])
    fill = np.concatenate([np.tile([np.inf, -np.inf, 1e308, -1e308, 5e-324, -5e-324, -0.0, 0.0, ABSENT],
                                   (rows.shape[0], 1)), want], axis=1)
    x = _padded(rows, n, n + 61, fill)
    got = select_rows(x, n, ranks)
    _assert_selected(got, rows, ranks, f"n={n} R={R}")
    # the path of each statistic: smallest index with those bits, padding never found
    for r in range(R):
        idx = _locate(x, 0, x.stride(0), n, got[:, r])
        for i in range(rows.shape[0]):
            assert idx[i] == _first_index(rows[i], got[i, r]), f"n={n} row {i} rank {ranks[i, r]}: index {idx[i]}"
    idx = _locate(x, 0, x.stride(0), n, np.full(rows.shape[0], ABSENT))
    assert np.all(idx >= n), f"n={n}: a target held only by the padding was found at {idx}"


def test_locate_tells_the_two_zeros_apart():
    """+0.0 at index 0, the first -0.0 at index 1 (and many of both later): the target -0.0 is path 1, +0.0 path 0;
    ties resolve to the smallest index."""
    n = 70001
    rng = np.random.default_rng(3)
    row = np.where(rng.random(n) < 0.5, -0.0, 0.0)
    row[0], row[1] = 0.0, -0.0
    row2 = np.round(rng.standard_normal(n) * 2.0) / 2.0     # heavy ties
    x = _dev(np.stack([row, row2]))
    n_neg = int(np.sum(np.signbit(row)))
    got = select_rows(x, n, np.array([[0, n_neg - 1, n_neg, n - 1], [0, n // 3, n // 2, n - 1]], dtype=np.int64))
    assert _bits(got[0]).tolist() == _bits([-0.0, -0.0, 0.0, 0.0]).tolist(), got[0]
    idx = _locate(x, 0, n, n, [-0.0, row2[n // 2]])
    assert idx[0] == 1 and idx[1] == _first_index(row2, row2[n // 2])
    idx = _locate(x, 0, n, n, [0.0, 0.5])
    assert idx[0] == 0 and idx[1] == _first_index(row2, 0.5)


def _n_flushes_of_block0(n, n_rows, candidate):
    """In-loop flushes of the staging buffer of block 0 of select_compact_kernel (4 x 256 elements per iteration,
    flush when more than 1024 are staged) for a row whose candidates are the mask `candidate`."""
    bx = min(-(-n // 2048), _sm_count() * 16 // n_rows + 1)
    stride = bx * 256
    staged = flushes = 0
    for base in range(0, n, 4 * stride):
        for j in range(4):
            i0 = base + j * stride
            staged += int(candidate[i0:min(i0 + 256, n)].sum())
        if staged > 2048 - 4 * 256:
            flushes, staged = flushes + 1, 0
    return flushes, bx


def test_select_compaction_at_its_capacity_and_with_repeated_flushes():
    """n_local = 2^19 + 77, 40 rows (so that the grid is capped and blocks loop):  row 0 has exactly
    n_local / 8 + 1024 candidates sharing the wanted 16-bit prefix (the compacted copy is used), row 1 one more (full
    reads), row 2 its candidates on block 0's elements, which flushes its staging buffer several times inside the loop;
    the other rows are plain.  Single shard and two emulated ranks."""
    n, n_rows = (1 << 19) + 77, 40
    cap = n // 8 + 1024
    rng = np.random.default_rng(11)
    x = rng.standard_normal((n_rows, n)) * 4.0 + 9.0
    lo, hi = 1.0, np.nextafter(1.0625, 0.0)      # [1, 1.0625): one 16-bit key prefix (sign, exponent, 4 bits)
    ranks = np.empty((n_rows, 3), dtype=np.int64)
    bx = None
    for r in range(n_rows):
        row = x[r]
        if r < 3:
            row[:] = np.where(rng.random(n) < 0.5, rng.uniform(-5.0, 0.99, n), rng.uniform(1.07, 5.0, n))
            if r < 2:
                sel = rng.choice(n, cap + r, replace=False)
            else:
                mask = (np.arange(n) % (min(-(-n // 2048), _sm_count() * 16 // n_rows + 1) * 256)) < 256
                sel = np.nonzero(mask)[0]
                assert sel.size <= cap
            row[sel] = np.minimum(rng.uniform(lo, hi, sel.size), hi)
            row[sel[::7]] = 1.03125                # ties inside the group
            below = int(np.sum(row < lo))
            ranks[r] = [below, below + sel.size // 2, below + sel.size - 1]
            if r == 2:
                cand = np.zeros(n, dtype=bool)
                cand[sel] = True
                flushes, bx = _n_flushes_of_block0(n, n_rows, cand)
                assert flushes >= 3, f"row 2 flushes block 0's staging buffer only {flushes} times (grid {bx})"
        else:
            k = int(rng.integers(1, n - 1))
            ranks[r] = [k - 1, k, k + 1]
    xd = _dev(x)
    got = select_rows(xd, n, ranks)
    _assert_selected(got, x, ranks, "compaction")
    for g in _select_sharded(xd, n, ranks, _shards(n, 4096, 2)):
        assert np.array_equal(_bits(g), _bits(got))


@pytest.mark.parametrize("n_rows, n", [(1, 300007), (7, 4097), (37, (1 << 18) + 3), (None, 3001)])
def test_select_past_the_grid_cap(n_rows, n):
    """1 row, a non-power-of-two row count, and more rows than the grid cap sm_count * 16 / n_rows + 1 gives more
    than one block (n_rows None: sm_count * 16 + 5 rows, one block per row)."""
    if n_rows is None:
        n_rows = _sm_count() * 16 + 5
    rng = np.random.default_rng(n_rows)
    x = np.round(rng.standard_normal((n_rows, n)) * 50.0) / 8.0
    ranks = np.stack([rng.integers(0, n, 3) for _ in range(n_rows)]).astype(np.int64)
    ranks[0] = [0, n // 2, n - 1]
    xd = _dev(x)
    got = select_rows(xd, n, ranks)
    _assert_selected(got, x, ranks, f"{n_rows} rows")
    idx = _locate(xd, 0, n, n, got[:, 1])
    want = [_first_index(x[i], got[i, 1]) for i in range(n_rows)]
    assert idx.tolist() == want


#: (world, n, chunk): ranks that compact (>= 65536 paths) and ranks that do not, one exactly at 65536, empty ranks
SHARD_CASES = [(1, 100003, 4096), (2, 126000, 4096), (3, 300007, 4096), (4, 9 * 32768 - 5000, 32768),
               (8, 24 * 16384 + 777, 16384)]


@pytest.mark.parametrize("world, n, chunk", SHARD_CASES)
def test_select_and_locate_over_emulated_ranks(world, n, chunk):
    """Every rank's finish equals the single-shard select bit for bit and the sort; the smallest global index over
    the ranks that find a statistic is the smallest global index among its ties (mcre/hybrid.py)."""
    parts = _shards(n, chunk, world)
    counts = [c for _, c in parts]
    rng = np.random.default_rng(world * 1000 + n % 1000)
    rows = _value_rows(n, rng)
    qi = int(0.95 * n)
    ranks = np.tile(np.array([qi - 1, qi, qi + 1], dtype=np.int64), (rows.shape[0], 1))
    ranks[0] = [0, 1, n - 1]
    ranks[6] = [n // 2 - 1, n // 2, n // 2 + 1]
    x = _dev(rows)
    single = select_rows(x, n, ranks)
    _assert_selected(single, rows, ranks, f"world={world}")
    for r, g in enumerate(_select_sharded(x, n, ranks, parts)):
        assert np.array_equal(_bits(g), _bits(single)), f"world={world} rank {r} (counts {counts})"
    for k in range(3):
        best = np.full(rows.shape[0], np.iinfo(np.int64).max)
        for b, c in parts:
            idx = _locate(x, b, n, c, single[:, k])
            assert np.all(idx >= 0) and (c > 0 or np.all(idx >= c)), f"world={world}: rank [{b}, {b + c}) {idx}"
            best = np.where(idx < c, np.minimum(best, idx + b), best)
        want = [_first_index(rows[i], single[i, k]) for i in range(rows.shape[0])]
        assert best.tolist() == want, f"world={world} rank slot {k}"


def test_locate_without_paths_and_select_of_an_empty_rank():
    """n_local = 0: locate reports "not here" and writes every row; count adds nothing to the histogram."""
    x = _dev(np.arange(10.0).reshape(2, 5))
    idx = _locate(x, 0, 5, 0, [1.0, 2.0])
    assert np.all(idx >= 0), idx
    L = _sel_lib()
    p = C.c_void_p()
    B.check(L.mcre_select_create(2, 1, C.byref(p)))
    try:
        rk = np.zeros(2, dtype=np.int64)
        B.check(L.mcre_select_begin(p, rk.ctypes.data_as(C.POINTER(C.c_int64)), RT.stream_ptr()))
        h = torch.full((2 * 256,), 7, dtype=torch.int64, device="cuda")
        B.check(L.mcre_select_count(p, x.data_ptr(), 5, 0, 0, h.data_ptr(), RT.stream_ptr()))
        assert int(h.abs().sum()) == 0
    finally:
        L.mcre_select_destroy(p)


# ---- 2. mcre_sum_stats ---------------------------------------------------------------------------------------------
def _stats_terms(x, shift, mode):
    v = x if mode == 0 else (np.maximum(x, 0.0) if mode == 1 else -np.maximum(-x, 0.0))
    d = v - shift[:, None]
    return d, d * d


def _sum_stats(x, shift, mode, chunk):
    """x: device [n_rows][n] -> host [n_rows][2]."""
    n_rows, n = x.shape
    out = _nan(n_rows * 2)
    partial = _nan(max(-(-n // chunk), 1) * n_rows * 2 + 1)
    B.check(B.lib().mcre_sum_stats(x.data_ptr(), n, n_rows, chunk, shift.data_ptr(), mode, partial.data_ptr(),
                                   out.data_ptr(), RT.stream_ptr()))
    return out.cpu().numpy().reshape(n_rows, 2)


def _stats_data(n_rows, n, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n_rows, n)) * rng.uniform(0.5, 50.0, (n_rows, 1)) + rng.uniform(-5.0, 5.0, (n_rows, 1))
    x[:, ::11] = 0.0
    shift = rng.uniform(-3.0, 3.0, n_rows)
    return x, shift


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("chunk", [32, 96, 256, 4096])
def test_sum_stats_matches_fsum(chunk, mode):
    """Modes 0 / 1 / 2 with a non-zero shift per row; n from 1 path to past 64 chunks (two tree levels; chunk 32 and
    96: past 2048 chunks, three levels); 67 rows at one size."""
    sizes = [(5, 1), (5, chunk - 1), (5, chunk + 1), (67, 3 * chunk + 7), (3, 70 * chunk + 5)]
    if chunk <= 96:
        sizes.append((3, 2100 * chunk + 31))
    for n_rows, n in sizes:
        x, shift = _stats_data(n_rows, n, seed=chunk * 10 + n % 1000 + mode)
        got = _sum_stats(_dev(x), _dev(shift), mode, chunk)
        t1, t2 = _stats_terms(x, shift, mode)
        for r in range(n_rows):
            what = f"chunk={chunk} mode={mode} n={n} row {r}"
            _assert_sum(got[r, 0], t1[r], what + " sum")
            _assert_sum(got[r, 1], t2[r], what + " sum of squares")


#: (n, chunk, worlds): every rank but the last holds a power-of-two number of chunks (2^k - 1 chunks: a ragged last
#: rank at every world, a ragged last chunk, two tree levels); 13 chunks over 8 ranks: the last rank is empty
SUM_SHARD_CASES = [(2046 * 32 + 17, 32, (1, 2, 4, 8)), (2046 * 96 + 50, 96, (1, 2, 4, 8)),
                   (126 * 256 + 100, 256, (1, 2, 4, 8)), (126 * 4096 + 99, 4096, (1, 2, 4, 8)),
                   (12 * 256 + 251, 256, (1, 8))]


def _tree(parts):
    return RT.tree_sum(parts)


@pytest.mark.parametrize("n, chunk, worlds", SUM_SHARD_CASES)
def test_sum_stats_is_bit_identical_over_emulated_ranks(n, chunk, worlds):
    """Per rank a contiguous copy of its columns, its own call, the partial results combined by RT.tree_sum: bit for
    bit the single-shard result."""
    x, shift = _stats_data(6, n, seed=n % 9973)
    sd = _dev(shift)
    for mode in (0, 1, 2):
        single = _sum_stats(_dev(x), sd, mode, chunk)
        for world in worlds:
            parts = _shards(n, chunk, world)
            n_ch = [-(-c // chunk) for _, c in parts]
            assert all(k & (k - 1) == 0 for k in n_ch[:-1]), n_ch
            outs = []
            for b, c in parts:
                xs = _cols(x, b, c)
                outs.append(_sum_stats(xs, sd, mode, chunk) if c else _sum_stats_empty(xs, sd, mode, chunk))
            got = _tree(outs)
            assert np.array_equal(_bits(got), _bits(single)), f"n={n} chunk={chunk} mode={mode} world={world}"


def _sum_stats_empty(x, shift, mode, chunk):
    n_rows = x.shape[0]
    out = _nan(n_rows * 2)
    partial = _nan(n_rows * 2 + 1)
    B.check(B.lib().mcre_sum_stats(x.data_ptr(), 0, n_rows, chunk, shift.data_ptr(), mode, partial.data_ptr(),
                                   out.data_ptr(), RT.stream_ptr()))
    return out.cpu().numpy().reshape(n_rows, 2)


def test_sum_stats_without_paths_and_bad_chunks():
    x, shift = _dev(np.ones((3, 4))), _dev(np.ones(3))
    for mode in (0, 1, 2):
        assert np.array_equal(_sum_stats_empty(x, shift, mode, 32), np.zeros((3, 2)))
    out, partial = _nan(6), _nan(64)
    for chunk in (0, -32, 48, 100, 31):
        rc = B.lib().mcre_sum_stats(x.data_ptr(), 4, 3, chunk, shift.data_ptr(), 0, partial.data_ptr(), out.data_ptr(),
                                    RT.stream_ptr())
        assert rc < 0, f"chunk {chunk} accepted"


# ---- 3. netting-set terms and the per-path CVA integrand -----------------------------------------------------------
def _thr(x, h):
    return np.where(x > h, x - h, np.where(x < -h, x + h, 0.0))


def _unsec_ref(expo, me, lag, coll, h):
    """products/netting_set.py:compute_unsecured_exposure_profiles with explicit metric / delayed indices."""
    out = []
    for m, xe in enumerate(me):
        now = expo[xe]
        if not coll:
            out.append(now if h == 0.0 else _thr(now, h))
        else:
            delayed = expo[xe - lag[m]] if lag[m] >= 0 else None
            coll_m = np.zeros_like(now) if delayed is None else (delayed if h == 0.0 else _thr(delayed, h))
            out.append(now - coll_m)
    return np.stack(out)


#: exposure index of each metric date (not the metric index) and the lags of a collateralised set (-1: none yet)
METRIC_EXPO = np.array([0, 2, 3, 5, 7, 8], dtype=np.int32)
LAGS = np.array([-1, 0, 1, 4, 2, 3], dtype=np.int32)
N_EXPO = 9


def _expo_data(n, h, seed):
    """[N_EXPO][n] exposures with values at exactly +-h, one ulp inside and outside, and exact zeros."""
    rng = np.random.default_rng(seed)
    e = rng.standard_normal((N_EXPO, n)) * 3.0
    edges = np.array([h, -h, np.nextafter(h, np.inf), np.nextafter(h, 0.0), np.nextafter(-h, -np.inf),
                      np.nextafter(-h, 0.0), 0.0, -0.0])
    pick = rng.random((N_EXPO, n)) < 0.25
    e[pick] = edges[rng.integers(0, edges.size, int(pick.sum()))]
    return e


@pytest.mark.parametrize("coll", [0, 1])
@pytest.mark.parametrize("h", [0.0, 0.75])
def test_unsecured_exposures_are_bit_identical_to_netting_set(coll, h):
    n = 3001
    expo = _expo_data(n, h, seed=int(h * 4) + 2 * coll)
    lag = LAGS if coll else np.full(METRIC_EXPO.size, -1, dtype=np.int32)
    out, ed = _nan(METRIC_EXPO.size, n), _dev(expo)
    me_k, me_p = B.as_ip(METRIC_EXPO)
    lg_k, lg_p = B.as_ip(lag)
    B.check(B.lib().mcre_eq_unsecured_exposures(ed.data_ptr(), n, METRIC_EXPO.size, me_p, lg_p, coll, h,
                                                out.data_ptr(), RT.stream_ptr()))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    want = _unsec_ref(expo, METRIC_EXPO, lag, coll, h)
    assert np.array_equal(got, want), f"coll={coll} h={h}: {np.sum(got != want)} values differ"
    nz = want != 0.0
    assert np.array_equal(_bits(got[nz]), _bits(want[nz]))


def _cva_chain(unsec, w, lgd):
    """fma(max(u, 0), w, tot) over m < n_metric - 1, each step rounded once, then * lgd."""
    n_metric, n = unsec.shape
    out = np.empty(n)
    for p in range(n):
        tot = 0.0
        for m in range(n_metric - 1):
            tot = float(Fraction(max(float(unsec[m, p]), 0.0)) * Fraction(float(w[m, p])) + Fraction(tot))
        out[p] = tot * lgd
    return out


@pytest.mark.parametrize("n_metric", [1, 2, 6])
def test_cva_paths_is_bit_identical_to_the_exactly_rounded_fma_chain(n_metric):
    n, lgd = 2999, 0.6
    rng = np.random.default_rng(n_metric)
    unsec = rng.standard_normal((n_metric, n)) * np.geomspace(1e-3, 1e3, n)
    w = rng.uniform(0.0, 0.05, (n_metric, n))
    w[-1] = 1e6                                  # the last metric date must not contribute
    out, ud, wd = _nan(n), _dev(unsec), _dev(w)
    B.check(B.lib().mcre_eq_cva_paths(ud.data_ptr(), wd.data_ptr(), n, n_metric, lgd, out.data_ptr(), RT.stream_ptr()))
    got = out.cpu().numpy()
    want = _cva_chain(unsec, w, lgd)
    if n_metric == 1:
        assert np.array_equal(got, np.zeros(n))
    bad = np.nonzero(_bits(got) != _bits(want))[0]
    assert bad.size == 0, f"n_metric={n_metric}: {bad.size} paths differ, first {bad[0]}: {got[bad[0]]!r} vs {want[bad[0]]!r}"


# ---- 4. exposure tangent sums --------------------------------------------------------------------------------------
def _tangent_ref(expo, tan, me, lag, coll, h, n_par, w=None, wp=None, lgd=None, wt=None):
    """-> dict of term arrays per (m, g, slot) and the scale of slot 2, by the rule of include/mcre.h."""
    n_wtan = 0 if wt is None else wt.shape[1]
    terms = {}
    for m, xe in enumerate(me):
        now = expo[xe]
        l = lag[m] if coll else -1
        delayed = expo[xe - l] if l >= 0 else np.zeros_like(now)
        u = now - _thr(delayed, h) if coll else _thr(now, h)
        dthr = lambda x: ((x > h) | (x < -h)).astype(np.float64)
        pos, neg = u > 0.0, u < 0.0
        for g in range(n_par):
            dnow = tan[g, xe]
            if coll:
                ddel = tan[g, xe - l] if l >= 0 else np.zeros_like(now)
                du = dnow - dthr(delayed) * ddel
            else:
                du = dthr(now) * dnow
            terms[m, g, 0], terms[m, g, 1] = du[pos], du[neg]
            terms[m, g, 2] = (du * wp[m])[pos] if wp is not None else du[pos]
        for j in range(n_wtan):
            terms[m, n_par + j, 2] = (u * wt[m, j])[pos]
    return terms


def _tangent_sums(expo, tan, n, n_par, coll, h, chunk, w=None, wp=None, lgd=0.0, wt=None, me=METRIC_EXPO, lag=LAGS):
    """Device arrays in -> host [n_metric][n_par + n_wtan][3]."""
    n_metric = len(me)
    n_wtan = 0 if wt is None else int(wt.shape[1])
    rows = n_par + n_wtan
    out = _nan(n_metric * rows * 3)
    partial = _nan(max(-(-n // chunk), 1) * n_metric * rows * 3 + 1)
    me_k, me_p = B.as_ip(me)
    lg_k, lg_p = B.as_ip(lag)
    L = B.lib()
    if wp is None:
        w_k, w_p = B.as_dp(w)
        B.check(L.mcre_exposure_tangent_sums(expo.data_ptr(), tan.data_ptr(), n, N_EXPO, n_par, n_metric, me_p, lg_p,
                                             coll, h, w_p, chunk, partial.data_ptr(), out.data_ptr(), RT.stream_ptr()))
    else:
        B.check(L.mcre_exposure_tangent_sums_paths(expo.data_ptr(), tan.data_ptr(), n, N_EXPO, n_par, n_metric, me_p,
                                                   lg_p, coll, h, wp.data_ptr(), lgd,
                                                   wt.data_ptr() if wt is not None else None, n_wtan, chunk,
                                                   partial.data_ptr(), out.data_ptr(), RT.stream_ptr()))
    return out.cpu().numpy().reshape(n_metric, rows, 3)


def _tangent_data(n, n_par, h, seed, n_wtan=4):
    rng = np.random.default_rng(seed)
    expo = _expo_data(n, h, seed)
    tan = rng.standard_normal((n_par, N_EXPO, n)) * rng.uniform(0.1, 10.0, (n_par, 1, 1))
    w = rng.uniform(0.001, 0.05, METRIC_EXPO.size)
    wp = rng.uniform(0.0, 0.05, (METRIC_EXPO.size, n))
    wt = rng.standard_normal((METRIC_EXPO.size, n_wtan, n)) * 0.01
    return expo, tan, w, wp, wt


def _check_tangents(got, terms, n_par, w, wp, lgd, wt, what):
    n_wtan = 0 if wt is None else wt.shape[1]
    for m in range(METRIC_EXPO.size):
        for g in range(n_par):
            _assert_sum(got[m, g, 0], terms[m, g, 0], f"{what} m={m} g={g} pos")
            _assert_sum(got[m, g, 1], terms[m, g, 1], f"{what} m={m} g={g} neg")
            _assert_sum(got[m, g, 2], terms[m, g, 2], f"{what} m={m} g={g} cva", scale=lgd if wp is not None else w[m])
        for j in range(n_wtan):
            assert got[m, n_par + j, 0] == 0.0 and got[m, n_par + j, 1] == 0.0, f"{what} m={m} credit row {j}"
            _assert_sum(got[m, n_par + j, 2], terms[m, n_par + j, 2], f"{what} m={m} credit row {j}", scale=lgd)


@pytest.mark.parametrize("weights", ["constant", "per_path"])
@pytest.mark.parametrize("coll", [0, 1])
@pytest.mark.parametrize("n_par", [1, 7])
@pytest.mark.parametrize("chunk", [256, 4096])
def test_exposure_tangent_sums_match_fsum(chunk, n_par, coll, weights):
    """Constant weights (slot 2 = w_m * slot 0) and per-path weights with 4 credit rows (slot 2 = lgd * sum relu(U)
    dw, slots 0 and 1 exactly 0); the delayed exposure's tangent enters with a minus sign; n across chunk edges and past
    64 chunks (two tree levels)."""
    h = 0.75
    lgd = 0.6
    for n in (1, chunk - 1, chunk + 1, 3 * chunk + 7) + ((67 * chunk + 3,) if chunk == 256 else ()):
        expo, tan, w, wp, wt = _tangent_data(n, n_par, h, seed=n % 1000 + n_par + 10 * coll)
        if weights == "constant":
            wp_, wt_ = None, None
        else:
            wp_, wt_ = wp, wt
        got = _tangent_sums(_dev(expo), _dev(tan), n, n_par, coll, h, chunk, w=w,
                            wp=None if wp_ is None else _dev(wp_), lgd=lgd, wt=None if wt_ is None else _dev(wt_))
        terms = _tangent_ref(expo, tan, METRIC_EXPO, LAGS, coll, h, n_par, w=w, wp=wp_, lgd=lgd, wt=wt_)
        _check_tangents(got, terms, n_par, w, wp_, lgd, wt_, f"chunk={chunk} n={n} n_par={n_par} coll={coll}")


def _torch_edge(now, delayed, dnow, ddel, coll, h):
    """(d relu(U), d -relu(-U)) by torch.autograd through the reference's expressions, one path."""
    t = torch.zeros((), dtype=torch.float64, requires_grad=True)
    e_now = torch.tensor(now, dtype=torch.float64) + t * dnow
    e_del = torch.tensor(delayed, dtype=torch.float64) + t * ddel

    def thr(x):
        return torch.where(x > h, x - h, torch.where(x < -h, x + h, torch.zeros_like(x)))
    u = e_now - thr(e_del) if coll else thr(e_now)
    gp, = torch.autograd.grad(torch.relu(u), t, retain_graph=True)
    gn, = torch.autograd.grad(-torch.relu(-u), t)
    return float(gp), float(gn)


def test_exposure_tangent_edges_follow_torch():
    """One path per call: exposures at exactly +-h, one ulp outside, U == 0 exactly.  dthr is 0 at +-h (seen only in a
    collateralised set whose delayed exposure sits on the edge while U != 0), relu' is 0 at U = 0, and a path with
    U == 0 counts in neither sum."""
    h = 0.75
    up, dn = np.nextafter(h, np.inf), np.nextafter(-h, -np.inf)
    cases = [  # (coll, now, delayed, dnow, ddel)
        (0, h, 0.0, 2.0, 0.0), (0, -h, 0.0, 2.0, 0.0), (0, up, 0.0, 2.0, 0.0), (0, dn, 0.0, 2.0, 0.0),
        (0, 0.3, 0.0, 2.0, 0.0), (0, 5.0, 0.0, 2.0, 0.0),
        (1, 5.0, h, 2.0, 3.0), (1, -5.0, -h, 2.0, 3.0), (1, 5.0, up, 2.0, 3.0), (1, -5.0, dn, 2.0, 3.0),
        (1, 5.0 - h, 5.0, 2.0, 3.0), (1, 0.0, 0.3, 2.0, 3.0), (1, 1.0, 0.3, 2.0, 3.0),
    ]
    me, lag = np.array([1], dtype=np.int32), np.array([1], dtype=np.int32)
    for coll, now, delayed, dnow, ddel in cases:
        expo = np.array([[delayed], [now]] + [[0.0]] * (N_EXPO - 2))
        tan = np.zeros((1, N_EXPO, 1))
        tan[0, 0, 0], tan[0, 1, 0] = ddel, dnow
        got = _tangent_sums(_dev(expo), _dev(tan), 1, 1, coll, h, 256, w=np.array([0.5]), me=me, lag=lag)[0, 0]
        gp, gn = _torch_edge(now, delayed, dnow, ddel, coll, h)
        what = f"coll={coll} now={now!r} delayed={delayed!r}"
        assert got[0] == gp and got[1] == gn and got[2] == 0.5 * gp, f"{what}: {got.tolist()} vs torch {gp}, {gn}"
        u = now - float(_thr(np.array(delayed), h)) if coll else float(_thr(np.array(now), h))
        if u == 0.0:
            assert got[0] == 0.0 and got[1] == 0.0, what


#: (n, chunk, worlds) as for mcre_sum_stats
TAN_SHARD_CASES = [(126 * 256 + 100, 256, (1, 2, 4, 8)), (127 * 4096 - 1, 4096, (1, 2, 4, 8)),
                   (12 * 256 + 251, 256, (1, 8))]


@pytest.mark.parametrize("n, chunk, worlds", TAN_SHARD_CASES)
def test_exposure_tangent_sums_are_bit_identical_over_emulated_ranks(n, chunk, worlds):
    """Contiguous per-rank copies of exposures, tangents, per-path weights and weight tangents; RT.tree_sum of the rank
    results equals the single-shard call bit for bit, and matches fsum; an empty rank gives zeros."""
    n_par, h, lgd = 7, 0.75, 0.6
    expo, tan, w, wp, wt = _tangent_data(n, n_par, h, seed=n % 977)
    for coll, per_path in ((1, True), (0, False)):
        kw = dict(wp=wp, wt=wt) if per_path else {}

        def run(b, c):
            dv = {k: _cols(v, b, c) for k, v in kw.items()}
            return _tangent_sums(_cols(expo, b, c), _cols(tan, b, c), c, n_par, coll, h, chunk, w=w, lgd=lgd, **dv)
        single = run(0, n)
        terms = _tangent_ref(expo, tan, METRIC_EXPO, LAGS, coll, h, n_par, w=w, lgd=lgd, **kw)
        _check_tangents(single, terms, n_par, w, kw.get("wp"), lgd, kw.get("wt"), f"n={n} chunk={chunk} coll={coll}")
        for world in worlds:
            outs = [run(b, c) for b, c in _shards(n, chunk, world)]
            for (b, c), o in zip(_shards(n, chunk, world), outs):
                if c == 0:
                    assert np.array_equal(o, np.zeros_like(o)), "an empty rank must give zeros"
            got = _tree(outs)
            assert np.array_equal(_bits(got), _bits(single)), f"n={n} chunk={chunk} coll={coll} world={world}"


# ---- 5. correlated normals -----------------------------------------------------------------------------------------
def _chol(dim, seed):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((dim, dim + 2))
    c = a @ a.T
    d = np.sqrt(np.diag(c))
    return np.linalg.cholesky(c / np.outer(d, d))


def _correlated(rng, n_sub, dim, chol, n):
    out = _nan(max(n_sub, 1), n, dim)
    ck, cp = B.as_dp(chol)
    rc = B.lib().mcre_correlated_normals(C.byref(rng), n_sub, dim, cp, n, out.data_ptr(), RT.stream_ptr())
    return rc, out


@pytest.mark.parametrize("dim", [1, 2, 3, 7, 16])
def test_correlated_normals_philox_matches_oracle(dim):
    """Several sub-steps (odd dims: the spare normal of a Box-Muller pair crosses a sub-step), a non-zero stream, n not
    a multiple of the 128-thread block."""
    from oracle import philox
    n, n_sub, seed, stream = 1000, 5, 42, 3
    chol = _chol(dim, dim)
    rng = B.Rng()
    rng.mode, rng.seed, rng.stream, rng.n_paths_total = B.RNG_PHILOX, seed, stream, n
    rc, out = _correlated(rng, n_sub, dim, chol, n)
    B.check(rc)
    want = philox.normals(np.arange(n, dtype=np.uint64), n_sub, dim, seed, stream) @ chol.T
    err = np.max(np.abs(out.cpu().numpy() - want))
    assert err <= 1e-12, f"dim={dim}: max abs error {err:.3e}"


@pytest.mark.parametrize("dim", [1, 3, 16])
def test_correlated_normals_inject_matches_numpy(dim):
    n, n_total, n_sub = 1000, 1003, 4
    chol = _chol(dim, 100 + dim)
    z = np.random.default_rng(dim).standard_normal((n_sub, n_total, dim))
    zd = _dev(z)
    rng = B.Rng()
    rng.mode, rng.d_z, rng.n_paths_total = B.RNG_INJECT, zd.data_ptr(), n_total
    rc, out = _correlated(rng, n_sub, dim, chol, n)
    B.check(rc)
    zs = z[:, :n]
    want = zs @ chol.T
    tol = 1e-15 * (np.abs(zs) @ np.abs(chol).T)
    err = np.abs(out.cpu().numpy() - want)
    assert np.all(err <= tol), f"dim={dim}: max abs error {err.max():.3e}"


def test_correlated_normals_rejects_bad_shapes():
    z = _dev(np.zeros((1, 10, 2)))
    rng = B.Rng()
    rng.mode, rng.seed, rng.n_paths_total = B.RNG_PHILOX, 1, 10
    for dim in (0, 17):
        rc, _ = _correlated(rng, 1, dim, np.eye(max(dim, 1)), 10)
        assert rc < 0, f"dim {dim} accepted"
    rng.mode, rng.d_z, rng.n_paths_total = B.RNG_INJECT, z.data_ptr(), 10
    rc, _ = _correlated(rng, 1, 2, np.eye(2), 11)
    assert rc < 0, "inject mode with fewer injected paths than requested accepted"
