"""The batched path without a tail evaluates the lines of the histogram that hold a count, and nothing else.

Without a tail the mass sum_j p_j does not enter the log-likelihood (models.py:103-107), so the bins of
the 64-slot lines without any count cannot change a result.  Such a context builds row tables from the
keys of the lines with counts (csrc/cvtables.h, cv_build_row_tables): the profile kernel evaluates
only those, writes the line of the sums as zeros, and the prefix kernel forms no mass.  The row
layout, and the `row_slots` it reports, stay as before: the lines with counts, then the line of the sums.

- Values on the prefix and GEMM paths match the oracle (1e-9) and the per-point kernel, which keeps the
  full tables (1e-11, the same -inf sets), for row tables of 1, 2, 4 and 8 rows per group.
- A histogram and the keys of its lines with counts (plus its largest key at count 0, so that max(hist),
  i.e. O_thr, stays) give bit-identical values: the bins of the other lines are not evaluated.
- COVEST_B200_ROWS=full and contexts with a tail keep the rows they had.
- A context that poisons its scratch (COVEST_B200_POISON=nan) gives the clean values bit for bit.
"""
import contextlib
import functools

import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests import test_gpu_rows
from tests.helpers import context_for, rel_err_ll

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-9
FAST_RTOL = 1e-11
BINS = 1000


def _counts(keys, counted, seed):
    rng = np.random.default_rng(seed)
    return {j: (int(rng.integers(1, 10 ** 6 // j + 2)) if counted(j) else 0) for j in keys}


def _cfg4():
    z = np.load(test_gpu_rows.__file__.replace('test_gpu_rows.py', 'golden/big_cfg4.npz'))
    return {int(j): int(h) for j, h in zip(z['hist_j'], z['hist_h'])}


# name -> (histogram, coverages, error rates and q of its lattice).  All have keys without counts in whole
# 64-slot lines.  The comments give the rows per group NA of their row tables (the full tables have 8);
# tests/test_row_tables_host.py checks them.
Q_LOW, Q_FAR = np.linspace(0.3, 1.0, 6), np.linspace(0.2, 0.7, 6)  # q small enough for ~50 copies: far bins
HISTS = {
    # NA = 1: counts in line 0 only
    'line0': (lambda: _counts(range(1, BINS + 1), lambda j: j <= 64, 1), (12.0, 18.0), (0.01, 0.04), Q_LOW),
    # NA = 1: counted bins that do not start at 1 (line 1)
    'line1': (lambda: _counts(range(1, BINS + 1), lambda j: 65 <= j <= 128, 2), (20.0, 30.0), (0.01, 0.04), Q_LOW),
    # NA = 1: only the last line (961 .. 1000) has counts
    'last_line': (lambda: _counts(range(1, BINS + 1), lambda j: j > 960, 3), (150.0, 200.0), (0.01, 0.04), Q_FAR),
    # NA = 2: lines 0, 1 and 3 (tests/test_gpu_rows.py, 700 keys): runs split at the gap
    'lines013': (test_gpu_rows.sparse_hist, (12.0, 18.0), (0.01, 0.04), Q_LOW),
    # NA = 4: lines 0 .. 5
    'lines0to5': (lambda: _counts(range(1, BINS + 1), lambda j: j <= 384, 4), (40.0, 60.0), (0.01, 0.04), Q_FAR),
    # NA = 2: lines 0, 2 and 5
    'lines025': (lambda: _counts(range(1, BINS + 1), lambda j: (j - 1) // 64 in (0, 2, 5), 6), (30.0, 45.0),
                 (0.01, 0.04), Q_FAR),
    # NA = 4 from three blocks of groups: sparse keys (every third number up to 3000), counts below 150
    # and around 700
    'sparse_keys': (lambda: _counts(range(1, 3001, 3), lambda j: j < 150 or 690 < j < 720, 5), (40.0, 60.0),
                    (0.01, 0.04), Q_FAR),
    # NA = 8 from two blocks of groups: 2000 keys, counts in lines 0 .. 8 (5 groups of 8 rows)
    'lines0to8': (lambda: _counts(range(1, 2 * BINS + 1), lambda j: j <= 576, 7), (40.0, 60.0), (0.01, 0.04), Q_FAR),
    # cfg4's 5000 keys (k = 31, r = 150), 45 of 80 lines with counts: its row tables would take 3 blocks of
    # groups, so it keeps the full tables (5 blocks) and only leaves out the mass
    'cfg4': (_cfg4, (200.0, 240.0), (0.005, 0.01), np.linspace(0.25, 0.5, 6)),
    # no count at all: every value is 0 (models.py:106), the prefix kernel reads the zero line of the sums
    'all_zero': (lambda: _counts(range(1, BINS + 1), lambda j: False, 8), (12.0, 18.0), (0.01, 0.04), Q_LOW),
}


@functools.lru_cache(maxsize=None)
def _hist(name):
    return HISTS[name][0]()


def _kr(name, S):
    return (31, 150) if name == 'cfg4' else (max(21, S - 1), 100)


def _axes(name):
    """q2 = 0 leaves one copy (b(2) = 0 cuts the series): -inf where the counted bins lie far out"""
    _, cov, err, q = HISTS[name]
    return [np.array(cov), np.array(err), np.array([0.4, 0.8]), np.array([0.0, 0.3, 0.7]), np.asarray(q)]


def _grid(axes):
    return np.ascontiguousarray(np.array(np.meshgrid(*axes, indexing='ij')).reshape(len(axes), -1).T)


def _line(j):
    """The 64-slot line of key j in the tables of keys 1 .. n with n > 512: groups of 128 keys from key 1."""
    return (j - 1) // 64


def _counted_lines(hist):
    return len({_line(j) for j, h in hist.items() if h})


@contextlib.contextmanager
def _context(hist, S, k, r, env=()):
    with pytest.MonkeyPatch.context() as mp:
        mp.delenv('COVEST_B200_POISON', raising=False)
        mp.delenv('COVEST_B200_ROWS', raising=False)
        for key, v in env:
            mp.setenv(key, v)
        ctx = context_for(orc.Model('repeats', k, r, hist, 0, max_error=S))
    try:
        yield ctx
    finally:
        ctx.close()


def _eval(ctx, path, pts):
    ctx.set_path(path)
    got = ctx.loglik(pts)
    return got, ctx.last_path_info()


CASES = [(name, 8) for name in HISTS if name != 'all_zero'] + [(name, S) for name in ('lines013', 'cfg4') for S in (1, 17, 32)]


@pytest.mark.parametrize('name,S', CASES, ids=['%s-S%d' % c for c in CASES])
def test_factored_paths_match_the_oracle_and_the_per_point_kernel(name, S):
    hist = _hist(name)
    k, r = _kr(name, S)
    pts = _grid(_axes(name))
    want = orc.Model('repeats', k, r, hist, 0, max_error=S).loglik_batch(pts, threads=8)
    with _context(hist, S, k, r) as ctx:
        ref, _ = _eval(ctx, ctx.PATH_PER_POINT, pts)
        assert np.array_equal(np.isinf(ref), np.isinf(want))
        assert np.isfinite(want).sum() >= len(pts) // 2
        for path in (ctx.PATH_FACTORED_PREFIX, ctx.PATH_FACTORED_GEMM):
            got, info = _eval(ctx, path, pts)
            assert info['path'] == 'factored'
            if name in ('line0', 'line1', 'last_line', 'lines013', 'lines0to5', 'lines0to8'):
                assert info['row_slots'] == 64 * _counted_lines(hist) + 32
            assert np.array_equal(np.isinf(got), np.isinf(want)), path
            assert np.array_equal(np.isinf(got), np.isinf(ref)), path
            assert rel_err_ll(got, want).max() <= LL_RTOL, (path, float(rel_err_ll(got, want).max()))
            assert rel_err_ll(got, ref).max() <= FAST_RTOL, (path, float(rel_err_ll(got, ref).max()))


def _counted_keys_only(hist, line_of):
    """The keys of the lines of `hist` that hold a count, plus its largest key at count 0."""
    lines = {line_of(j) for j, h in hist.items() if h}
    out = {j: h for j, h in hist.items() if line_of(j) in lines}
    out.setdefault(max(hist), 0)
    return out


# Histogram B of a pair is too small for row tables of its own: it runs on its full tables, which are the
# row tables of A plus one group for the last key, in a line without counts (tests/test_row_tables_host.py).
# So the pairs show that A's batched path runs on its row tables, for NA = 1, 2, 4 and 8.
PAIRS = ('line0', 'line1', 'last_line', 'lines013', 'lines0to5', 'lines025', 'lines0to8')


@pytest.mark.parametrize('pair', PAIRS)
def test_bins_of_lines_without_counts_are_not_evaluated(pair):
    a = _hist(pair)
    b = _counted_keys_only(a, _line)
    assert max(a) == max(b) and len(b) < len(a)
    k, r = _kr(pair, 8)
    pts = _grid(_axes(pair))
    with _context(a, 8, k, r) as ca, _context(b, 8, k, r) as cb:
        for path in (ca.PATH_FACTORED_PREFIX, ca.PATH_FACTORED_GEMM):
            va, ia = _eval(ca, path, pts)
            vb, ib = _eval(cb, path, pts)
            assert np.isfinite(va).sum() >= len(pts) // 2
            assert ia['row_slots'] == ib['row_slots']
            assert np.array_equal(va.view(np.uint64), vb.view(np.uint64)), path


@pytest.mark.parametrize('name', ['line0', 'lines013', 'lines0to5'])
def test_full_rows_and_tails_keep_their_rows(name):
    hist = _hist(name)
    pts = _grid(_axes(name))
    counted = _counted_lines(hist)
    table_lines = 16  # 700 and 1000 keys from key 1: one block of 8 groups of 8 rows
    with _context(hist, 8, 21, 100) as ctx:
        ref, _ = _eval(ctx, ctx.PATH_PER_POINT, pts)
    # every line of the tables (no row tables, no line of sums)
    with _context(hist, 8, 21, 100, env=(('COVEST_B200_ROWS', 'full'),)) as ctx:
        for path in (ctx.PATH_FACTORED_PREFIX, ctx.PATH_FACTORED_GEMM):
            got, info = _eval(ctx, path, pts)
            assert info['row_slots'] == 64 * table_lines
            assert np.array_equal(np.isinf(got), np.isinf(ref))
            assert rel_err_ll(got, ref).max() <= FAST_RTOL
    # with a tail: every bin enters the mass, the lines without counts through the line of the sums.  Here
    # the histogram holds all but a minute part of the mass, so the tail term tail * log(1 - mass) hangs on
    # the last bits of the mass (tests/bigpoints.py, ll_tolerance): the values of this path are pinned by
    # tests/test_gpu_rows.py, this checks its rows
    m = orc.Model('repeats', 21, 100, hist, 500, max_error=8)
    with pytest.MonkeyPatch.context() as mp:
        mp.delenv('COVEST_B200_POISON', raising=False)
        mp.delenv('COVEST_B200_ROWS', raising=False)
        ctx = context_for(m)
    try:
        ref, _ = _eval(ctx, ctx.PATH_PER_POINT, pts)
        for path in (ctx.PATH_FACTORED_PREFIX, ctx.PATH_FACTORED_GEMM):
            got, info = _eval(ctx, path, pts)
            assert info['row_slots'] == 64 * counted + 32
            assert np.array_equal(np.isinf(got), np.isinf(ref))
    finally:
        ctx.close()


@pytest.mark.parametrize('name,S', CASES, ids=['%s-S%d' % c for c in CASES])
def test_poisoned_scratch_gives_the_clean_values(name, S):
    hist = _hist(name)
    k, r = _kr(name, S)
    pts = _grid(_axes(name))
    with _context(hist, S, k, r) as clean, _context(hist, S, k, r, env=(('COVEST_B200_POISON', 'nan'),)) as dirty:
        for path in (clean.PATH_FACTORED_PREFIX, clean.PATH_FACTORED_GEMM):
            want, iw = _eval(clean, path, pts)
            got, ig = _eval(dirty, path, pts)
            assert iw['row_slots'] == ig['row_slots']
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), path


@pytest.mark.parametrize('poison', [None, 'nan'])
def test_a_histogram_without_counts_gives_zeros(poison):
    """No line has a count: the row keeps only the line of the sums, which K1 writes as zeros.  The prefix
    kernel must still form every point's sum from it rather than finish points from partials it never
    wrote (COVEST_B200_POISON=nan turns such a read into NaN)."""
    hist = _hist('all_zero')
    axes = _axes('all_zero')
    pts = _grid(axes)
    want = orc.Model('repeats', 21, 100, hist, 0, max_error=8).loglik_batch(pts, threads=8)
    assert np.array_equal(want, np.zeros(len(pts)))
    env = (('COVEST_B200_POISON', poison),) if poison else ()
    with _context(hist, 8, 21, 100, env=env) as ctx:
        for path in (ctx.PATH_FACTORED_PREFIX, ctx.PATH_FACTORED_GEMM):
            got, info = _eval(ctx, path, pts)
            assert info['path'] == 'factored' and info['row_slots'] == 32
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), path
            ctx.set_path(path)
            by_axes, _ = ctx.lattice_eval(axes)
            assert np.array_equal(by_axes.view(np.uint64), want.view(np.uint64)), path
