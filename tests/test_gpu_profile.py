"""Profile likelihoods on the device (cvb_lattice_profile) and the likelihood-ratio intervals built on them.

A. The rows equal, bit for bit, the numpy reduction of cvb_lattice_eval's values for the same slice and
   path (tests/test_profile_host.reference_rows): both models, the e0.05, cfg3 (1000 bins) and cfg4
   (k = 31, r = 150) histograms, every non-empty keep mask, the slices of shard_blocked and shard_strided
   for W = 1, 2, 3, 8 and every rank (segments left empty by a slice included), the automatic,
   per-point, GEMM and prefix paths; a coverage axis with a repeated value, and points that are -inf
   (coverage 10^6 at error rate 0, and more where the lattice misses the histogram), whole segments too.
B. The cfg3 lattice (10^6 points): coverage alone (40 segments of 25 000 points), (c, e), every axis.
C. A device out_rows on a torch stream: the call only enqueues; the rows are ordered behind it.
D. Poisoned contexts give the clean rows; every row is written and nothing around it.
E. Per-rank rows merged by parallel.merge_segments are the single call's rows, W = 1..8 (bit for bit on
   the per-point path; on the factored path, whose last bits may depend on the slicing, bit for bit
   against the reduction of each rank's own values, within 1e-12 of the single call, and another point
   than the single call's only where the two are a near-tie within 1e-12).
F. Basic model against the pinned C oracle: profile values, the oracle's value at the refined points,
   the coverage endpoints against brentq on the oracle's profile.
G. Repeats model (cfg2 of e2e_golden.json): properties of the intervals.
H. `covest ... --ci 0.95 --polish` adds exactly the interval keys.
"""
import ctypes
import functools
import io
import json
import os
from contextlib import redirect_stdout

import numpy as np
import pytest
import yaml
from scipy.optimize import brentq, minimize_scalar
from scipy.stats import chi2

from covest_b200 import data, parallel
from covest_b200.covest import CoverageEstimator
from covest_b200.histogram import process_histogram
from covest_b200.models import BasicModel, select_model
from oracle import covest_oracle as orc
from tests import bigpoints
from tests.helpers import GOLDEN, case_hist, context_for, load_case
from tests.test_gpu_poison import Framed, _context
from tests.test_profile_host import reference_rows

pytestmark = pytest.mark.gpu

PATHS = {'auto': 0, 'per_point': 1, 'gemm': 3, 'prefix': 4}
KR = {'e05_basic': (21, 100), 'e05_repeats': (21, 100), 'cfg3_repeats_dense1000': (21, 100),
      'cfg4_repeats_k31': (31, 150)}


@functools.lru_cache(maxsize=None)
def _oracle(name):
    case = load_case(name)
    k, r = KR[name]
    return orc.Model(case['model'], k, r, case_hist(case), case['tail'], max_error=8)


def _axes(kind, ascending=False):
    """A small lattice: a coverage axis with a repeated value (unless `ascending`) that ends at 10^6, and
    an error-rate axis that starts at 0.  At coverage 10^6 and error rate 0 every histogram here has bins
    no error-free k-mer explains: those points are -inf, and so is every segment made of them alone."""
    err = np.concatenate(([0.0], np.geomspace(0.002, 0.2, 29)))
    if kind == 'basic':
        cov = np.geomspace(5.0, 60.0, 38)
        return [np.concatenate((cov, [1e6])) if ascending else np.concatenate((cov, [60.0, 1e6])), err]
    cov = [12.0, 20.0, 30.0, 45.0, 1e6] if ascending else [12.0, 20.0, 20.0, 30.0, 45.0, 1e6]
    return [np.array(cov), err, np.array([0.3, 0.65, 1.0]), np.array([0.0, 0.5, 1.0]), np.array([0.05, 0.2, 0.5, 1.0])]


def _slices(total, block):
    """(first, stride, block, count, lattice indices) of every rank's slice, blocked and strided."""
    for W in (1, 2, 3, 8):
        for r in range(W):
            for first, stride, blk, count in (parallel.shard_blocked(total, block, r, W),
                                              parallel.shard_strided(total, r, W)[:2] + (1,) +
                                              parallel.shard_strided(total, r, W)[2:]):
                i = np.arange(count)
                yield first, stride, blk, count, (first + (i // blk) * stride) * blk + i % blk


def _assert_rows(got, want, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, what
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    differ = (nan_g != nan_w) | (~nan_w & (got.view(np.uint64) != want.view(np.uint64)))
    if differ.any():
        r = np.flatnonzero(differ.any(axis=1))
        raise AssertionError('%s: %d of %d rows differ, first %s: %r instead of %r'
                             % (what, len(r), len(got), r[:4].tolist(), got[r[0]].tolist(), want[r[0]].tolist()))


CASES_A = [('e05_basic', 'auto'), ('e05_basic', 'per_point')] + \
    [(name, path) for name in ('e05_repeats', 'cfg3_repeats_dense1000', 'cfg4_repeats_k31') for path in PATHS]


@pytest.mark.parametrize('name,path', CASES_A)
def test_rows_equal_the_reference_reduction(name, path):
    m = _oracle(name)
    axes = _axes('basic' if m.kind == 0 else 'repeats')
    n = len(axes)
    lens = [len(a) for a in axes]
    total = int(np.prod(lens))
    block = int(np.prod(lens[2:])) if n > 2 else 1
    ctx = context_for(m)
    try:
        ctx.set_path(PATHS[path])
        whole = np.array(ctx.lattice_eval(axes)[0])
        assert np.isneginf(whole).any() and np.isfinite(whole).any()
        empty_seen = False
        for first, stride, blk, count, idx in _slices(total, block):
            ll = np.array(ctx.lattice_eval(axes, first=first, stride=stride, block=blk, count=count)[0]) \
                if count else np.empty(0)
            for mask in range(1, 1 << n):
                got = ctx.lattice_profile(axes, mask, first=first, stride=stride, block=blk, count=count)
                want = reference_rows(ll, idx, axes, mask)
                _assert_rows(got, want, '%s %s mask %d slice %r' % (name, path, mask, (first, stride, blk, count)))
                empty_seen = empty_seen or bool(np.isnan(want[:, 1]).any())
        assert empty_seen
        # a segment whose points are all -inf (or NaN): -inf with the axis values of its lowest lattice index
        rows = ctx.lattice_profile(axes, 3)
        seg = (np.arange(total) // block)  # the (c, e) segment of every lattice index
        dead = [g for g in range(lens[0] * lens[1]) if not np.any(whole[seg == g] > -np.inf)]
        assert dead
        for g in dead:
            low = int(np.flatnonzero(seg == g)[0])
            digits = np.unravel_index(low, lens)
            assert rows[g, 0] == -np.inf and rows[g, 1:].tolist() == [axes[a][digits[a]] for a in range(n)]
        # a repeated coverage value: equal values at different indices go to the lower index
        rows = ctx.lattice_profile(axes, 1)
        dup = [i for i in range(1, lens[0]) if axes[0][i] == axes[0][i - 1]]
        assert dup and all(rows[i, 0] == rows[i - 1, 0] for i in dup)
    finally:
        ctx.close()


@pytest.mark.parametrize('mask', [1, 3, 31])
def test_large_lattice_rows(mask):
    big = bigpoints.load_big('cfg3')
    m = orc.Model('repeats', 21, 100, big['hist'], big['tail'], max_error=8)
    axes = bigpoints.lattice_axes('cfg3')
    ctx = context_for(m)
    try:
        ll = np.array(ctx.lattice_eval(axes)[0])
        assert len(ll) == 10 ** 6
        got = ctx.lattice_profile(axes, mask)
        _assert_rows(got, reference_rows(ll, np.arange(len(ll)), axes, mask), 'cfg3 mask %d' % mask)
    finally:
        ctx.close()


def test_device_rows_are_enqueued_on_the_stream():
    import torch
    m = _oracle('e05_repeats')
    axes = _axes('repeats')
    ctx = context_for(m)
    try:
        want = ctx.lattice_profile(axes, 3)
        s = torch.cuda.Stream()
        rows = torch.full(want.shape, float('nan'), dtype=torch.float64, device='cuda')
        ctx.lattice_profile(axes, 3, out_rows=rows, stream=s)  # the context's buffers have their size
        s.synchronize()
        with torch.cuda.stream(s):
            rows.fill_(float('nan'))
            torch.cuda._sleep(200_000_000)  # ~0.1 s of device time ahead of the call on the stream
            ctx.lattice_profile(axes, 3, out_rows=rows, stream=s)
            pending = not s.query()
            copy = rows.clone()
        assert pending, 'the call waited for the stream'
        s.synchronize()
        _assert_rows(copy.cpu().numpy(), want, 'device rows')
    finally:
        ctx.close()


@pytest.mark.parametrize('device', [False, True], ids=['host', 'device'])
@pytest.mark.parametrize('poison', ['nan', 'finite'])
def test_poisoned_contexts_write_every_row(poison, device):
    m = _oracle('e05_repeats')
    axes = _axes('repeats')
    lens = np.array([len(a) for a in axes], dtype=np.int32)
    vals = np.concatenate(axes)
    total = int(np.prod(lens))
    M = int(np.prod(lens[2:]))
    with _context(m) as clean, _context(m, poison) as dirty:
        for path in (0, 1):
            clean.set_path(path)
            dirty.set_path(path)
            for first, stride, block, count in ((0, 1, 1, total), (1, 3, M, 2 * M), (5, 7, 1, 100), (0, 1, 1, 0)):
                for mask in (1, 2, 3, 28, 31):
                    want = clean.lattice_profile(axes, mask, first=first, stride=stride, block=block, count=count)
                    out = Framed(want.size, device)
                    rc = dirty._lib.cvb_lattice_profile(dirty._ctx, lens.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                                        vals.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), first,
                                                        stride, block, count, mask, out.ptr, None)
                    assert rc == 0, dirty._lib.cvb_last_error(dirty._ctx).decode()
                    _assert_rows(out.values(poison).reshape(want.shape), want, '%s mask %d' % (poison, mask))


def test_bad_masks_are_refused():
    m = _oracle('e05_repeats')
    axes = _axes('repeats')
    ctx = context_for(m)
    try:
        lens = np.array([len(a) for a in axes], dtype=np.int32)
        vals = np.concatenate(axes)
        out = np.empty(10 ** 4)
        for mask in (0, 32, 33, 1 << 31):
            rc = ctx._lib.cvb_lattice_profile(ctx._ctx, lens.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                              vals.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 0, 1, 1, 10,
                                              mask, out.ctypes.data_as(ctypes.c_void_p), None)
            assert rc == -1 and ctx._lib.cvb_last_error(ctx._ctx)
        big = np.array([1 << 13] * 5, dtype=np.int32)  # 2^65 segments
        bv = np.zeros(5 << 13)
        rc = ctx._lib.cvb_lattice_profile(ctx._ctx, big.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                          bv.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 0, 1, 1, 10, 31,
                                          out.ctypes.data_as(ctypes.c_void_p), None)
        assert rc == -1 and b'int64' in ctx._lib.cvb_last_error(ctx._ctx)
        # the context still works
        assert np.isfinite(ctx.lattice_profile(axes, 1)[1:, 0]).all()
    finally:
        ctx.close()


@pytest.mark.parametrize('kind', ['basic', 'repeats'])
def test_merged_rank_rows_equal_the_single_call(kind):
    """On the per-point path a point's value does not depend on the slice it is evaluated in: the merged
    rows are the single call's, bit for bit.  The factored path may round a point of another slicing in
    its last bits (its tiles differ), so there the merge is held bit for bit to the reduction of each
    rank's own values; against the single call the values agree within 1e-12, and where the merged row
    names another point than the single call, the two points are a near-tie of the single call's own
    values (within 1e-12), which such last bits decide."""
    m = _oracle('e05_%s' % kind)
    axes = _axes(kind, ascending=True)
    lens = [len(a) for a in axes]
    total = int(np.prod(lens))
    block = int(np.prod(lens[2:])) if len(lens) > 2 else 1
    ctx = context_for(m)

    def index_of(rows):  # lattice index of each row's point (ascending axes without repeats)
        idx = np.zeros(len(rows), dtype=np.int64)
        for a, ax in enumerate(axes):
            idx = idx * len(ax) + np.searchsorted(ax, rows[:, 1 + a])
        return idx

    try:
        for path in (1, 0):
            ctx.set_path(path)
            ll_whole = np.array(ctx.lattice_eval(axes)[0])
            for mask in range(1, 1 << len(axes)):
                whole = ctx.lattice_profile(axes, mask)
                for W in range(1, 9):
                    parts, ref = [], []
                    for f, s, b, c in (parallel.shard_blocked(total, block, r, W) for r in range(W)):
                        parts.append(ctx.lattice_profile(axes, mask, first=f, stride=s, block=b, count=c))
                        i = np.arange(c)
                        ll = np.array(ctx.lattice_eval(axes, first=f, stride=s, block=b, count=c)[0]) if c else []
                        ref.append(reference_rows(ll, (f + (i // b) * s) * b + i % b, axes, mask))
                    merged = parallel.merge_segments(np.stack(parts))
                    what = 'path %d mask %d W %d' % (path, mask, W)
                    _assert_rows(merged, parallel.merge_segments(np.stack(ref)), what)
                    if path == 1:
                        _assert_rows(merged, whole, what)
                        continue
                    assert np.array_equal(np.isnan(merged[:, 1]), np.isnan(whole[:, 1])), what
                    fin = np.isfinite(whole[:, 0])
                    assert np.array_equal(fin, np.isfinite(merged[:, 0])), what
                    assert np.array_equal(merged[~fin, 0], whole[~fin, 0]), what
                    assert np.allclose(merged[fin, 0], whole[fin, 0], rtol=1e-12, atol=0), what
                    live = ~np.isnan(whole[:, 1])
                    other = live & np.any(merged[:, 1:] != whole[:, 1:], axis=1)
                    if other.any():
                        a = ll_whole[index_of(merged[other])]
                        b = ll_whole[index_of(whole[other])]
                        assert np.allclose(a, b, rtol=1e-12, atol=0), (what, merged[other], whole[other], a, b)
    finally:
        ctx.close()


# ---- F: basic model against the oracle ---------------------------------------------------------------
def _estimate(model, guess):
    est = CoverageEstimator(model)
    x, ok = est.compute_coverage(guess)
    x = list(x)
    xp, _ = est.polish(x)
    return est, xp


def test_basic_profile_matches_the_oracle():
    case = load_case('e05_basic')
    hist = case_hist(case)
    model = BasicModel(21, 100, hist, case['tail'], max_error=8)
    om = orc.Model('basic', 21, 100, hist, case['tail'], max_error=8)
    _, _, _, gc, ge = process_histogram(hist, 21, 100, trim=0, sample_factor=1)
    est, x_hat = _estimate(model, [gc, ge])
    free = [0, 1]
    se = est._standard_errors(np.array(x_hat), free)
    values = np.linspace(x_hat[0] - 4 * se[0], x_hat[0] + 4 * se[0], 33)
    prof = est.profile('coverage', values, est.nuisance_axes(0, np.array(x_hat), se, free), x_hat)
    assert prof.success.all() and np.all(prof.fun <= prof.lattice_fun)

    def oracle_profile(c):
        r = minimize_scalar(lambda e: -om.loglik_batch(np.array([[c, e]]))[0], bounds=(1e-6, 0.5), method='bounded',
                            options={'xatol': 1e-13})
        return -r.fun

    want = np.array([oracle_profile(c) for c in values])
    assert np.allclose(-prof.fun, want, rtol=1e-9, atol=0)
    at = om.loglik_batch(prof.x)
    assert np.allclose(at, -prof.fun, rtol=1e-9, atol=0)
    # endpoints at 0.95 against brentq on the oracle's profile
    iv = est.likelihood_intervals(x_hat, level=0.95, params=['coverage'])['coverage']
    top = -minimize_scalar(lambda c: -oracle_profile(c), bounds=(values[0], values[-1]), method='bounded',
                           options={'xatol': 1e-10}).fun
    thr = top - chi2.ppf(0.95, 1) / 2
    lo = brentq(lambda c: oracle_profile(c) - thr, values[0], x_hat[0], xtol=1e-12)
    hi = brentq(lambda c: oracle_profile(c) - thr, x_hat[0], values[-1], xtol=1e-12)
    half = (hi - lo) / 2
    assert abs(iv.lo - lo) <= 1e-3 * half and abs(iv.hi - hi) <= 1e-3 * half, (iv, lo, hi)
    assert not any(iv.flags.values()), iv


# ---- G: repeats model ----------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _cfg2():
    with open(os.path.join(GOLDEN, 'e2e_golden.json')) as f:
        g = json.load(f)['cfg2_repeats']
    hist = {int(j): int(h) for j, h in g['hist']}
    h2, tail, sf, gc, ge = process_histogram(hist, g['k'], g['r'], **g['flags'])
    return g, hist, h2, tail, gc, ge


def test_repeats_intervals():
    g, hist, h2, tail, gc, ge = _cfg2()
    model = select_model(g['model'])(g['k'], g['r'], h2, tail, max_error=8)
    guess = list(model.defaults)
    guess[:2] = gc, ge
    est, x_hat = _estimate(model, guess)
    x_hat = np.array(x_hat)
    ivs = est.likelihood_intervals(x_hat, level=0.95)
    assert list(ivs) == list(model.params)
    free = list(range(5))
    se = est._standard_errors(x_hat, free)
    for p, name in enumerate(model.params):
        iv = ivs[name]
        assert iv.lo <= x_hat[p] <= iv.hi, iv
        if p < 2:  # coverage and error rate are pinned down by the histogram
            assert not iv.flags['open'] and not iv.flags['at_bound'], iv
        if not iv.flags['open']:  # an end that is not a bound is a crossing of the threshold
            ends = [v for v in (iv.lo, iv.hi) if v not in model.bounds[p]]
            prof = est.profile(p, np.array(ends), est.nuisance_axes(p, x_hat, se, free), x_hat)
            assert np.all(np.abs(-prof.fun - iv.threshold) <= 0.05), (name, -prof.fun, iv.threshold)
        coarse = est.profile(p, iv.values, est.nuisance_axes(p, x_hat, se, free), x_hat)
        assert np.all(coarse.fun <= coarse.lattice_fun)
        assert np.array_equal(coarse.x[:, p].view(np.uint64), np.asarray(iv.values, dtype=np.float64).view(np.uint64))
    rep = data.interval_report(hist, model, 1, ivs, 0.95)
    kmers = sum(j * h for j, h in hist.items())
    assert rep['genome_size_ci'] == [int(round(kmers / model.correct_c(ivs['coverage'].hi))),
                                     int(round(kmers / model.correct_c(ivs['coverage'].lo)))]


# ---- H: the command line ---------------------------------------------------------------------------------
def _cli(tmp_path, extra):
    from covest_b200 import covest as cli
    g = _cfg2()[0]
    path = tmp_path / 'cfg2.hist'
    path.write_text(''.join('%d %d\n' % (j, h) for j, h in g['hist']))
    buf = io.StringIO()
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        with redirect_stdout(buf):
            cli.run([str(path), '-m', 'repeat', '-k', '21', '-r', '100', '-sf', '1', '--polish', '--seed', '1'] + extra)
    finally:
        os.chdir(cwd)
    return buf.getvalue()


def test_cli_ci_adds_exactly_the_interval_keys(tmp_path):
    plain = _cli(tmp_path, [])
    with_ci = _cli(tmp_path, ['--ci', '0.95'])
    a, b = yaml.safe_load(plain), yaml.safe_load(with_ci)
    new = {'ci_level', 'genome_size_ci', 'ci_flags'} | {'%s_ci' % p for p in ('coverage', 'error_rate', 'q1', 'q2', 'q')}
    assert set(b) - set(a) == new and set(a) <= set(b)
    assert {k: b[k] for k in a} == a
    assert b['ci_level'] == 0.95
    assert b['coverage_ci'][0] <= b['coverage'] <= b['coverage_ci'][1]
    assert b['genome_size_ci'][0] <= b['genome_size'] <= b['genome_size_ci'][1]
    # without --ci the report is the one print_output writes for the estimate alone
    for key in new:
        b.pop(key)
    assert yaml.dump(b, indent=4, default_flow_style=False) == yaml.dump(a, indent=4, default_flow_style=False)
