"""Profile likelihoods and likelihood-ratio intervals, host side (no device needed).

The interval logic of CoverageEstimator.likelihood_intervals runs against fake models whose
log-likelihood is known in closed form; the one step that is the device's -- the best row per
segment of a lattice (cvb_lattice_profile) -- is replaced by the numpy reduction `reference_rows`,
which tests/test_gpu_profile.py also holds the device to.  Also here: the per-segment merge of
per-rank rows, the validation of keep masks and of the --ci arguments, and the genome-size interval.
"""
import itertools

import numpy as np
import pytest
from scipy.stats import chi2

from covest_b200 import covest as cli
from covest_b200 import data, engine, parallel
from covest_b200.covest import CoverageEstimator


# ---- the reference reduction ---------------------------------------------------------------------
def reference_rows(ll, idx, axes, keep_mask):
    """Rows (value, params...) of the best point per segment, for the points at lattice indices `idx`
    with values `ll`: larger value first, NaN as -inf, -0 tied with +0, ties to the lower lattice index;
    the value as the radix top-K reports it (NaN -> -inf, -0 -> +0); (-inf, NaN...) for an empty segment."""
    lens = [len(a) for a in axes]
    kept = [a for a in range(len(axes)) if keep_mask >> a & 1]
    n_seg = int(np.prod([lens[a] for a in kept]))
    rows = np.full((n_seg, 1 + len(axes)), np.nan)
    rows[:, 0] = -np.inf
    idx = np.asarray(idx, dtype=np.int64)
    if len(idx) == 0:
        return rows
    v = np.asarray(ll, dtype=np.float64).copy()
    v[np.isnan(v)] = -np.inf
    v[v == 0] = 0.0
    digits = np.unravel_index(idx, lens)
    seg = np.ravel_multi_index([digits[a] for a in kept], [lens[a] for a in kept])
    order = np.lexsort((idx, -v, seg))
    first = order[np.r_[True, seg[order][1:] != seg[order][:-1]]]
    rows[seg[first], 0] = v[first]
    for a in range(len(axes)):
        rows[seg[first], 1 + a] = np.asarray(axes[a], dtype=np.float64)[digits[a][first]]
    return rows


# ---- fake models --------------------------------------------------------------------------------
class FakeModel:
    """Two parameters (coverage, error_rate); loglikelihood_batch is `fn(c, e)` on the host."""
    params = ('coverage', 'error_rate')

    def __init__(self, fn, bounds=((0.01, None), (0, 0.5))):
        self.fn = fn
        self.bounds = bounds
        self.r, self.k = 100, 21

    @property
    def param_count(self):
        return len(self.params)

    def loglikelihood_batch(self, rows):
        rows = np.asarray(rows, dtype=np.float64).reshape(-1, 2)
        lo = np.array([b[0] if b[0] is not None else -np.inf for b in self.bounds])
        hi = np.array([b[1] if b[1] is not None else np.inf for b in self.bounds])
        rows = np.clip(rows, lo, hi)  # the device clips to the bounds
        return self.fn(rows[:, 0], rows[:, 1])

    def correct_c(self, c):
        return c * (self.r - self.k + 1) / self.r


class HostEstimator(CoverageEstimator):
    """CoverageEstimator whose lattice profile is the reference reduction over a host evaluation."""

    def _lattice_profile(self, model_axes, keep_mask):
        pts = np.array(list(itertools.product(*model_axes)), dtype=np.float64)
        return reference_rows(self.model.loglikelihood_batch(pts), np.arange(len(pts)), model_axes, keep_mask)


C0, SC, E0, SE = 10.0, 0.2, 0.05, 0.005
Z = float(np.sqrt(chi2.ppf(0.95, 1)))


def quadratic(rho=0.6, c0=C0):
    cov = np.array([[SC * SC, rho * SC * SE], [rho * SC * SE, SE * SE]])
    P = np.linalg.inv(cov)

    def fn(c, e):
        d0, d1 = c - c0, e - E0
        return -0.5 * (P[0, 0] * d0 * d0 + 2 * P[0, 1] * d0 * d1 + P[1, 1] * d1 * d1)
    return fn


def test_quadratic_profile_gives_z_times_se():
    est = HostEstimator(FakeModel(quadratic()))
    iv = est.likelihood_intervals([C0, E0], level=0.95)
    assert iv['coverage'].lo == pytest.approx(C0 - Z * SC, abs=1e-3 * SC)
    assert iv['coverage'].hi == pytest.approx(C0 + Z * SC, abs=1e-3 * SC)
    assert iv['error_rate'].lo == pytest.approx(E0 - Z * SE, abs=1e-3 * SE)
    assert iv['error_rate'].hi == pytest.approx(E0 + Z * SE, abs=1e-3 * SE)
    for v in iv.values():
        assert not any(v.flags.values()), v


def test_level_sets_the_width():
    est = HostEstimator(FakeModel(quadratic(rho=0.0)))
    for level in (0.5, 0.99):
        iv = est.likelihood_intervals([C0, E0], level=level, params=['coverage'])['coverage']
        z = np.sqrt(chi2.ppf(level, 1))
        assert iv.hi - C0 == pytest.approx(z * SC, rel=1e-3)
        assert C0 - iv.lo == pytest.approx(z * SC, rel=1e-3)


def test_profile_refines_from_the_lattice_rows():
    est = HostEstimator(FakeModel(quadratic()))
    vals = np.linspace(C0 - 0.5, C0 + 0.5, 9)
    prof = est.profile('coverage', vals, [None, np.linspace(0.03, 0.07, 5)], [C0, E0])
    assert np.all(prof.fun <= prof.lattice_fun)
    assert np.array_equal(prof.x[:, 0], vals)  # the profiled coordinate is held
    want = 0.5 * ((vals - C0) / SC) ** 2
    assert np.allclose(prof.fun, want, atol=1e-9)
    assert prof.success.all()


def test_at_bound_when_a_bound_cuts_the_interval():
    est = HostEstimator(FakeModel(quadratic(rho=0.0), bounds=((C0 - SC, None), (0, 0.5))))
    iv = est.likelihood_intervals([C0, E0], params=['coverage'])['coverage']
    assert iv.flags['at_bound'] and not iv.flags['open']
    assert iv.lo == C0 - SC
    assert iv.hi == pytest.approx(C0 + Z * SC, abs=1e-3 * SC)


def test_disjoint_for_a_two_well_profile():
    def fn(c, e):
        w1 = -0.5 * ((c - C0) / SC) ** 2
        w2 = -1.0 - 0.5 * ((c - (C0 + 3.2 * SC)) / (0.3 * SC)) ** 2
        return np.maximum(w1, w2) - 0.5 * ((e - E0) / SE) ** 2
    est = HostEstimator(FakeModel(fn))
    iv = est.likelihood_intervals([C0, E0], params=['coverage'])['coverage']
    assert iv.flags['disjoint']
    assert iv.hi == pytest.approx(C0 + Z * SC, abs=1e-3 * SC)
    assert iv.lo == pytest.approx(C0 - Z * SC, abs=1e-3 * SC)


def test_moved_when_the_estimate_is_off_the_optimum():
    est = HostEstimator(FakeModel(quadratic(rho=0.0)))
    iv = est.likelihood_intervals([C0 - 0.5 * SC, E0], params=['coverage'])['coverage']
    assert iv.flags['moved']
    assert iv.lo == pytest.approx(C0 - Z * SC, abs=1e-3 * SC)
    assert iv.hi == pytest.approx(C0 + Z * SC, abs=1e-3 * SC)
    still = est.likelihood_intervals([C0, E0], params=['coverage'])['coverage']
    assert not still.flags['moved']


def test_span_doubles_until_the_threshold_is_crossed():
    # curvature 1 / SC^2 at the optimum (se = SC) but heavy tails: the crossing lies at ~6.75 se
    def fn(c, e):
        return -0.5 * np.log1p(((c - C0) / SC) ** 2) - 0.5 * ((e - E0) / SE) ** 2
    est = HostEstimator(FakeModel(fn))
    iv = est.likelihood_intervals([C0, E0], params=['coverage'])['coverage']
    half = SC * np.sqrt(np.expm1(chi2.ppf(0.95, 1)))
    assert half > 4 * SC
    assert not iv.flags['open'] and not iv.flags['at_bound']
    assert iv.hi == pytest.approx(C0 + half, abs=1e-2 * SC)
    assert iv.lo == pytest.approx(C0 - half, abs=1e-2 * SC)


def test_open_when_three_doublings_do_not_reach_the_threshold():
    def fn(c, e):
        return -1e-3 * np.log1p(((c - C0) / SC) ** 2) - 0.5 * ((e - E0) / SE) ** 2
    est = HostEstimator(FakeModel(fn))
    iv = est.likelihood_intervals([C0, E0], params=['coverage'])['coverage']
    assert iv.flags['open']


def test_fixed_parameters_get_no_interval():
    est = HostEstimator(FakeModel(quadratic()), fix=[None, E0])
    iv = est.likelihood_intervals([C0, E0])
    assert list(iv) == ['coverage']
    # with e held at its optimum the profile of c is the conditional one: se = SC * sqrt(1 - rho^2)
    assert iv['coverage'].hi - C0 == pytest.approx(Z * SC * np.sqrt(1 - 0.36), rel=1e-3)
    with pytest.raises(ValueError):
        est.likelihood_intervals([C0, E0], params=['error_rate'])
    with pytest.raises(ValueError):
        est.likelihood_intervals([C0, E0], level=1.0)


def test_error_scale_maps_the_error_rate_interval_back():
    est = HostEstimator(FakeModel(quadratic(rho=0.0)), err_scale=1000)
    iv = est.likelihood_intervals([C0, E0 * 1000], params=['error_rate'])['error_rate']
    assert iv.lo == pytest.approx(E0 - Z * SE, abs=1e-3 * SE)
    assert iv.hi == pytest.approx(E0 + Z * SE, abs=1e-3 * SE)


# ---- merge of per-rank rows ----------------------------------------------------------------------
def _synthetic_blocks(rng, W, n_seg, C=4):
    blocks = np.empty((W, n_seg, C))
    blocks[:, :, 0] = rng.choice([-5.0, -3.0, -1.0, -0.0, 0.0, -np.inf, np.nan], size=(W, n_seg))
    blocks[:, :, 1:] = rng.choice([0.5, 1.0, 2.0, np.nan], size=(W, n_seg, C - 1))
    empty = rng.uniform(size=(W, n_seg)) < 0.2
    blocks[empty, 0] = -np.inf
    blocks[empty, 1:] = np.nan
    return blocks


@pytest.mark.parametrize('W', [1, 2, 3, 5, 8])
def test_merge_segments_follows_merge_topk(W):
    rng = np.random.default_rng(W)
    blocks = _synthetic_blocks(rng, W, 400)
    got = parallel.merge_segments(blocks)
    for s in range(blocks.shape[1]):
        want = parallel.merge_topk(blocks[:, s, :], 1).numpy()[0]
        assert np.array_equal(got[s], want, equal_nan=True), (s, blocks[:, s, :], got[s], want)


def test_merge_segments_of_sharded_reference_rows_is_the_single_call():
    axes = [np.array([1.0, 2.0, 3.0]), np.array([0.1, 0.2]), np.array([0.3, 0.6, 0.9]),
            np.array([0.0, 0.5]), np.array([0.2, 0.4, 0.8])]
    lens = [len(a) for a in axes]
    total = int(np.prod(lens))
    block = int(np.prod(lens[2:]))
    rng = np.random.default_rng(3)
    ll = rng.choice([-3.0, -2.0, -1.0, -np.inf, np.nan], size=total)
    for mask in (1, 2, 3, 5, 16, 31):
        whole = reference_rows(ll, np.arange(total), axes, mask)
        for W in range(1, 9):
            parts = []
            for r in range(W):
                first, stride, blk, count = parallel.shard_blocked(total, block, r, W)
                i = np.arange(count)
                idx = (first + (i // blk) * stride) * blk + i % blk
                parts.append(reference_rows(ll[idx], idx, axes, mask))
            assert np.array_equal(parallel.merge_segments(np.stack(parts)), whole, equal_nan=True), (mask, W)


def test_reference_rows_order():
    axes = [np.array([1.0, 1.0, 2.0]), np.array([5.0, 6.0])]  # a repeated value on axis 0
    ll = np.array([-1.0, -1.0, np.nan, -2.0, -0.0, 0.0])
    rows = reference_rows(ll, np.arange(6), axes, 1)
    assert np.array_equal(rows[:, 0], [-1.0, -2.0, 0.0])
    assert rows[0, 2] == 5.0 and rows[2, 2] == 5.0  # ties go to the lower lattice index
    assert rows[1, 1] == 1.0 and rows[1, 2] == 6.0  # NaN counts as -inf
    assert np.signbit(rows[2, 0]) == False  # noqa: E712 -- -0 reported as +0
    rows = reference_rows([-np.inf], [5], axes, 2)  # a segment without a point, one all -inf
    assert np.isneginf(rows[0, 0]) and np.isnan(rows[0, 1:]).all()
    assert rows[1, 0] == -np.inf and rows[1, 2] == 6.0


# ---- validation -----------------------------------------------------------------------------------
def test_keep_mask_validation():
    assert engine.profile_segments([4, 5, 6, 7, 8], 1) == 4
    assert engine.profile_segments([4, 5, 6, 7, 8], 0b10110) == 5 * 6 * 8
    assert engine.profile_segments([4, 5], 3) == 20
    for bad in (0, -1, 1 << 5, 0b100001):
        with pytest.raises(ValueError):
            engine.profile_segments([4, 5, 6, 7, 8], bad)
    with pytest.raises(ValueError):
        engine.profile_segments([4, 5], 4)
    with pytest.raises(ValueError):
        engine.profile_segments([1 << 13] * 5, 31)


@pytest.mark.parametrize('argv', [['--ci', '0'], ['--ci', '1'], ['--ci', '1.5'], ['--ci', '-0.5'], ['--ci', 'x'],
                                  ['--ci', '0.95', '--load', 'out.yaml'], ['--ci', '0.95', '-ll']])
def test_ci_argument_errors(argv, capsys):
    with pytest.raises(SystemExit) as err:
        cli.run(['no_such.hist'] + argv)
    assert err.value.code == 2
    assert '--ci' in capsys.readouterr().err


def test_ci_defaults_to_off():
    args = cli.build_parser().parse_args(['h.hist'])
    assert args.ci is None
    assert cli.build_parser().parse_args(['h.hist', '--ci', '0.9']).ci == 0.9


# ---- genome size ------------------------------------------------------------------------------------
def test_genome_size_decreases_with_coverage():
    model = FakeModel(quadratic())
    hist = {1: 100, 5: 40, 10: 900, 11: 800, 20: 30}
    cs = np.linspace(2.0, 40.0, 50)
    for sf in (1, 3):
        gs = [data.genome_size(hist, model, c, sf) for c in cs]
        assert all(a >= b for a, b in zip(gs, gs[1:]))
        kmers = sum(j * h for j, h in hist.items())
        assert gs[0] == round(kmers / model.correct_c(cs[0] * sf))


def test_interval_report_keys():
    est = HostEstimator(FakeModel(quadratic()))
    iv = est.likelihood_intervals([C0, E0])
    hist = {1: 100, 10: 900, 11: 800}
    rep = data.interval_report(hist, est.model, 2, iv, 0.95)
    assert set(rep) == {'ci_level', 'coverage_ci', 'error_rate_ci', 'genome_size_ci', 'ci_flags'}
    assert rep['coverage_ci'] == [iv['coverage'].lo * 2, iv['coverage'].hi * 2]
    lo, hi = rep['genome_size_ci']
    assert lo == data.genome_size(hist, est.model, iv['coverage'].hi, 2)
    assert hi == data.genome_size(hist, est.model, iv['coverage'].lo, 2)
    assert lo < hi
    assert rep['ci_flags'] == {'coverage': [], 'error_rate': []}
