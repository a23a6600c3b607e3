"""Every number of error classes S (max_error, CvModelDesc.n_err) on every device path, against the
pinned C oracle.

S sets the term layout of every likelihood kernel: the profile kernel of the factored path pads a
copy to S rounded up to a multiple of 4 slots and packs 32 / that many copies into a tile (S <= 32
only; beyond, every mode falls back to the per-point kernel), the per-point kernel takes one copy
per group of terms and two passes of 32 terms per copy once S > 32, and the term-by-term kernel
a second pass of 32 classes.  The CLI uses S = 8, but BasicModel / RepeatsModel default to
S = k + 1 and the C ABI accepts any S in [1, min(k + 1, 64)].  The histograms cover the four
row-group widths NA = 1, 2, 4, 8 of the histogram tables (csrc/cvtables.h), one of them with a tail.
"""
import functools
import math

import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests.bigpoints import MASS_ULPS, ll_tolerance
from tests.helpers import case_hist, context_for, load_case, rel_err_ll

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-9    # BASELINE.json north_star: per-point log-likelihood within 1e-9 relative
P_RTOL = 1e-12    # SURVEY.md section 8(d): per-bin probabilities where p_j > 1e-300
FAST_RTOL = 1e-11  # the fast paths among themselves

S_ALL = [1, 2, 3, 5, 6, 7, 9, 11, 12, 13, 16, 17, 18, 22, 31, 32, 33, 40, 63, 64]
S_SOME = [1, 6, 12, 32, 33, 64]
K_NATURAL = [15, 31, 40, 63]  # max_error=None: S = k + 1

# histogram -> rows per group NA: e05 1, cfg2 2, dense400 4, cfg3 8, trim120 1 (with a tail of 175)
HISTS_FULL = ['cfg2_repeats', 'cfg3_repeats_dense1000', 'e05_repeats']
HISTS_SOME = ['dense400', 'cfg2_repeats_trim120']


def _cases():
    """(histogram, k, r, max_error) -- max_error None is the model's default S = k + 1."""
    out = []
    for name in HISTS_FULL + HISTS_SOME:
        for S in (S_ALL if name in HISTS_FULL else S_SOME):
            k = max(21, S - 1)
            out.append((name, k, 100, None if k in K_NATURAL and k + 1 == S else S))
        for k in K_NATURAL if name in HISTS_FULL else ():
            if (name, k, 100, None) not in out:
                out.append((name, k, 100, None))
    # shapes at the edges: k = 1 and 2 (S <= k + 1 <= 3), r = k (the smallest (r - k + 1) / r), cfg4's k and r
    out += [('cfg2_repeats', 1, 100, 2), ('cfg2_repeats', 2, 100, 3), ('e05_repeats', 21, 21, None),
            ('cfg2_repeats', 31, 150, 32)]
    return out


CASES = _cases()


def _case_id(case):
    name, k, r, S = case
    return '%s-S%d-k%d-r%d%s' % (name, k + 1 if S is None else S, k, r, '-default' if S is None else '')


@functools.lru_cache(maxsize=None)
def _hist(name):
    if name == 'dense400':  # 400 keys with counts: 7 groups of 4 rows
        j = np.arange(1, 401)
        h = np.rint(2e6 * np.exp(-0.5 * ((j - 24) / 6.0) ** 2) + 4e4 * np.exp(-j / 60.0) + 3)
        return dict(zip(j.tolist(), h.astype(int).tolist())), 0
    case = load_case(name)
    return case_hist(case), case['tail']


@functools.lru_cache(maxsize=None)
def _oracle(kind, case):
    name, k, r, S = case
    hist, tail = _hist(name)
    return orc.Model(kind, k, r, hist, tail, max_error=S)


def _n_err(case):
    return _oracle('repeats', case).max_error


def _clipped(m, pts):
    pts = np.array(pts, dtype=np.float64)
    for i, (lo, hi) in enumerate(m.bounds):
        pts[:, i] = np.clip(pts[:, i], -np.inf if lo is None else lo, np.inf if hi is None else hi)
    return pts


def _gate(m, pts, want, rtol):
    """How close a device value must be to the oracle's `want` at `pts`: rtol * |ll|; with a tail, plus
    what MASS_ULPS ulps of the mass move tail * log(1 - mass) by (tests/bigpoints.py: that term is
    ill-conditioned where nearly all mass is inside the histogram).  Where the mass is within those
    ulps of 1, the last bit decides whether the reference adds the term at all (mass < 1,
    models.py:103-104): there `base` holds the value without the term (NaN elsewhere), see
    _assert_close."""
    gate = dict(tol=rtol * np.abs(want), base=np.full(len(want), np.nan), rtol=rtol, tail=m.tail)
    if m.tail:
        omm = np.array([1.0 - math.fsum(m.probs(p)) for p in _clipped(m, pts)])
        gate['tol'] = ll_tolerance(dict(ll=want, tail=m.tail, one_minus_mass=omm), rtol)
        near = np.abs(omm) <= MASS_ULPS * 2.0 ** -53
        with np.errstate(divide='ignore', invalid='ignore'):
            gate['base'] = np.where(near, want - np.where(omm > 0, m.tail * np.log(omm), 0.0), np.nan)
    return gate


def _assert_close(got, want, gate, what):
    """got within gate['tol'] of want.  Where gate['base'] is set, instead: got is the value without
    the tail term (within rtol), or that value plus the tail term of a mass within 2 MASS_ULPS ulps of
    1, i.e. tail * log(1 - mass) in [tail * log(2^-53), tail * log(2 MASS_ULPS 2^-53)]."""
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), (what, 'the -inf sets differ')
    fin = np.isfinite(want)
    with np.errstate(invalid='ignore'):  # -inf - -inf: those points are compared as -inf sets
        ok = np.abs(got - want) <= gate['tol']
    near = fin & ~np.isnan(gate['base'])
    if near.any():
        base = gate['base'][near]
        d = got[near] - base
        slack = gate['rtol'] * np.abs(base)
        lo = gate['tail'] * math.log(2.0 ** -53) - slack
        hi = gate['tail'] * math.log(2 * MASS_ULPS * 2.0 ** -53) + slack
        ok[near] = (np.abs(d) <= slack) | ((d >= lo) & (d <= hi))
    bad = fin & ~ok
    assert not bad.any(), (what, int(bad.sum()), float(rel_err_ll(got[fin], want[fin]).max()))


# ---- 1. the repeats lattice on every path ------------------------------------------------------
# q down to 0.05: cut-offs of up to ~300 copies, many K-chunks of the profile kernel (16 copies each);
# 300 copies x 40 x 0.8 stays below the rates where the reference overflows (~11 360).
# n_s = comb[s] * (1.0 - exp(-l_s)) is exactly 0 once l_s < 2^-53: at e = 0.03 every class above 8 is
# dead.  e = 0.3 gives classes up to ~16 a weight, so that the profile kernel's later MMA slices of a
# copy (4 classes each) hold live terms.  Its small rates put the counted bins beyond ~20 out of the
# double range (-inf), so it runs on the 15-bin histogram, which takes the full list of S.
HIGH_ERROR_HISTS = ('e05_repeats',)
AUTO_MIN_POINTS = 2048  # include/covest_b200.h, cvb_set_path: smaller batches take the per-point kernel


@functools.lru_cache(maxsize=None)
def _lattice(name):
    """(axes, the same lattice as explicit points, last axis fastest)."""
    errs = [0.004, 0.03] + ([0.3] if name in HIGH_ERROR_HISTS else [])
    axes = (np.array([20.0, 40.0]), np.array(errs), np.array([0.3, 0.65, 1.0]), np.array([0.0, 0.5, 1.0]),
            np.array([0.05, 0.1, 0.2, 0.4, 0.7, 1.0]))
    return axes, np.ascontiguousarray(np.array(np.meshgrid(*axes, indexing='ij')).reshape(5, -1).T)

PATHS = {'auto': 0, 'per_point': 1, 'gemm': 3, 'prefix': 4, 'term_by_term': 5}


@functools.lru_cache(maxsize=None)
def _lattice_oracle(case):
    m = _oracle('repeats', case)
    pts = _lattice(case[0])[1]
    want = m.loglik_batch(pts, threads=8)
    assert not np.any(np.isnan(want) | np.isposinf(want))  # inside the reference's numeric domain
    return want, _gate(m, pts, want, LL_RTOL), _gate(m, pts, want, FAST_RTOL)


@functools.lru_cache(maxsize=None)
def _lattice_device(case, path):
    """(lattice_eval values, loglik values on the explicit grid, path info of each)."""
    axes, pts = _lattice(case[0])
    with context_for(_oracle('repeats', case)) as ctx:
        ctx.set_path(PATHS[path])
        by_axes, _ = ctx.lattice_eval(axes)
        info_axes = ctx.last_path_info()
        by_points = ctx.loglik(pts)
        info_points = ctx.last_path_info()
    return np.array(by_axes), np.array(by_points), info_axes, info_points


def _expected_kernel(path, S, n_points):
    """The kernel include/covest_b200.h (cvb_set_path) promises for a repeats batch."""
    if path == 'term_by_term':
        return 'cv_faithful_kernel'
    if S > 32 or path == 'per_point' or (path == 'auto' and n_points < AUTO_MIN_POINTS):
        return 'cv_loglik_kernel'  # the factored path holds S <= 32 only: every other mode falls back
    return {'gemm': 'cvf_gemm_kernel', 'prefix': 'cvf_prefix_kernel'}[path]


@pytest.mark.parametrize('path', list(PATHS))
@pytest.mark.parametrize('case', CASES, ids=_case_id)
def test_lattice_on_every_path_matches_the_oracle(case, path):
    S = _n_err(case)
    want, gate, gate_fast = _lattice_oracle(case)
    by_axes, by_points, info_axes, info_points = _lattice_device(case, path)
    kernel = _expected_kernel(path, S, len(by_points))
    for info in (info_axes, info_points):
        assert info['kernel'] == kernel, (info['kernel'], kernel)
        if S <= 32 and path in ('gemm', 'prefix'):
            assert info['path'] == 'factored' and info['kernel'] in ('cvf_gemm_kernel', 'cvf_prefix_kernel')
    if kernel == 'cvf_prefix_kernel':
        assert info_axes['analytic_plan']  # the plan of lattice_eval follows from the axes
    # the two ways of handing over the same points are the same evaluation
    assert np.array_equal(by_axes, by_points, equal_nan=True)
    _assert_close(by_points, want, gate, (path, 'oracle'))
    if path not in ('per_point', 'term_by_term'):
        ref = _lattice_device(case, 'per_point')[1]
        _assert_close(by_points, ref, gate_fast, (path, 'per-point kernel'))


# ---- 2. random points, both models -------------------------------------------------------------
# coverages at which a far-off point has bins with counts in the subnormal band at e = 0.01 on the
# 1000-bin histogram: S = 5 (k = 21), S = 33 (k = 32), S = 64 (k = 63) -- re-evaluated term by term
FAR_COVERAGES = (7.2, 9.3, 23.0)
MARKED_ON_CFG3 = (5, 33, 64)


@functools.lru_cache(maxsize=None)
def _random_points(n_params, tail=False):
    n = 48
    rng = np.random.default_rng(2024)
    cols = [30 * 3 ** rng.uniform(-1, 1, n), np.exp(rng.uniform(np.log(1e-4), np.log(.5), n))]
    if tail:  # where the histogram holds most of the mass, as tests/bigpoints.py does for its tail config:
        # with all but ~1e-14 of it inside, the mass's last ulps decide tail * log(1 - mass)
        cols = [30 * 3 ** rng.uniform(-.5, .5, n), np.exp(rng.uniform(np.log(3e-3), np.log(.2), n))]
    if n_params == 5:
        cols += [rng.uniform(.3, 1, n), rng.uniform(0, 1, n), rng.uniform(.02, 1, n)]
    pts = np.column_stack(cols)
    # the first rows stay inside the bounds (the probabilities below are taken there): bound values
    if n_params == 5:
        pts[0] = [30, 0.0, .7, .5, .5]
        pts[1] = [30, .03, 1.0, .5, .5]
        pts[2] = [30, .03, .7, 0.0, .5]
        pts[3] = [30, .03, .7, .5, 0.0]
        pts[4] = [30, .03, .7, .5, 1.0]
        pts[5] = [12, .2, .4, .3, .1]
        far = [[c, .01, 1.0, 0.0, 0.0] for c in FAR_COVERAGES] + [[30, .9, .1, 2, -1], [0.001, .03, .7, .5, .5]]
    else:
        pts[0] = [30, 0.0]
        pts[1] = [30, 0.5]
        pts[2] = [12, .2]
        far = [[c, .01] for c in FAR_COVERAGES] + [[30, .9], [0.001, .03]]
    pts[-len(far):] = far
    return np.ascontiguousarray(pts)


@pytest.mark.parametrize('kind', ['repeats', 'basic'])
@pytest.mark.parametrize('case', CASES, ids=_case_id)
def test_random_points_match_the_oracle(case, kind):
    m = _oracle(kind, case)
    pts = _random_points(m.n_params, bool(m.tail))
    want = m.loglik_batch(pts, threads=8)
    # parity is defined inside the reference's numeric domain (its long double product overflows at
    # rates above ~11 360: +inf / NaN there)
    inside = ~(np.isposinf(want) | np.isnan(want))
    assert inside.sum() >= 0.75 * len(pts)
    gate = _gate(m, pts[inside], want[inside], LL_RTOL)
    with context_for(m) as ctx:
        for path in ('per_point', 'auto', 'term_by_term'):
            ctx.set_path(PATHS[path])
            got = ctx.loglik(pts)
            info = ctx.last_path_info()
            assert info['kernel'] == ('cv_faithful_kernel' if path == 'term_by_term' else 'cv_loglik_kernel')
            _assert_close(got[inside], want[inside], gate, path)
            if path == 'per_point' and case[0] == 'cfg3_repeats_dense1000' and m.max_error in MARKED_ON_CFG3:
                assert info['refined_points'] > 0


# ---- 3. per-bin probabilities -------------------------------------------------------------------
ZERO_UNITS = 64  # units of 2^-1074 a device probability may show where the reference's is 0


@pytest.mark.parametrize('kind', ['repeats', 'basic'])
@pytest.mark.parametrize('case', CASES, ids=_case_id)
def test_probabilities_match_the_oracle(case, kind):
    m = _oracle(kind, case)
    pts = _random_points(m.n_params, bool(m.tail))[:6]
    assert np.array_equal(_clipped(m, pts), pts)  # the oracle's probs do not clip
    with context_for(m) as ctx:
        got, ll = ctx.probs(pts, clip=True, with_loglik=True)
    for i, row in enumerate(got):
        want = m.probs(pts[i])
        ok = want > 1e-300
        rel = np.abs(row[ok] - want[ok]) / want[ok]
        assert not ok.any() or rel.max() <= P_RTOL, (i, float(rel.max()))
        # exact zeros where the reference has them -- up to a few units of the subnormal grid: there the
        # reference's per-term roundings decide (csrc/cvmodel.h, CV_P_BAND), and the log-likelihood of
        # such a point is evaluated again term by term, its per-bin probabilities are not
        zero = want == 0
        assert np.all(row[zero] <= ZERO_UNITS * 2.0 ** -1074), (i, float(row[zero].max() / 2.0 ** -1074))
    want_ll = m.loglik_batch(pts)
    _assert_close(ll, want_ll, _gate(m, pts, want_ll, LL_RTOL), 'probs loglik')


# ---- 4. the sweep can see one class too few -----------------------------------------------------
def _class_weights(m, point):
    """a_s of the first copy (models.py:81-88, :221-229) as the oracle's model computes it."""
    c, e = point[0], point[1]
    ck = c * (m.r - m.k + 1) / m.r
    l_s = [ck * 3.0 ** -s * (1.0 - e) ** (m.k - s) * e ** s for s in range(m.max_error)]
    n_s = [m.comb[s] * (1.0 - math.exp(-l_s[s])) for s in range(m.max_error)]
    return np.array(n_s) / (sum(n_s) or 1)


# (S, k, coverages, error rates): the last class has a weight above 1e-6 only where e is large enough.
# n_s = comb[s] * (1.0 - exp(-l_s)) is exactly 0 in double arithmetic once l_s < 2^-53, so the classes
# near 32 also take a coverage of 10^12 or more: l_s = c_k 3^-s (1 - e)^(k - s) e^s is c_k 6^-s 2^-(k - s)
# at e = 0.5.  With k = 32 class 32 weighs at most 2^-32, hence k = 40 at S = 32 and 33.
SENSITIVITY = [(2, 21, (10.0, 40.0), (.02, .05)), (5, 21, (10.0, 40.0), (.15, .3)), (12, 21, (10.0, 40.0), (.4, .5)),
               (16, 21, (10.0, 40.0), (.4, .5)), (32, 40, (1e12, 1e13), (.5,)), (33, 40, (1e12, 1e13), (.5,))]


@pytest.mark.parametrize('S,k,covs,errs', SENSITIVITY, ids=['S%d' % s[0] for s in SENSITIVITY])
def test_a_context_without_the_last_class_fails_the_gate(S, k, covs, errs):
    """On every kernel that holds the model: for S <= 32 also the factored path, whose profile kernel
    puts class S - 1 into the last MMA slice of a copy."""
    hist, tail = _hist('e05_repeats')  # 15 bins: the small rates of large error rates keep p_15 finite
    full = orc.Model('repeats', k, 100, hist, tail, max_error=S)
    short = orc.Model('repeats', k, 100, hist, tail, max_error=S - 1)
    pts = np.array([[c, e, q1, .5, .3] for c in covs for e in errs for q1 in (.5, 1.0)])
    assert all(_class_weights(full, p)[S - 1] > 1e-6 for p in pts)
    want = full.loglik_batch(pts)
    assert np.isfinite(want).all()
    for path in ('per_point', 'gemm', 'prefix') if S <= 32 else ('per_point',):
        with context_for(full) as ctx:
            ctx.set_path(PATHS[path])
            same = ctx.loglik(pts)
            assert ctx.last_path_info()['kernel'] == _expected_kernel(path, S, len(pts))
        with context_for(short) as ctx:
            ctx.set_path(PATHS[path])
            dropped = ctx.loglik(pts)
            assert ctx.last_path_info()['kernel'] == _expected_kernel(path, S - 1, len(pts))
        assert rel_err_ll(same, want).max() <= LL_RTOL, path
        assert np.all(rel_err_ll(dropped, want) > LL_RTOL), (path, rel_err_ll(dropped, want))


# ---- 5. k > 63: the default S = k + 1 is more than the library holds -------------------------------
@pytest.mark.parametrize('cls', ['BasicModel', 'RepeatsModel'])
def test_default_max_error_above_64_is_an_error(cls):
    from covest_b200 import models
    from covest_b200.engine import DeviceError
    hist, _ = _hist('e05_repeats')
    model = getattr(models, cls)(70, 100, hist, 0)
    assert model.max_error == 71
    try:
        with pytest.raises(DeviceError, match='max_error'):
            model.device_context
        with pytest.raises(DeviceError, match='max_error'):
            model.loglikelihood_batch(np.array([[10.0, .05, .5, .5, .5][:model.param_count]]))
    finally:
        model.close()
