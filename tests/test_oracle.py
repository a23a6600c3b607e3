"""Pins the CPU oracle (oracle/covest_oracle.c) to the reference: every golden vector under
tests/golden/ was produced by the unmodified reference (gen_golden.py)."""
import math
import os

import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests.helpers import (case_ctor_kwargs, case_hist, golden_case_names, load_case,
                           load_tp_kat)


def _same(a, b):
    if isinstance(a, float) and isinstance(b, float) and math.isnan(a) and math.isnan(b):
        return True
    return a == b


def test_truncated_poisson_known_answers_bit_exact():
    for l, j, want in load_tp_kat():
        got = orc.truncated_poisson(l, j)
        assert _same(got, want), (l, j, got, want)


def test_survey_known_answers():
    # SURVEY.md section 8(c), measured on the reference
    assert orc.truncated_poisson(200.001, 200) == 28.211828828910424
    assert orc.truncated_poisson(7.9, 5) == 0.09510182368327921
    assert orc.truncated_poisson(11400, 11400) == math.inf
    hist = case_hist(load_case('e05_basic'))
    assert orc.Model('basic', 21, 100, hist, 0, max_error=8).loglik(10, .05) == -3678684.968587441
    rep = orc.Model('repeats', 21, 100, hist, 0, max_error=8)
    assert rep.loglik(10, .05, .8, .5, .5) == -3707976.263880685
    assert rep.loglik(10, .05, 1, 0, 0) == -3678684.968587441
    assert rep.loglik(10, .9, .1, 2, -1) == rep.loglik(10, .5, .3, 1, 0) == -31698818.11119928


@pytest.mark.parametrize('name', golden_case_names())
@pytest.mark.parametrize('mode', [orc.LADDER, orc.FAITHFUL])
def test_loglik_matches_reference_bit_exact(name, mode):
    case = load_case(name)
    if mode == orc.FAITHFUL and len(case['hist']) > 400:
        pytest.skip('one call per term is only exercised on the small cases')
    m = orc.Model(case['model'], case['k'], case['r'], case_hist(case), case['tail'],
                  **case_ctor_kwargs(case))
    got = m.loglik_batch(case['points'], mode=mode, threads=4)
    for p, g, w in zip(case['points'], got, case['ll']):
        assert _same(float(g), float(w)), (name, p, g, w)


@pytest.mark.parametrize('name', golden_case_names())
def test_probabilities_match_reference_bit_exact(name):
    case = load_case(name)
    m = orc.Model(case['model'], case['k'], case['r'], case_hist(case), case['tail'],
                  **case_ctor_kwargs(case))
    for idx, want in case['probs'].items():
        point = list(case['points'][int(idx)])
        # golden probabilities were taken at the clipped point (gen_golden._eval_point)
        for i, (lo, hi) in enumerate(m.bounds):
            if lo is not None and point[i] < lo:
                point[i] = lo
            elif hi is not None and point[i] > hi:
                point[i] = hi
        got = m.probs(point)
        assert all(_same(float(g), float(w)) for g, w in zip(got, want)), (name, idx)


def test_ladder_equals_one_call_per_term():
    rng = np.random.default_rng(5)
    for _ in range(50):
        lam = float(np.exp(rng.uniform(np.log(1e-10), np.log(3000))))
        j = int(rng.integers(1, 800))
        m = orc.Model('basic', 21, 100, {jj: 1 for jj in range(1, j + 1)}, 0, max_error=1)
        # with S=1 and a_0 = 1 the mixture is the truncated Poisson itself (times a_0 = n/n = 1)
        c = lam / ((100 - 21 + 1) / 100)
        a = m.probs([c, 0.0], mode=orc.LADDER)
        b = m.probs([c, 0.0], mode=orc.FAITHFUL)
        assert np.array_equal(a, b)


def test_restatement_against_compiled_reference_module():
    """The Python restatement of models.py (bench.py's CPU arm) reproduces the reference's stored
    values bit for bit: driven by the oracle's truncated_poisson (pinned to the reference above) on
    every small golden case, and driven by the reference's own compiled module when oracle/_ref has
    it."""
    for name in golden_case_names():
        case = load_case(name)
        if len(case['hist']) > 400:
            continue
        m = orc.Model(case['model'], case['k'], case['r'], case_hist(case), case['tail'],
                      **case_ctor_kwargs(case))
        for p, w in zip(case['points'][:12], case['ll'][:12]):
            assert _same(orc.py_loglik(m, list(map(float, p)), orc.truncated_poisson), float(w)), (name, p)
    ref = orc.ref_module()
    if ref is None:
        return
    for l, j, want in load_tp_kat()[:200]:
        assert _same(ref.truncated_poisson(l, j), want)
    case = load_case('e05_repeats')
    m = orc.Model('repeats', 21, 100, case_hist(case), 0, max_error=8)
    pts = case['points'][:12]
    got = orc.ref_loglik_batch(m, pts, processes=2)
    for g, w in zip(got, case['ll'][:12]):
        assert _same(float(g), float(w))
