"""The per-point formulation at every number of error classes S, without a GPU.

tests/host_math/emulate.cpp runs the phase functions of the per-point kernel (csrc/cvpoint.h) lane by
lane.  S decides how many copies share a group of 32 terms and, beyond 32, how many passes of 32
terms a copy takes; the CLI's S = 8 and the k + 1 = 22 of the golden cases leave most of those
layouts unvisited.  Here every S of the sweep is compared with the oracle on random points of the
box, both models, on a 163-key (2 rows per group) and a 1000-key (8 rows per group) histogram.  The
factored and term-by-term kernels have no host emulation: tests/test_gpu_error_classes.py.
"""
import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests import emulation as emu
from tests.helpers import case_hist, load_case, rel_err_ll

LL_RTOL = 1e-9  # BASELINE.json north_star: per-point log-likelihood within 1e-9 relative

# (S, k): k = 21 where S allows it, k + 1 = S at the large S, and the small k where S <= k + 1 <= 3
SWEEP = [(1, 21), (2, 1), (2, 21), (3, 2), (3, 21), (5, 21), (6, 5), (6, 21), (9, 21), (12, 11), (12, 63),
         (17, 21), (32, 31), (33, 32), (33, 40), (41, 40), (41, 63), (64, 63)]
HISTS = {'cfg2_repeats': 60, 'cfg3_repeats_dense1000': 24}  # histogram -> points


@pytest.mark.parametrize('kind', ['basic', 'repeats'])
@pytest.mark.parametrize('name', list(HISTS))
@pytest.mark.parametrize('S,k', SWEEP, ids=['S%d-k%d' % sk for sk in SWEEP])
def test_emulated_loglik_matches_the_oracle_at_every_S(S, k, name, kind):
    case = load_case(name)
    m = orc.Model(kind, k, 100, case_hist(case), case['tail'], max_error=S)
    assert m.max_error == S
    n = HISTS[name]
    rng = np.random.default_rng(1000 * S + k)
    cols = [30 * 3 ** rng.uniform(-1, 1, n), np.exp(rng.uniform(np.log(1e-4), np.log(.5), n))]
    if kind == 'repeats':
        cols += [rng.uniform(.3, 1, n), rng.uniform(0, 1, n), rng.uniform(.05, 1, n)]
    pts = np.column_stack(cols)
    want = m.loglik_batch(pts, threads=8)
    got = emu.loglik_batch(m, pts)
    # marked points: the GPU's term-by-term kernel; beyond the reference's overflow (~11 360): no parity
    keep = ~emu.marked(got) & ~(np.isposinf(want) | np.isnan(want))
    assert keep.mean() >= 0.75
    assert np.array_equal(np.isneginf(got[keep]), np.isneginf(want[keep]))
    rel = rel_err_ll(got[keep], want[keep])
    assert rel.max() <= LL_RTOL, (int(rel.argmax()), pts[keep][int(rel.argmax())])
