"""The reference-facing API on the device: compute_loglikelihood_multi, lattices handed over as axes
(analytic plan) against explicit point arrays (general plan), grid-search rounds kept on the device,
the lock-step multi-start.  Needs a B200."""
import json
import os
import random

import numpy as np
import pytest

from covest_b200 import constants, grid, workload
from covest_b200.covest import CoverageEstimator
from covest_b200.histogram import process_histogram
from covest_b200.models import BasicModel, RepeatsModel
from tests.helpers import GOLDEN, case_hist, load_case

pytestmark = pytest.mark.gpu
constants.VERBOSE = False


def test_compute_loglikelihood_multi_is_the_batched_map():
    """models.py:109-117: {tuple(args): loglikelihood}, keyed by the arguments as given (unclipped);
    thread_count is accepted and ignored."""
    case = load_case('e05_repeats')
    model = RepeatsModel(21, 100, case_hist(case), 0, max_error=8)
    try:
        args_list = [tuple(p) for p in case['points'][:40]] + [(10, .9, .1, 2, -1)]
        got = model.compute_loglikelihood_multi(args_list, thread_count=3)
        assert list(got) == args_list or set(got) == set(args_list)
        for a in args_list:
            assert got[a] == model.compute_loglikelihood(*a)
        for a, want in zip(args_list[:40], case['ll'][:40]):
            assert got[a] == pytest.approx(want, rel=1e-9) or (np.isinf(want) and got[a] == want)
        assert got[(10, .9, .1, 2, -1)] == model.compute_loglikelihood(10, .5, .3, 1, 0)   # clipped, keyed unclipped
        assert model.compute_loglikelihood_multi([]) == {}
        lists = model.compute_loglikelihood_multi([[10, .05, .8, .5, .5]], 1)
        assert lists[(10, .05, .8, .5, .5)] == pytest.approx(-3707976.263880685, rel=1e-9)
    finally:
        model.close()
    basic = BasicModel(21, 100, case_hist(case), 0, max_error=8)
    try:
        assert basic.compute_loglikelihood_multi([(10, .05)])[(10, .05)] == pytest.approx(-3678684.968587441, rel=1e-9)
    finally:
        basic.close()


def test_counts_changed_in_place_reach_the_device():
    hist = case_hist(load_case('e05_basic'))
    model = BasicModel(21, 100, hist, 0, max_error=8)
    try:
        a = model.compute_loglikelihood(10, .05)
        first = next(iter(hist))
        hist[first] += 1000        # same dict object, same length
        b = model.compute_loglikelihood(10, .05)
        fresh = BasicModel(21, 100, dict(hist), 0, max_error=8)
        assert b != a and b == fresh.compute_loglikelihood(10, .05)
        fresh.close()
    finally:
        model.close()


@pytest.fixture(scope='module')
def cfg2():
    case = load_case('cfg2_repeats')
    model = RepeatsModel(21, 100, case_hist(case), 0, max_error=8)
    yield model
    model.close()


def test_lattice_by_axes_equals_explicit_points(cfg2):
    """The plan derived from the axes (no sort, nothing read back) and the general plan give the same
    values bit for bit -- also for unsorted and repeated axis values, values outside the bounds
    (clipped, models.py:60-69), slices and device buffers."""
    import torch
    ctx = cfg2.device_context
    axes = [np.geomspace(12, 80, 11), np.array([.05, .011, .03]), np.array([.9, .2, .55, 1.3, .31]),
            np.array([0., 1., .5, -1., .25, .75]), np.array([.6, .05, 1., .05, .333, 2., .11])]
    pts = workload.lattice_points(axes)
    ll_axes, rows = ctx.lattice_eval(axes, k_best=8)
    info = ctx.last_path_info()
    assert info['kernel'] == 'cvf_prefix_kernel' and info['analytic_plan'], info
    assert info['groups'] == 33 and info['q_runs'] == 33 * 7
    ll_pts = ctx.loglik(pts)
    assert not ctx.last_path_info()['analytic_plan']
    assert np.array_equal(ll_axes, ll_pts, equal_nan=True)
    order = np.lexsort((np.arange(len(ll_pts)), -ll_pts))[:8]
    assert np.array_equal(rows[:, 0], ll_pts[order]) and np.array_equal(rows[:, 1:], pts[order])
    # whole groups dealt to 3 "ranks"
    block = 5 * 6 * 7
    seen = np.full(len(pts), np.nan)
    for r in range(3):
        part, _ = ctx.lattice_eval(axes, first=r, stride=3, block=block)
        assert len(part) == 11 * block and ctx.last_path_info()['analytic_plan']   # 2310 points: the batched path
        i = np.arange(len(part))
        seen[(r + (i // block) * 3) * block + i % block] = part
    assert np.array_equal(seen, ll_pts, equal_nan=True)
    # device outputs: only enqueued
    dev_ll = torch.empty(len(pts), dtype=torch.float64, device='cuda')
    dev_rows = torch.empty((8, 6), dtype=torch.float64, device='cuda')
    ctx.lattice_eval(axes, k_best=8, out_ll=dev_ll, out_rows=dev_rows)
    torch.cuda.synchronize()
    assert np.array_equal(dev_ll.cpu().numpy(), ll_pts, equal_nan=True)
    assert np.array_equal(dev_rows.cpu().numpy(), rows)
    # a second lattice (other axes) right behind the first one on the same stream
    axes2 = [a * 1.01 if i < 2 else a for i, a in enumerate(axes)]
    ll2, _ = ctx.lattice_eval(axes2)
    assert np.array_equal(ll2, ctx.loglik(workload.lattice_points(axes2)), equal_nan=True)


def test_prefix_kernel_agrees_with_the_other_paths(cfg2):
    ctx = cfg2.device_context
    axes = [np.geomspace(10, 90, 9), np.geomspace(.01, .09, 5), np.linspace(.3, 1, 7), np.linspace(0, 1, 6),
            np.linspace(.02, 1, 23)]
    ll, _ = ctx.lattice_eval(axes)
    pts = workload.lattice_points(axes)
    try:
        ctx.set_path(ctx.PATH_PER_POINT)
        direct = ctx.loglik(pts)
        ctx.set_path(ctx.PATH_FACTORED_GEMM)
        gemm = ctx.loglik(pts)
    finally:
        ctx.set_path(ctx.PATH_AUTO)
    fin = np.isfinite(direct)
    assert np.array_equal(np.isfinite(ll), fin) and np.array_equal(np.isfinite(gemm), fin)
    assert np.max(np.abs(ll[fin] - direct[fin]) / np.abs(direct[fin])) <= 1e-11
    assert np.max(np.abs(gemm[fin] - direct[fin]) / np.abs(direct[fin])) <= 1e-11


def test_grid_rounds_on_the_device_walk_the_same_centres(cfg2):
    """optimize_grid through lattice_best (one row back per round) against the rounds evaluated as
    arrays with the reference's sequential bookkeeping (grid.py:56-72)."""
    est = CoverageEstimator(cfg2)
    start = [29.0, .031, .72, .48, .52]
    fn = est.likelihood_f
    on_device = list(grid.optimize_grid(fn, start, bounds=est.bounds))
    launches = est.launches

    class ArraysOnly:
        def __call__(self, x):
            return fn(x)

        def batch(self, pts):
            return fn.batch(pts)
    by_arrays = list(grid.optimize_grid(ArraysOnly(), start, bounds=est.bounds))
    assert on_device == by_arrays
    assert launches <= 40
    # with a fixed parameter and an error scale
    est2 = CoverageEstimator(cfg2, err_scale=10, fix=[None, None, None, .5, None])
    s2 = [29.0, .31, .72, .5, .52]
    a = list(grid.optimize_grid(est2.likelihood_f, s2, bounds=est2.bounds, fix=est2.fix))
    f2 = est2.likelihood_f

    class ArraysOnly2(ArraysOnly):
        def __call__(self, x):
            return f2(x)

        def batch(self, pts):
            return f2.batch(pts)
    b = list(grid.optimize_grid(ArraysOnly2(), s2, bounds=est2.bounds, fix=est2.fix))
    assert a == b and a[3] == .5


def test_lockstep_multi_start_reaches_the_polished_reference_optimum():
    """`-sp 8` with the lock-step optimiser on the cfg2 histogram of the e2e goldens: the best start
    ends at the optimum the polished reference run ends at (1e-6 on coverage, BASELINE.json)."""
    with open(os.path.join(GOLDEN, 'e2e_golden.json')) as f:
        g = json.load(f)['cfg2_repeats']
    hist = {int(j): int(h) for j, h in g['hist']}
    h2, tail, sf, gc, ge = process_histogram(hist, g['k'], g['r'], **g['flags'])
    model = RepeatsModel(g['k'], g['r'], h2, tail, max_error=8)
    try:
        guess = list(model.defaults)
        guess[:2] = gc, ge
        est = CoverageEstimator(model, optimizer='lockstep')
        random.seed(11)
        x, ok = est.compute_coverage(guess, starting_points=8)
        assert ok and est.launches < 250
        assert est.likelihood_f(x) <= g['polished']['objective'] * (1 + 1e-12)
        if est.likelihood_f(x) >= g['polished']['objective'] * (1 - 1e-10):   # the same optimum (not a better one)
            assert x[0] == pytest.approx(g['polished']['x'][0], rel=1e-6)
    finally:
        model.close()
