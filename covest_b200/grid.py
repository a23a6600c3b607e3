"""Candidate generators of the estimator, evaluated a whole set per device launch
(reference: covest/grid.py).

initial_grid      the random multi-start points (grid.py:82-114)
optimize_grid     the multiplicative grid refinement (grid.py:17-79): every round's Cartesian
                  candidate set -- 6^n points, 7776 for the repeats model -- is one batched
                  evaluation instead of a Pool.map over pickled calls.

`fn` may be any scalar objective.  If it has a `batch` attribute (CoverageEstimator.likelihood_f
does) the round is a single call `fn.batch(list_of_points)`; a plain function is simply mapped.
"""
import itertools
import random

import numpy as np

from . import constants
from .perf import running_time, running_time_decorator
from .utils import verbose_print


def evaluate_all(fn, points):
    """Objective values of `points`, through fn.batch when the objective offers it."""
    if not isinstance(points, np.ndarray):
        points = list(points)
    if len(points) == 0:
        return []
    batch = getattr(fn, 'batch', None)
    if batch is not None:
        return [float(v) for v in batch(points)]
    return [fn(p) for p in points]


def _interval_in_bounds(interval, bounds, i):
    if bounds is None or len(bounds) <= i or len(bounds[i]) != 2:
        return interval
    lo, hi = interval
    b_lo, b_hi = bounds[i]
    if b_lo is not None:
        lo = max(lo, b_lo)
    if b_hi is not None:
        hi = min(hi, b_hi)
    return lo, hi


def _inside(value, bounds, i):
    if bounds is None or len(bounds) <= i or len(bounds[i]) != 2:
        return True
    lo, hi = bounds[i]
    return (lo is None or value >= lo) and (hi is None or value <= hi)


def grid_axes(center, step, depth, bounds=None, fix=None):
    """Per coordinate the candidate values center_i * step**d, d in -depth..depth without 0, kept
    inside the bounds; a fixed coordinate contributes its fixed value only (grid.py:20-43).  The
    centre itself is never a candidate and a zero coordinate stays zero."""
    axes = []
    for i, var in enumerate(center):
        if fix is not None and fix[i] is not None:
            axes.append([fix[i]])
            continue
        axes.append([v for v in (var * step ** d for d in range(-depth, depth + 1) if d != 0)
                     if _inside(v, bounds, i)])
    return axes


def grid_candidates(center, step, depth, bounds=None, fix=None):
    """Cartesian product of grid_axes, in the order of itertools.product (grid.py:33)."""
    return list(itertools.product(*grid_axes(center, step, depth, bounds, fix)))


def _product_rows(axes):
    """The rows of itertools.product(*axes) as one float64 array (last axis fastest)."""
    if any(len(a) == 0 for a in axes):
        return np.empty((0, len(axes)))
    mesh = np.meshgrid(*[np.asarray(a, dtype=np.float64) for a in axes], indexing='ij')
    return np.ascontiguousarray(np.stack([m.ravel() for m in mesh], axis=1))


@running_time_decorator
def optimize_grid(fn, initial_guess, bounds=None, maximize=False, fix=None,
                  n_threads=constants.DEFAULT_THREAD_COUNT):
    """Shrinking multiplicative grid search around the best point so far; returns the best
    arguments.  `n_threads` is accepted for compatibility (the reference forks that many
    workers); evaluation is batched instead."""
    if fix is None:
        fix = [None] * len(initial_guess)
    sign = -1 if maximize else 1
    best_val = sign * evaluate_all(fn, [initial_guess])[0]
    best_args = initial_guess
    step = constants.STEP
    depth = constants.GRID_DEPTH
    diff = 1
    rounds = 0
    try:
        while diff > 0.1 or step > 1.001:
            rounds += 1
            diff = 0.0
            batch = getattr(fn, 'batch', None)
            lattice_best = getattr(fn, 'lattice_best', None) if not maximize else None
            found = None
            if lattice_best is not None:
                # the round stays on the device: candidates generated there from the axes, the
                # arg-min taken there, one row comes back.  The sequential bookkeeping of
                # grid.py:65-69 adds up the strict improvements in candidate order, which
                # telescopes to (best before the round) - (best of the round), and keeps the FIRST
                # candidate that attains the minimum -- the tie-break of the device's top-K.
                axes = grid_axes(best_args, step, depth, bounds, fix)
                size = int(np.prod([len(a) for a in axes]))
                verbose_print('Iter : {}, Grid size: {}'.format(rounds, size))
                with running_time('grid iteration'):
                    found = lattice_best(axes) if size else (float('inf'), None)
            if found is not None:
                value, point = found
                if point is not None and value < best_val:
                    diff += best_val - value
                    best_val = value
                    best_args = point
            elif batch is not None:
                # the whole round as one array and one launch; the bookkeeping of grid.py:65-69
                # (strict improvements in candidate order, its use of the raw value included) on
                # the running minimum
                grid = _product_rows(grid_axes(best_args, step, depth, bounds, fix))
                verbose_print('Iter : {}, Grid size: {}'.format(rounds, len(grid)))
                with running_time('grid iteration'):
                    values = np.asarray(batch(grid), dtype=np.float64) if len(grid) else np.empty(0)
                signed = sign * values
                before = np.fmin.accumulate(np.concatenate(([best_val], signed)))[:-1]
                for i in np.nonzero(signed < before)[0]:
                    diff += float(before[i]) - float(values[i])
                    best_val = float(signed[i])
                    best_args = tuple(float(v) for v in grid[i])
            else:
                grid = grid_candidates(best_args, step, depth, bounds, fix)
                verbose_print('Iter : {}, Grid size: {}'.format(rounds, len(grid)))
                with running_time('grid iteration'):
                    values = evaluate_all(fn, grid)
                # same sequential bookkeeping as grid.py:65-69, including its use of the raw value
                for args, val in zip(grid, values):
                    if sign * val < best_val:
                        diff += best_val - val
                        best_val = sign * val
                        best_args = args
            if diff < 1.0:
                step = 1 + (step - 1) * 0.75
            verbose_print('d:{} s:{}'.format(diff, step))
            verbose_print('New args: {}, ll: {}'.format(best_args, best_val))
    except KeyboardInterrupt:
        verbose_print('Grid search interrupted')
    verbose_print('Number of iterations in grid search:{}'.format(rounds))
    return best_args


def initial_grid(initial_guess, count=constants.INITIAL_GRID_COUNT, bounds=None, fix=None):
    """`count` starting points: the guess itself, then count-1 points with every free coordinate
    drawn uniformly from [v / 3, 3 v] cut to the bounds (grid.py:82-114; Python's global
    `random`, seed it for reproducible runs)."""
    if fix is None:
        fix = [None] * len(initial_guess)
    if count < 1:
        return []
    step = constants.INITIAL_GRID_STEP
    points = [initial_guess]
    for _ in range(count - 1):
        boxes = [_interval_in_bounds((v / step, v * step), bounds, i)
                 for i, v in enumerate(initial_guess)]
        points.append([random.uniform(*box) if fix[i] is None else fix[i]
                       for i, box in enumerate(boxes)])
    return points


def lattice_search(model, axes, k_best=64):
    """Best rows of a Cartesian candidate lattice, sharded over the ranks of torch.distributed
    when it is initialised (SURVEY.md section 8(e)): the (coverage, error_rate) groups of the
    lattice are dealt round-robin to the ranks, every rank evaluates its groups with points
    generated on the device, the per-rank best rows are all-gathered, and every rank returns the
    same global (k_best, 1 + n_param) best-first array."""
    from . import parallel
    lens = [len(a) for a in axes]
    total = int(np.prod(lens))
    block = int(np.prod(lens[2:])) if len(lens) > 2 else 1
    ctx = model.device_context

    def evaluate_slice(first, stride, block, count):
        _, rows = ctx.lattice_eval(axes, first=first, stride=stride, block=block, count=count,
                                   want_ll=False, k_best=k_best)
        rank, world = parallel.world()
        if world > 1:
            import torch
            return torch.from_numpy(rows).to(torch.device('cuda', ctx.device))
        return rows

    rows = parallel.sharded_best_rows(evaluate_slice, total, k_best, block=block)
    return rows.cpu().numpy() if hasattr(rows, 'cpu') else np.asarray(rows)


def lattice_profile(model, axes, keep_mask):
    """The profile rows of a Cartesian lattice (LikelihoodContext.lattice_profile): for every segment --
    every combination of values of the axes whose bit is set in keep_mask, last kept axis fastest -- the
    (loglik, params...) row of its best point.  Sharded like lattice_search: every rank profiles its
    whole (coverage, error_rate) groups, the (n_seg, 1 + n_param) blocks are all-gathered and merged
    segment by segment on the host (parallel.merge_segments).  With ascending axes every rank returns
    the rows of one call over the whole lattice, whatever the number of ranks."""
    from . import parallel
    lens = [len(a) for a in axes]
    total = int(np.prod(lens))
    block = int(np.prod(lens[2:])) if len(lens) > 2 else 1
    ctx = model.device_context
    rank, world = parallel.world()
    first, stride, block, count = parallel.shard_blocked(total, block, rank, world)
    rows = ctx.lattice_profile(axes, keep_mask, first=first, stride=stride, block=block, count=count)
    if world == 1:
        return rows
    device = None
    import torch.distributed as dist
    if dist.get_backend() == 'nccl':
        import torch
        device = torch.device('cuda', ctx.device)
    gathered = parallel.allgather_rows(parallel.to_comm(rows, device)).cpu().numpy()
    return parallel.merge_segments(gathered.reshape(world, rows.shape[0], rows.shape[1]))
