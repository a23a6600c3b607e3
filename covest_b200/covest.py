"""CoverageEstimator and the `covest` command line (reference: covest/covest.py), with every
likelihood evaluation on the device and every candidate set -- finite-difference stencils,
multi-start fronts, grid rounds -- a single batched launch.

What is kept: constructor, likelihood_f / _optimize / compute_coverage signatures and semantics
(scipy L-BFGS-B with its own forward-difference gradient, bounds, err_scale, fix), argparse flags,
YAML report.  What changes is scheduling only:

  * the n perturbed points of a forward-difference gradient are handed to scipy through its
    `workers` map hook and evaluated as one launch (the reference: n+1 sequential objective calls);
  * the starts of a multi-start run live in threads whose evaluations are merged into common
    launches by a LaunchBatcher (the reference: one forked process per start, covest.py:67-68);
  * grid-search rounds are one launch each (grid.py); for a device-resident model the round is
    handed over as its axes and only the best candidate comes back (cvb_lattice_eval, k_best = 1).

Additions (not in the reference):

  * `optimizer='lockstep'` (CLI `--optimizer lockstep`): the multi-start refinement as a lock-step
    projected Newton iteration, all starts per launch (optimizer.py), instead of scipy in threads;
  * under torch.distributed (one process per GPU, torchrun) the starts of a multi-start run are
    dealt round-robin to the ranks, refined there, and the refined optima are all-gathered
    (`refine_starts`); `compute_coverage_from_lattice` first evaluates a sharded candidate lattice
    and takes the global best rows as starts (SURVEY.md section 8(e));
  * `polish` (CLI `--polish`): Newton iteration on central differences.

`-T / n_threads` is accepted and ignored.
"""
import argparse
import os
import threading
from pathlib import Path

import numpy as np
from scipy.optimize import minimize

from . import constants, version_string
from .data import interval_report, load_histogram, parse_data, print_output, save_histogram
from . import parallel
from .grid import initial_grid, lattice_profile, lattice_search, optimize_grid
from .optimizer import lockstep_minimize
from .histogram import process_histogram
from .models import models, select_model
from .perf import running_time, running_time_decorator
from .utils import nonefloat, verbose_print


class LaunchBatcher:
    """Merges the evaluation requests of several client threads into common device launches: a
    launch happens when every client that is still running has a request pending."""

    def __init__(self, evaluate, n_clients):
        self._evaluate = evaluate
        self._active = n_clients
        self._cv = threading.Condition()
        self._pending = []
        self.launches = 0
        self.points = 0

    def submit(self, points):
        points = [list(p) for p in points]
        slot = {'points': points, 'values': None, 'error': None}
        with self._cv:
            self._pending.append(slot)
            if len(self._pending) >= self._active:
                self._flush()
            while slot['values'] is None and slot['error'] is None:
                self._cv.wait()
        if slot['error'] is not None:
            raise slot['error']
        return slot['values']

    def retire(self):
        """A client is done and will not submit again."""
        with self._cv:
            self._active -= 1
            if self._pending and len(self._pending) >= self._active:
                self._flush()

    def _flush(self):  # holds the lock
        batch, self._pending = self._pending, []
        flat = [p for slot in batch for p in slot['points']]
        try:
            values = list(self._evaluate(flat))
            self.launches += 1
            self.points += len(flat)
            at = 0
            for slot in batch:
                n = len(slot['points'])
                slot['values'] = values[at:at + n]
                at += n
        except BaseException as exc:  # hand the failure to every waiting client
            for slot in batch:
                slot['error'] = exc
        self._cv.notify_all()


class _Objective:
    """estimator.likelihood_f: callable on one point like the reference's bound method
    (covest.py:26-31), plus `.batch(points)` for whole candidate sets."""

    def __init__(self, estimator):
        self._est = estimator

    def __call__(self, x):
        return float(self._est.likelihood_batch([x])[0])

    def batch(self, points):
        return self._est.likelihood_batch(points)

    def lattice_best(self, axes):
        """(objective, point) of the best candidate of the Cartesian lattice of `axes` (optimiser
        coordinates, last axis fastest; ties to the first candidate in itertools.product order) --
        or None when the model has no device lattice evaluator.  One grid-search round
        (grid.py:56-69) without the candidates or their values crossing the bus."""
        return self._est.lattice_best(axes)


class CoverageEstimator:
    def __init__(self, model, err_scale=1, fix=None, optimizer=None):
        self.model = model
        self.fix = fix
        self.err_scale = err_scale
        # 'scipy': L-BFGS-B per start, as the reference; 'lockstep': optimizer.py (multi-start only)
        self.optimizer = optimizer or os.environ.get('COVEST_B200_OPTIMIZER', 'scipy')
        if self.optimizer not in ('scipy', 'lockstep'):
            raise ValueError('optimizer must be scipy or lockstep')
        self.bounds = list(self.model.bounds)
        self.bounds[1] = self.bounds[1][0], self.bounds[1][1] * self.err_scale
        self.launches = 0
        self.evaluations = 0

    # -- objective --------------------------------------------------------------------------
    def _model_rows(self, points):
        rows = np.array(points, dtype=np.float64)  # a copy: fix / err_scale are applied in place
        rows = rows.reshape(len(points), self.model.param_count)
        if self.fix is not None:
            for i, v in enumerate(self.fix):
                if v is not None:
                    rows[:, i] = v
        rows[:, 1] /= self.err_scale
        return rows

    def likelihood_batch(self, points):
        """-loglikelihood of every point (optimiser coordinates: error rate times err_scale,
        fixed parameters overridden), one launch."""
        if len(points) == 0:
            return np.empty(0)
        self.launches += 1
        self.evaluations += len(points)
        return -self.model.loglikelihood_batch(self._model_rows(points))

    @property
    def likelihood_f(self):
        return _Objective(self)

    def lattice_best(self, axes):
        """See _Objective.lattice_best.  Needs a model whose evaluator is the device context
        (a subclass that overrides loglikelihood_batch is evaluated through `batch` instead)."""
        from .models import BasicModel
        if type(self.model).loglikelihood_batch is not BasicModel.loglikelihood_batch:
            return None
        axes = [np.asarray(a, dtype=np.float64).ravel() for a in axes]
        if any(len(a) == 0 for a in axes):
            return None
        model_axes = [a.copy() for a in axes]
        if self.fix is not None:
            for i, v in enumerate(self.fix):
                if v is not None:
                    model_axes[i] = np.full(len(axes[i]), float(v))
        model_axes[1] = model_axes[1] / self.err_scale
        _, rows = self.model.device_context.lattice_eval(model_axes, want_ll=False, k_best=1)
        self.launches += 1
        self.evaluations += int(np.prod([len(a) for a in axes]))
        if not np.isfinite(rows[0, 0]) and not np.isneginf(rows[0, 0]):
            return None
        # back to optimiser coordinates: the row holds the model-side axis values bit for bit
        point = []
        for a, ma, v in zip(axes, model_axes, rows[0, 1:]):
            hit = np.flatnonzero(ma == v)
            point.append(float(a[hit[0]]) if len(hit) else float(v))
        return -float(rows[0, 0]), tuple(point)

    # -- optimisation -----------------------------------------------------------------------
    def _optimize(self, r, evaluate=None):
        """scipy L-BFGS-B from `r` (covest.py:33-39).  `evaluate(points) -> values` defaults to
        this estimator's own batched objective; multi-start passes a LaunchBatcher's submit."""
        evaluate = evaluate or self.likelihood_batch

        def fun(x):
            return float(evaluate([x])[0])

        def stencil_map(_fun, xs):
            # scipy hands over the perturbed points of one finite-difference gradient
            return [float(v) for v in evaluate(list(xs))]

        options = {}
        if _scipy_has_workers():
            options['workers'] = stencil_map
        return minimize(fun, r, method=constants.OPTIMIZATION_METHOD, bounds=self.bounds,
                        options=options)

    def _optimize_many(self, starts):
        """L-BFGS-B from every start, in threads that share launches."""
        batcher = LaunchBatcher(self.likelihood_batch, len(starts))
        results = [None] * len(starts)
        errors = []

        def work(i):
            try:
                results[i] = self._optimize(starts[i], evaluate=batcher.submit)
            except BaseException as exc:
                errors.append(exc)
            finally:
                batcher.retire()

        threads = [threading.Thread(target=work, args=(i,), daemon=True) for i in range(len(starts))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return results

    def compute_coverage(self, guess, starting_points=1, use_grid_search=False,
                         n_threads=constants.DEFAULT_THREAD_COUNT):
        """-> (parameters, success); flow and tie-breaking as covest.py:41-96."""
        r = list(guess)
        r[1] *= self.err_scale
        success = True
        try:
            verbose_print('Bounds: {}'.format(self.bounds))
            if starting_points == 1:
                with running_time('First optimization'):
                    res = self._optimize(r)
                    success = res.success
                    if not success:
                        verbose_print('Optimization unsuccessful.\n'
                                      'Initial params:{}\nResult{}'.format(r, res))
                    r = res.x
            elif starting_points > 1 and (self.optimizer == 'lockstep' or parallel.world()[1] > 1):
                params = initial_grid(r, count=starting_points, bounds=self.bounds, fix=self.fix)
                params = parallel.broadcast_rows(np.array(params, dtype=np.float64), self._comm_device())
                with running_time('Initial grid optimization'):
                    r, _, success, _ = self.refine_starts(params)
            elif starting_points > 1:
                params = initial_grid(r, count=starting_points, bounds=self.bounds, fix=self.fix)
                with running_time('Initial grid optimization'):
                    best = None
                    for res in self._optimize_many(params):
                        if best is None or best > res.fun:
                            best = res.fun
                            success = res.success
                            if not success:
                                verbose_print('Optimization unsuccessful.\n'
                                              'Initial params:{}\nResult{}'.format(r, res))
                            r = res.x
            if use_grid_search is None and not success:
                use_grid_search = True  # grid search only on failure
            if use_grid_search:
                verbose_print('Starting grid search with guess: {}'.format(r))
                r = list(optimize_grid(self.likelihood_f, r, bounds=self.bounds, fix=self.fix,
                                       n_threads=n_threads))
        except KeyboardInterrupt:
            pass
        verbose_print('Estimation finished with status: %s.' % ('success' if success else 'failure'))
        r = list(r)
        r[1] /= self.err_scale
        return r, success

    # -- multi-start refinement, sharded over the ranks (new) ---------------------------------
    def _comm_device(self):
        """Where the small tensors of the collectives live: the model's GPU under NCCL, the host
        under gloo."""
        rank, world = parallel.world()
        if world > 1:
            import torch.distributed as dist
            if dist.get_backend() == 'nccl':
                import torch
                return torch.device('cuda', self.model.device_context.device)
        return None

    def refine_starts(self, starts, fixed=None):
        """Refine every row of `starts` (optimiser coordinates) and return the best result:
        (x, objective, success, table) with table = one row (objective, success, x...) per start.
        Start i belongs to rank i % W (parallel.split_starts); every rank refines its share -- all
        of them per launch with the lock-step optimiser, or scipy L-BFGS-B in threads -- and the
        refined optima are all-gathered, so every rank returns the same answer.  The reference's
        counterpart is Pool.map(self._optimize, params) and the arg-min over it (covest.py:63-78).
        `fixed`: a boolean mask of coordinates that keep each start's value, on top of the
        estimator's `fix`; the lock-step optimiser then runs whatever `optimizer` says (a profile
        likelihood holds its profiled coordinate this way)."""
        starts = np.asarray(starts, dtype=np.float64).reshape(-1, self.model.param_count)
        rank, world = parallel.world()
        mine = parallel.split_starts(starts, rank, world)
        n = self.model.param_count
        per_rank = (len(starts) + world - 1) // world
        table = np.full((per_rank, 2 + n), np.nan)
        table[:, 0] = np.inf
        table[:, 1] = 0.0
        if len(mine):
            if self.optimizer == 'lockstep' or fixed is not None:
                held = [self.fix is not None and self.fix[i] is not None for i in range(n)]
                if fixed is not None:
                    held = [bool(h or f) for h, f in zip(held, fixed)]
                results, launches = lockstep_minimize(self.likelihood_batch, mine, self.bounds, fixed=held)
            else:
                results = self._optimize_many([list(s) for s in mine])
            for j, res in enumerate(results):
                table[j, 0] = res.fun if np.isfinite(res.fun) else np.inf
                table[j, 1] = 1.0 if res.success else 0.0
                table[j, 2:] = res.x
        if world > 1:
            gathered = parallel.allgather_rows(parallel.to_comm(table, self._comm_device()))
            table = gathered.cpu().numpy().reshape(world, per_rank, 2 + n)
            table = table.transpose(1, 0, 2).reshape(-1, 2 + n)[:len(starts)]  # back to start order
        else:
            table = table[:len(starts)]
        best = int(np.argmin(table[:, 0]))  # ties: the earliest start, as the reference's strict `>`
        return table[best, 2:].copy(), float(table[best, 0]), bool(table[best, 1]), table

    def compute_coverage_from_lattice(self, axes, k_best=64):
        """SURVEY.md section 8(e): evaluate the candidate lattice of `axes` (model coordinates)
        sharded over the ranks, all-gather every rank's k_best best rows, refine the global best
        rows as starts (dealt round-robin), all-gather the refined optima.
        Returns (parameters, success, rows) like compute_coverage plus the global best rows."""
        rows = lattice_search(self.model, axes, k_best=k_best)
        keep = np.isfinite(rows[:, 0])
        starts = rows[keep, 1:].copy()
        if len(starts) == 0:
            raise ValueError('no lattice point has a finite log-likelihood')
        starts[:, 1] *= self.err_scale
        x, fun, success, _ = self.refine_starts(starts)
        x = list(x)
        x[1] /= self.err_scale
        return x, success, rows

    # -- polish (new) -----------------------------------------------------------------------
    def polish(self, x, iterations=40, rel_step=1e-4, tol=1e-11):
        """Projected Newton iteration on central differences (step rel_step * |x_i|): the
        optimum L-BFGS-B's 1e-8 forward differences can only approach to ~1e-4 relative
        (SURVEY.md section 7.3 item 3).  Every iteration's 2n^2 + 1 stencil points are one
        launch.  `x` is in optimiser coordinates (error rate times err_scale).
        Returns (x, objective)."""
        x = np.array([float(v) for v in x], dtype=np.float64)
        n = len(x)
        lo = np.array([-np.inf if b[0] is None else b[0] for b in self.bounds], dtype=np.float64)
        hi = np.array([np.inf if b[1] is None else b[1] for b in self.bounds], dtype=np.float64)
        fixed = np.array([self.fix is not None and self.fix[i] is not None for i in range(n)])
        fx = None
        for _ in range(iterations):
            h = rel_step * np.maximum(np.abs(x), 1e-3)
            at_lo = (x - h < lo)
            at_hi = (x + h > hi)
            free = ~(fixed | at_lo | at_hi)
            idx = np.flatnonzero(free)
            if len(idx) == 0:
                break
            fx, g, H = self._central_differences(x, idx, h)
            if not np.all(np.isfinite(g)) or not np.all(np.isfinite(H)):
                break
            try:
                step = np.linalg.solve(H, -g)
            except np.linalg.LinAlgError:
                break
            if g @ step > 0:  # not a descent direction: the Hessian is not positive definite here
                step = -g * (h[idx] ** 2)
            new = x.copy()
            new[idx] = np.minimum(np.maximum(x[idx] + step, lo[idx]), hi[idx])
            moved = np.max(np.abs(new - x) / np.maximum(np.abs(x), 1e-300))
            x = new
            if moved < tol:
                break
        fx = float(self.likelihood_batch([x])[0])
        return x, fx

    def _central_differences(self, x, idx, h):
        """(objective, gradient, Hessian) at `x` over the coordinates `idx`, steps h[i]: the 2m^2 + 1
        points of the central-difference stencil in one launch."""
        pts = [x.copy()]
        for i in idx:
            for s in (1, -1):
                p = x.copy()
                p[i] += s * h[i]
                pts.append(p)
        pairs = [(a, b) for ai, a in enumerate(idx) for b in idx[ai + 1:]]
        for a, b in pairs:
            for sa, sb in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                p = x.copy()
                p[a] += sa * h[a]
                p[b] += sb * h[b]
                pts.append(p)
        vals = np.asarray(self.likelihood_batch(pts), dtype=np.float64)
        fx = vals[0]
        m = len(idx)
        g = np.empty(m)
        H = np.empty((m, m))
        for t, i in enumerate(idx):
            fp, fm = vals[1 + 2 * t], vals[2 + 2 * t]
            g[t] = (fp - fm) / (2 * h[i])
            H[t, t] = (fp - 2 * fx + fm) / (h[i] * h[i])
        base = 1 + 2 * m
        pos = {int(i): t for t, i in enumerate(idx)}
        for q, (a, b) in enumerate(pairs):
            fpp, fpm, fmp, fmm = vals[base + 4 * q: base + 4 * q + 4]
            v = (fpp - fpm - fmp + fmm) / (4 * h[a] * h[b])
            H[pos[int(a)], pos[int(b)]] = H[pos[int(b)], pos[int(a)]] = v
        return fx, g, H

    # -- profile likelihoods and likelihood-ratio intervals (new) ---------------------------------
    def _param_index(self, param):
        return self.model.params.index(param) if isinstance(param, str) else int(param)

    def _held(self):
        n = self.model.param_count
        return np.array([self.fix is not None and self.fix[i] is not None for i in range(n)], dtype=bool)

    def _lattice_profile(self, model_axes, keep_mask):
        """Profile rows of a lattice in model coordinates (grid.lattice_profile: on the device, sharded
        over the ranks)."""
        return lattice_profile(self.model, model_axes, keep_mask)

    def _refine_profile(self, p, values, starts):
        """Refine every start with coordinate p held at values[j] (and the estimator's `fix`), all
        starts per launch: (objective, x, success) arrays."""
        starts = np.array(starts, dtype=np.float64).reshape(len(values), self.model.param_count)
        starts[:, p] = values
        fixed = np.zeros(self.model.param_count, dtype=bool)
        fixed[p] = True
        table = self.refine_starts(starts, fixed=fixed)[3]
        return table[:, 0].copy(), table[:, 2:].copy(), table[:, 1] > 0

    def profile(self, param, values, nuisance_axes, x_hat):
        """The profile of -loglikelihood over parameter `param` (index or name) at `values`, in
        optimiser coordinates (error rate times err_scale, as compute_coverage_from_lattice): for
        each value the minimum over the other free parameters.  One lattice -- the profiled axis =
        `values`, axis j = nuisance_axes[j], or x_hat[j] where that is None; a fixed parameter takes
        its fixed value -- whose best point per value is taken on the device (grid.lattice_profile),
        then every finite row refined as a start with the profiled coordinate held, all starts per
        launch (lockstep_minimize).  A refined value is never worse than its lattice row.  Returns a
        Profile (values, fun, x, success, lattice_fun)."""
        n = self.model.param_count
        p = self._param_index(param)
        values = np.asarray(values, dtype=np.float64).ravel()
        x_hat = np.asarray(x_hat, dtype=np.float64).ravel()
        held = self._held()
        axes = []
        for i in range(n):
            if i == p:
                axes.append(values)
            elif held[i] or nuisance_axes[i] is None:
                axes.append(np.array([x_hat[i]]))
            else:
                axes.append(np.asarray(nuisance_axes[i], dtype=np.float64).ravel())
        model_axes = [a.copy() for a in axes]
        for i in range(n):
            if held[i]:
                model_axes[i] = np.full(len(axes[i]), float(self.fix[i]))
        model_axes[1] = model_axes[1] / self.err_scale  # as _model_rows: the lattice holds its points bit for bit
        rows = np.asarray(self._lattice_profile(model_axes, 1 << p), dtype=np.float64)
        self.launches += 1
        self.evaluations += int(np.prod([len(a) for a in axes]))
        lattice_fun = np.where(np.isnan(rows[:, 0]), np.inf, -rows[:, 0])
        # back to optimiser coordinates: the rows hold the model-side axis values bit for bit
        starts = np.empty((len(values), n))
        for i in range(n):
            for j, v in enumerate(rows[:, 1 + i]):
                hit = np.flatnonzero(model_axes[i] == v)
                starts[j, i] = axes[i][hit[0]] if len(hit) else v
        starts[:, p] = values
        fun = lattice_fun.copy()
        x = np.full((len(values), n), np.nan)
        success = np.zeros(len(values), dtype=bool)
        live = np.flatnonzero(np.isfinite(lattice_fun))
        if len(live):
            f, xs, ok = self._refine_profile(p, values[live], starts[live])
            better = f <= lattice_fun[live]  # the flat end game of lockstep_minimize may take a step of no gain
            fun[live] = np.where(better, f, lattice_fun[live])
            x[live] = np.where(better[:, None], xs, starts[live])
            success[live] = ok
        return Profile(values, fun, x, success, lattice_fun)

    def _standard_errors(self, x, free):
        """sqrt(diag(H^-1)) of the central-difference Hessian of the objective at x over the free
        coordinates that are not within a stencil step of a bound (one launch, as polish); 1 % of
        max(|x_i|, 1e-3) where that does not exist (H not positive definite, a coordinate at a bound)."""
        lo =np.array([-np.inf if b[0] is None else b[0] for b in self.bounds], dtype=np.float64)
        hi = np.array([np.inf if b[1] is None else b[1] for b in self.bounds], dtype=np.float64)
        h = 1e-4 * np.maximum(np.abs(x), 1e-3)
        se = 0.01 * np.maximum(np.abs(x), 1e-3)
        idx = np.array([i for i in free if x[i] - h[i] >= lo[i] and x[i] + h[i] <= hi[i]], dtype=np.int64)
        if len(idx):
            _, _, H = self._central_differences(x.copy(), idx, h)
            if np.all(np.isfinite(H)):
                try:
                    np.linalg.cholesky(H)
                    d = np.diag(np.linalg.inv(H))
                    ok = np.isfinite(d) & (d > 0)
                    se[idx[ok]] = np.sqrt(d[ok])
                except np.linalg.LinAlgError:
                    pass
        return se

    def likelihood_intervals(self, x_hat, level=0.95, params=None):
        """Likelihood-ratio intervals: for each free parameter (or those named in `params`) the
        connected range around x_hat where the profile log-likelihood stays within chi2_1(level) / 2
        of the maximum.  x_hat in optimiser coordinates (error rate times err_scale); the intervals
        come back in model coordinates, as compute_coverage returns its estimate.

          scale      standard errors from the central-difference Hessian at x_hat (_standard_errors)
          coarse     33 profile values over x_hat +- 4 se (clipped to the bounds), nuisance axes of 12
                     values over +- 4 se (64 for the basic model's one), one lattice each (profile);
                     a side where the threshold is not crossed doubles its span, at most three times
          endpoints  17 values inside each bracket of a crossing, refined from the nearer coarse
                     optimum; the endpoint interpolates the crossing linearly there
          flags      at_bound: a side reached a bound without crossing; open: a side crossed neither
                     within the widest span nor at a bound (the end is the last value profiled);
                     disjoint: a coarse profile value outside the interval is above the threshold;
                     moved: the profile beat the log-likelihood of x_hat (x_hat is not the optimum)

        Returns {name: Interval}."""
        from scipy.stats import chi2
        if not 0.0 < float(level) < 1.0:
            raise ValueError('level must lie in (0, 1), not %r' % (level,))
        n = self.model.param_count
        x_hat = np.array([float(v) for v in x_hat], dtype=np.float64)
        held = self._held()
        free = [i for i in range(n) if not held[i]]
        want = free if params is None else [self._param_index(q) for q in params]
        for p in want:
            if held[p]:
                raise ValueError('%s is fixed: it has no interval' % self.model.params[p])
        lo = np.array([-np.inf if b[0] is None else b[0] for b in self.bounds], dtype=np.float64)
        hi = np.array([np.inf if b[1] is None else b[1] for b in self.bounds], dtype=np.float64)
        half = float(chi2.ppf(level, 1)) / 2
        se = self._standard_errors(x_hat, free)
        ll_hat = -float(self.likelihood_batch([x_hat])[0])
        out = {}
        for p in want:
            out[self.model.params[p]] = self._interval(p, x_hat, se, free, half, ll_hat, lo, hi, level)
        return out

    def nuisance_axes(self, p, x_hat, se, free):
        """The lattice axes of the parameters profiled out of parameter p (profile's nuisance_axes):
        x_hat +- 4 se over 12 values (64 for the basic model's one), clipped to the bounds."""
        n = self.model.param_count
        n_nuis = 64 if n == 2 else 12
        nuisance = [None] * n
        for j in free:
            if j != p:
                lo, hi = self.bounds[j]
                lo, hi = -np.inf if lo is None else lo, np.inf if hi is None else hi
                nuisance[j] = np.unique(np.clip(np.linspace(x_hat[j] - 4 * se[j], x_hat[j] + 4 * se[j], n_nuis),
                                                lo, hi))
        return nuisance

    def _interval(self, p, x_hat, se, free, half, ll_hat, lo, hi, level):
        nuisance = self.nuisance_axes(p, x_hat, se, free)
        width = [4 * se[p], 4 * se[p]]  # below, above x_hat
        for doubling in range(4):
            a, b = max(x_hat[p] - width[0], lo[p]), min(x_hat[p] + width[1], hi[p])
            values = np.unique(np.clip(np.linspace(a, b, 33), lo[p], hi[p]))
            prof = self.profile(p, values, nuisance, x_hat)
            pll = np.where(np.isfinite(prof.fun), -prof.fun, -np.inf)
            top = max(ll_hat, float(np.max(pll)))
            thr = top - half
            c = int(np.argmin(np.abs(values - x_hat[p])))
            if pll[c] < thr:  # x_hat itself is outside: the region around the best value
                c = int(np.argmax(pll))
            left, right = c, c
            while left > 0 and pll[left - 1] >= thr:
                left -= 1
            while right < len(values) - 1 and pll[right + 1] >= thr:
                right += 1
            short = [left == 0 and values[0] > lo[p], right == len(values) - 1 and values[-1] < hi[p]]
            if not any(short) or doubling == 3:
                break
            width = [w * 2 if s else w for w, s in zip(width, short)]
        moved = bool(np.max(pll) > ll_hat + 1e-9 * max(1.0, abs(ll_hat)))
        ends = [values[left], values[right]]
        at_bound = [left == 0 and values[0] <= lo[p], right == len(values) - 1 and values[-1] >= hi[p]]
        open_side = [left == 0 and not at_bound[0], right == len(values) - 1 and not at_bound[1]]
        # endpoints: 17 values inside each bracket, warm-started from the nearer coarse optimum
        brackets = []
        if left > 0:
            brackets.append((0, left, left - 1))
        if right < len(values) - 1:
            brackets.append((1, right, right + 1))
        if brackets:
            inner, starts = [], []
            for _, i_in, i_out in brackets:
                v = np.linspace(values[i_in], values[i_out], 19)[1:-1]
                inner.append(v)
                near_in = np.abs(v - values[i_in]) <= np.abs(v - values[i_out])
                xs_in = np.where(np.isfinite(prof.x[i_in]), prof.x[i_in], x_hat)
                xs_out = np.where(np.isfinite(prof.x[i_out]), prof.x[i_out], xs_in)
                starts.append(np.where(near_in[:, None], xs_in[None, :], xs_out[None, :]))
            f, _, _ = self._refine_profile(p, np.concatenate(inner), np.concatenate(starts))
            f = np.where(np.isfinite(f), -f, -np.inf)
            at = 0
            for (side, i_in, i_out), v in zip(brackets, inner):
                vs = np.concatenate(([values[i_in]], v, [values[i_out]]))
                fs = np.concatenate(([pll[i_in]], f[at:at + len(v)], [pll[i_out]]))
                at += len(v)
                k = 0
                while fs[k + 1] >= thr:  # the last value is below the threshold
                    k += 1
                if np.isfinite(fs[k + 1]):
                    ends[side] = vs[k] + (thr - fs[k]) * (vs[k + 1] - vs[k]) / (fs[k + 1] - fs[k])
                else:
                    ends[side] = vs[k]
        disjoint = bool(np.any(pll[:left] >= thr) or np.any(pll[right + 1:] >= thr))
        scale = self.err_scale if p == 1 else 1.0
        return Interval(self.model.params[p], float(ends[0]) / scale, float(ends[1]) / scale, level,
                        {'at_bound': any(at_bound), 'open': any(open_side), 'disjoint': disjoint, 'moved': moved},
                        thr, values / scale, pll)


class Profile:
    """CoverageEstimator.profile: per profiled value (optimiser coordinates) the refined objective
    (-loglikelihood; inf where the lattice had no finite point), its point, whether the refinement
    converged, and the objective of the lattice row it started from."""

    def __init__(self, values, fun, x, success, lattice_fun):
        self.values, self.fun, self.x, self.success, self.lattice_fun = values, fun, x, success, lattice_fun


class Interval:
    """A likelihood-ratio interval [lo, hi] of one parameter (model coordinates) at `level`, its flags,
    the profile log-likelihood threshold, and the coarse profile (values, log-likelihoods) it rests on."""

    def __init__(self, param, lo, hi, level, flags, threshold, values, profile):
        self.param, self.lo, self.hi, self.level, self.flags = param, lo, hi, level, flags
        self.threshold, self.values, self.profile = threshold, values, profile

    def __repr__(self):
        return 'Interval(%s, [%r, %r], %s)' % (self.param, self.lo, self.hi,
                                               [k for k, v in self.flags.items() if v])


def candidate_lattice(model, guess, bounds, shape=None):
    """Axes of a candidate lattice over the box initial_grid draws from (covest/grid.py:95-110: every
    coordinate in [v / 3, 3 v] cut to the bounds): coverage and error rate log-spaced around the guess,
    the copy-number parameters over their whole ranges.  Model coordinates."""
    n = model.param_count
    shape = shape or ((24, 16, 8, 8, 8) if n == 5 else (64, 48))
    axes = []
    for i in range(n):
        lo, hi = bounds[i]
        v = float(guess[i])
        if i < 2:
            a, b = v / constants.INITIAL_GRID_STEP, v * constants.INITIAL_GRID_STEP
            a = max(a, lo if lo is not None else a, 1e-12)
            b = min(b, hi) if hi is not None else b
            axes.append(np.geomspace(a, max(b, a), shape[i]))
        else:
            axes.append(np.linspace(lo if lo is not None else 0.0, hi if hi is not None else 1.0, shape[i]))
    return axes


def _scipy_has_workers():
    import scipy
    major, minor = (int(v) for v in scipy.__version__.split('.')[:2])
    return (major, minor) >= (1, 16)


@running_time_decorator
def main(args):
    if args.load:  # a previous report: nothing is estimated (covest.py:102-105)
        with open(args.load) as f:
            parsed_data = parse_data(f)
            args.sample_factor = parsed_data.sample_factor
    verbose_print('Loading histogram {} with parameters k={} r={}.'.format(
        args.input_histogram, args.kmer_size, args.read_length))
    hist_orig, meta = load_histogram(args.input_histogram)
    hist, tail, sample_factor, guess_c, guess_e = process_histogram(
        hist_orig, args.kmer_size, args.read_length, trim=args.trim,
        sample_factor=args.sample_factor)

    orig_sample_factor = 1
    if 'sample_factor' in meta:
        try:
            orig_sample_factor = int(meta['sample_factor'])
        except ValueError as exc:
            print(exc)
    if sample_factor > 1:
        fname = '%s.covest.sampled_x%d.hist' % (Path(args.input_histogram).stem, sample_factor)
        save_histogram(hist, fname, {'tool': version_string,
                                     'sample_factor': sample_factor * orig_sample_factor})
    err_scale = args.error_scale
    if sample_factor is None:
        sample_factor = 1
    if args.coverage:
        args.coverage /= sample_factor

    model = select_model(args.model)(
        args.kmer_size, args.read_length, hist, tail, max_error=constants.MAX_ERRORS,
        max_cov=args.max_coverage, min_single_copy_ratio=args.min_q1)

    orig = [None] * model.param_count
    for i, v in zip(range(model.param_count), (args.coverage, args.error_rate) + tuple(args.params)):
        orig[i] = v
    fix = orig if args.fix else None

    if args.ll_only:
        print('Loglikelihood:', model.compute_loglikelihood(*orig))
        return
    if args.load:
        guess = parsed_data.guess
        res = parsed_data.estimated
    else:
        verbose_print('Estimating coverage...')
        if args.start_original:
            guess = list(orig)
        else:
            guess = list(model.defaults)
            if not (guess_c == 0 and guess_e == 1):  # the moment guess worked
                guess[:2] = guess_c, guess_e
            if fix:
                for i, v in enumerate(fix):
                    if v is not None:
                        guess[i] = v
        guess_ll = model.compute_loglikelihood(*guess)
        if guess_ll == -constants.INF:
            verbose_print('Unable to compute likelihood. '
                          'Please, try to trim the histogram, or use more complex model')
            raise SystemExit(1)
        verbose_print('Initial guess: {} ll:{}'.format(guess, guess_ll))

        estimator = CoverageEstimator(model, err_scale=err_scale, fix=fix,
                                      optimizer=getattr(args, 'optimizer', None))
        if getattr(args, 'lattice_starts', 0) and not fix:
            # starts = the best rows of a candidate lattice (sharded over the ranks under torchrun)
            # instead of random draws; refined with all starts per launch
            estimator.optimizer = 'lockstep'
            res, success, _ = estimator.compute_coverage_from_lattice(
                candidate_lattice(model, guess, model.bounds), k_best=args.lattice_starts)
        else:
            res, success = estimator.compute_coverage(
                guess, starting_points=args.starting_points, use_grid_search=args.grid,
                n_threads=args.thread_count)
        if getattr(args, 'polish', False):
            scaled = list(res)
            scaled[1] *= err_scale
            polished, _ = estimator.polish(scaled)
            res = list(polished)
            res[1] /= err_scale
        extra = None
        if getattr(args, 'ci', None) is not None:
            scaled = list(res)
            scaled[1] *= err_scale
            with running_time('Likelihood-ratio intervals'):
                intervals = estimator.likelihood_intervals(scaled, level=args.ci)
            extra = interval_report(hist_orig, model, sample_factor, intervals, args.ci)
        verbose_print('Device launches: {}, evaluations: {}'.format(
            estimator.launches, estimator.evaluations))
        print_output(hist_orig, model, success, sample_factor, res, guess, orig,
                     reads_size=args.reads_size, orig_sample_factor=orig_sample_factor,
                     starting_points=args.starting_points, use_grid_search=args.grid, extra=extra)
    if args.plot is not None:
        model.plot_probs(res, guess, orig, cumulative=args.plot, log_scale=constants.PLOT_LOG_SCALE)


def build_parser():
    p = argparse.ArgumentParser(
        description='Estimate coverage, error rate and genome size from a k-mer abundance '
                    'histogram (CovEst interface, likelihood on NVIDIA B200)')
    p.add_argument('input_histogram', type=str, help='Input histogram')
    p.add_argument('-v', '--version', action='version', version=version_string,
                   help='Print version and exit.')
    p.add_argument('-m', '--model', type=str, default='basic',
                   help='Select models for estimation. Options: {}'.format(list(models.keys())))
    p.add_argument('-k', '--kmer-size', type=int, default=constants.DEFAULT_K, help='Kmer size')
    p.add_argument('-r', '--read-length', type=int, default=constants.DEFAULT_READ_LENGTH,
                   help='Read length')
    p.add_argument('-rs', '--reads-size', type=int, help='Calculate genome size from reads size')
    p.add_argument('-sp', '--starting-points', type=int, default=1,
                   help='Number of point to start optimization from.')
    p.add_argument('-T', '--thread-count', default=constants.DEFAULT_THREAD_COUNT, type=int,
                   help='Thread count (accepted for compatibility; evaluation is batched on the GPU)')
    p.add_argument('--plot', type=bool, nargs='?', const=False,
                   help='Plot probabilities (use --plot 1 to plot "probs * j")')
    p.add_argument('--load', type=str, help='Load covest output file')
    p.add_argument('-t', '--trim', type=int, default=None,
                   help='Trim histogram at this value. Set to 0 to disable automatic trimming.')
    p.add_argument('-sf', '--sample-factor', type=int, default=None,
                   help='Use fixed sample factor for histogram sampling instead of automatic.'
                        ' Set to 1 to not sample at all.')
    p.add_argument('-g', '--grid', action='store_true', default=False,
                   help='Use grid search for fine-tuning.')
    p.add_argument('-f', '--fix', action='store_true', help='Fix some params, optimize others')
    p.add_argument('-c', '--coverage', type=float, help='Coverage')
    p.add_argument('-M', '--max-coverage', type=int, help='Upper coverage limit')
    p.add_argument('-e', '--error-rate', type=float, help='Error rate')
    p.add_argument('-es', '--error-scale', type=float, default=constants.DEFAULT_ERR_SCALE,
                   help='Error scale')
    p.add_argument('-mq1', '--min-q1', type=float, default=constants.DEFAULT_MIN_SINGLECOPY_RATIO,
                   help='minimum single copy ratio')
    p.add_argument('-p', '--params', type=nonefloat, nargs='*', default=tuple(),
                   help='Additional model parameters.')
    p.add_argument('-ll', '--ll-only', action='store_true',
                   help='Only compute log likelihood from provided values')
    p.add_argument('-so', '--start-original', action='store_true',
                   help='Start optimization form provided values')
    # additions (not in the reference)
    p.add_argument('--polish', action='store_true',
                   help='Newton-polish the optimum on central differences after L-BFGS-B')
    p.add_argument('--optimizer', choices=['scipy', 'lockstep'], default=None,
                   help='Multi-start refinement: scipy L-BFGS-B per start (the reference\'s optimiser, '
                        'default) or the lock-step Newton iteration with all starts per launch')
    p.add_argument('--lattice-starts', type=int, default=0, metavar='K',
                   help='Refine from the K best points of a candidate lattice over the initial-grid box '
                        '(evaluated on the device, sharded over the GPUs under torchrun) instead of -sp random starts')
    p.add_argument('--seed', type=int, default=None,
                   help='Seed Python\'s random (multi-start points, histogram sampling)')
    p.add_argument('--ci', type=float, default=None, metavar='LEVEL',
                   help='Add likelihood-ratio intervals at LEVEL (in (0, 1), e.g. 0.95) for every free parameter '
                        'and the genome size to the report, from profile likelihoods on the device. The intervals '
                        'rest on the estimate: use --polish, or the flag "moved" may report an L-BFGS-B optimum '
                        'short of the maximum')
    return p


def check_args(parser, args):
    """Combinations argparse cannot check on its own (parser.error exits)."""
    if args.ci is not None:
        if not 0.0 < args.ci < 1.0:
            parser.error('--ci LEVEL must lie in (0, 1), not %r' % args.ci)
        if args.load:
            parser.error('--ci needs an estimate: it cannot be combined with --load')
        if args.ll_only:
            parser.error('--ci needs an estimate: it cannot be combined with --ll-only')


def run(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    check_args(parser, args)
    if args.seed is not None:
        import random
        random.seed(args.seed)
    main(args)


if __name__ == '__main__':
    run()
