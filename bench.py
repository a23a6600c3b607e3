#!/usr/bin/env python
"""bench.py -- throughput of the batched log-likelihood path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg3|cfg5]

Metric (BASELINE.json): log-likelihood evaluations per second counted as parameter point x
histogram bin.  A step is one pass of the hot path over one batch of candidate points: every rank
evaluates its slice of the candidate lattice (points resident in HBM), keeps its 64 best rows on
the device and -- for N > 1 -- all-gathers them (NCCL) so that every rank holds the global best
rows.  Weak scaling: the lattice is refined with N so that every rank always evaluates the same
number of points.

  value      the rank's slice of the lattice handed over as its axes (cvb_lattice_eval: what
             grid.py's callers hand over), values and best rows left in HBM, CUDA-event timed, max
             over ranks.  `explicit_points`: the same batch as an explicit point array resident in
             HBM (cvb_loglik_batch + cvb_topk: the general plan with its sort).  `random_points`:
             seeded uniform-random points of the initial_grid box (no two share coverage and error
             rate: the per-point kernel).  `sustained`: steps back to back for >= 2 s.
  e2e        the same call with HOST buffers: the axes go in, all values (8 B per point) and the
             best rows come back to host memory inside the timed region.  `e2e_points`: the batch
             as an explicit host array (40 B per point in; pinned and pageable).
  roofline   FP64 pipe, dominant kernel (cvf_prefix_kernel: running sums over the copy numbers per
             q-run, three-term combination and log-likelihood epilogue per point; with
             --path gemm cvf_gemm_kernel: copy weights x bin profiles on the FP64 tensor cores): its
             algorithmic flop per launch / its CUDA-event duration / the DFMA peak measured in this
             run (MEASURED_PEAKS.json has no FP64 figure; DESIGN.md section 6).  `phases` breaks the
             whole evaluation down.
  cpu_baseline / --impl reference: the reference's own C module (oracle/_ref) driven by a Python
             restatement of models.py with a fork pool over all host cores, on a bounded sample.

--dump-outputs DIR writes what the last timed step of the headline leg handed back (rank 0) as
DIR/loglik.npy and DIR/best_rows.npy (float64, every value finite: DIR/<name>_nonfinite.npy marks
the entries that were -inf, +inf or NaN).  The workload histogram is drawn from the CPU oracle's
p_j, so the inputs are the same for every build and two builds compare output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_BEST = 64
METRIC = 'loglik_point_bin_evals_per_sec'
UNIT = 'point*bin/s'
POINTS_PER_RANK = {'cfg3': 1000000, 'cfg4': 100000, 'cfg5': 12500000}
DUMP_MAX_VALUES = 4 << 20  # 32 MiB of float64: a dump stays under 64 MB on every workload


def workload_axes(name, world):
    """cfg3: 40 x 25 x 10 x 10 x 10 = 1e6 points (SURVEY.md section 8(d)); with N ranks the
    coverage axis is refined N-fold (weak scaling).  cfg5: 1e8 points over 8 ranks."""
    from covest_b200 import workload
    theta = workload.CONFIGS[name]['theta']
    if name == 'cfg3':
        return workload.lattice_axes(theta, n_c=40 * world, n_e=25)
    if name == 'cfg4':  # k = 31, r = 150, 5000 bins, coverage 200: 10^5 points per rank
        return workload.lattice_axes(theta, n_c=10 * world, n_e=10)
    return workload.lattice_axes(theta, n_c=25 * world, n_e=50, n_q1=10, n_q2=10, n_q=100)


class ClockSampler:
    """SM clock and throttle reasons of one GPU while the timed region runs: NVML every 5 ms
    (pynvml), or nvidia-smi every 200 ms when NVML cannot be loaded."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.index = index
        self.sm, self.mx, self.reasons = [], [], set()
        self.source = None
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        try:
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
            bits = {'hw_slowdown': getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8),
                    'hw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
                    'sw_thermal_slowdown': getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20),
                    'sw_power_cap': getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4)}
            get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.source = 'nvml'
            while not self._stop.is_set():
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(h))
                for name, bit in bits.items():
                    if mask & bit:
                        self.reasons.add(name)
                self._stop.wait(0.005)
        finally:
            nv.nvmlShutdown()

    def _run_smi(self):
        self.source = 'nvidia-smi'
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True,
                                     text=True, timeout=5).stdout.strip()
                r = [x.strip() for x in out.split(',')] if out else []
                if r and r[0].replace('.', '').isdigit():
                    self.sm.append(float(r[0]))
                if len(r) > 1 and r[1].replace('.', '').isdigit():
                    self.mx.append(float(r[1]))
                for i, name in enumerate(self.NAMES):
                    if len(r) > 3 + i and r[3 + i].lower().startswith('active'):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.2)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            if not self.sm:
                self._run_smi()

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        return {'sm_mhz': float(np.median(self.sm)) if self.sm else None,
                'sm_max_mhz': max(self.mx) if self.mx else None,
                'reasons': [n for n in self.NAMES if n in self.reasons], 'samples': len(self.sm),
                'source': self.source}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ---------------------------------------------------------------------------------------------
def cpu_sample_points(axes, n, seed=4242):  # noqa: D103
    from covest_b200 import workload
    total = int(np.prod([len(a) for a in axes]))
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.choice(total, size=n, replace=False))
    return np.vstack([workload.lattice_points(axes, first=int(i), count=1) for i in idx])


class CpuReference:
    """The reference's CPU path on the host cores: its own C module (oracle/_ref) driven by a
    restatement of models.py over a fork pool of all cores (the reference's parallelism,
    models.py:109-117) -- or the C port of the oracle when the module is not built.  The pool is
    created once, outside every timed region, and each timing maps a few hundred seeded lattice
    points over it (dynamic scheduling: the points differ 100x in cost)."""

    def __init__(self, hist, cfg, axes, cores):
        from oracle import covest_oracle as orc
        self.orc = orc
        self.kind = 'reference' if orc.ref_module() is not None else 'port'
        self.detail = ('reference C module (c_src/covest_poissonmodule.c compiled into oracle/_ref) driven by a '
                       'restatement of models.py:81-107, :211-242 (pinned bit for bit to the reference package)'
                       if self.kind == 'reference' else 'C port of the oracle, one truncated_poisson per term')
        self.model = orc.Model(cfg['model'], cfg['k'], cfg['r'], hist, 0, max_error=8)
        self.axes, self.cores, self.bins = axes, cores, len(hist)
        self.pool = orc.ref_pool(cores) if self.kind == 'reference' and cores > 1 else None
        if self.pool is not None:
            self.pool.map(abs, range(4 * cores))  # the workers exist before anything is timed

    def rate(self, n_points, seed=4242):
        """-> (point*bin/s, seconds) for n_points seeded lattice points."""
        pts = cpu_sample_points(self.axes, n_points, seed)
        t0 = time.perf_counter()
        if self.kind == 'reference':
            self.orc.ref_loglik_batch(self.model, pts, processes=self.cores, pool=self.pool)
        else:
            self.model.loglik_batch(pts, mode=self.orc.FAITHFUL, threads=self.cores)
        dt = time.perf_counter() - t0
        return n_points * self.bins / dt, dt

    def sized_rate(self, target_s=10.0, seed=4242):
        """A sample sized for about target_s seconds (>= 64 points): a probe sets the size."""
        n0 = max(64, 4 * self.cores)
        rate, dt = self.rate(n0, seed)
        if dt >= 0.8 * target_s:
            return rate, dt, n0
        n = int(min(4096, max(n0, n0 * target_s / max(dt, 1e-3))))
        rate, dt = self.rate(n, seed + 1)
        return rate, dt, n

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
            self.pool = None


def covest_end_to_end(cores):
    """Wall time of the estimator flow (process_histogram -> model -> CoverageEstimator, the body of
    `covest cfg2.hist -m repeat -k 21 -r 100 -sf 1`) on the synthetic cfg2 histogram: on the device,
    and with the likelihood routed to the reference's own C module over a fork pool of all host
    cores (the same batches, so both arms follow the same optimiser path)."""
    from covest_b200 import constants
    from covest_b200.covest import CoverageEstimator
    from covest_b200.histogram import process_histogram
    from covest_b200.models import RepeatsModel
    from oracle import covest_oracle as orc
    constants.VERBOSE = False
    with open(os.path.join(ROOT, 'tests', 'golden', 'e2e_golden.json')) as f:
        g = json.load(f)['cfg2_repeats']
    hist = {int(j): int(h) for j, h in g['hist']}

    def flow(cls):
        t0 = time.perf_counter()
        h2, tail, sf, gc, ge = process_histogram(hist, g['k'], g['r'], sample_factor=1)
        model = cls(g['k'], g['r'], h2, tail, max_error=8)
        guess = list(model.defaults)
        guess[:2] = gc, ge
        est = CoverageEstimator(model)
        x, ok = est.compute_coverage(guess)
        return time.perf_counter() - t0, [float(v) for v in x], est.evaluations

    class CpuRepeats(RepeatsModel):  # likelihood on the host cores, everything else unchanged
        def loglikelihood_batch(self, points):
            m = orc.Model('repeats', self.k, self.r, self.hist, self.tail, max_error=self.max_error)
            pts = np.asarray(points, dtype=np.float64).reshape(-1, self.param_count)
            if orc.ref_module() is not None:
                return orc.ref_loglik_batch(m, pts, processes=min(cores, len(pts)))
            return m.loglik_batch(pts, mode=orc.FAITHFUL, threads=cores)

    def flow_device(optimizer='scipy', **kw):  # the reference's experiment invocations (tools/run_covest.py: -sp 16; -g)
        import random
        random.seed(7)
        t0 = time.perf_counter()
        h2, tail, sf, gc, ge = process_histogram(hist, g['k'], g['r'], sample_factor=1)
        model = RepeatsModel(g['k'], g['r'], h2, tail, max_error=8)
        guess = list(model.defaults)
        guess[:2] = gc, ge
        est = CoverageEstimator(model, optimizer=optimizer)
        x, ok = est.compute_coverage(guess, **kw)
        wall = time.perf_counter() - t0
        xs = list(x)
        polished, fpol = est.polish(xs)
        return {'seconds': wall, 'coverage': float(x[0]), 'evaluations': est.evaluations, 'launches': est.launches,
                'objective': float(est.likelihood_f(xs)), 'polished_coverage': float(polished[0]),
                'polished_objective': float(fpol)}

    flow(RepeatsModel)  # warm-up: context creation, first launches
    runs = [flow(RepeatsModel) for _ in range(5)]  # a ~10 ms flow right after seconds of host-only work: the median of five
    dev_s, dev_x, dev_n = sorted(runs, key=lambda r: r[0])[2]
    cpu_s, cpu_x, cpu_n = flow(CpuRepeats)
    extra = {}
    try:
        flow_device(optimizer='lockstep', starting_points=16)  # warm-up of the batch shapes
        def median3(**kw):  # flows of tens of ms: the median of three
            return sorted((flow_device(**kw) for _ in range(3)), key=lambda r: r['seconds'])[1]
        extra = {'device_multi_start_16': median3(starting_points=16),
                 'device_multi_start_16_lockstep': median3(optimizer='lockstep', starting_points=16),
                 'device_grid_search': median3(starting_points=1, use_grid_search=True)}
    except Exception as exc:
        extra = {'extra_error': repr(exc)}
    return {'workload': 'cfg2: repeats model k=21 r=100, %d bins, single start, L-BFGS-B' % len(hist),
            'device_s': dev_s, 'device_s_runs': [r[0] for r in runs], 'device_coverage': dev_x[0], 'device_evaluations': dev_n,
            'cpu_s': cpu_s, 'cpu_coverage': cpu_x[0], 'cpu_evaluations': cpu_n, 'cpu_cores': cores,
            'cpu_kind': 'reference' if orc.ref_module() is not None else 'port', **extra}


def reference_histogram(name):
    """The workload histogram of both arms: workload.synthetic_histogram with p_j from the CPU oracle
    instead of the device (the same numbers to ~1e-15), so that it does not depend on the build."""
    from covest_b200 import workload
    from oracle import covest_oracle as orc
    c = workload.CONFIGS[name]
    probe = orc.Model(c['model'], c['k'], c['r'], {j: 1 for j in range(1, c['bins'] + 1)}, 0, max_error=8)
    p = probe.probs(list(c['theta']))
    rng = np.random.default_rng(c['seed'])
    h = rng.poisson(c['kmers'] * np.maximum(p, 0.0))
    return {j: int(v) for j, v in zip(range(1, c['bins'] + 1), h)}


def save_finite(out_dir, name, a):
    """<name>.npy holds `a` with its non-finite entries set to 0 and <name>_nonfinite.npy (float32)
    says which they were: 0 finite, -1 -inf, 1 +inf, 2 NaN.  A point whose likelihood is 0 (a bin
    with counts that it gives probability 0) has log-likelihood -inf, as in the reference."""
    kind = np.where(np.isnan(a), 2, np.where(np.isinf(a), np.sign(a), 0)).astype(np.float32)
    np.save(os.path.join(out_dir, name + '.npy'), np.where(kind == 0, a, 0.0))
    np.save(os.path.join(out_dir, name + '_nonfinite.npy'), kind)


def dump_outputs(out_dir, ll, rows):
    """The log-likelihood of every point of the slice (a fixed seeded sample of them, in index
    order, when there are more than DUMP_MAX_VALUES) and the best rows, as .npy files."""
    os.makedirs(out_dir, exist_ok=True)
    ll = ll.cpu().numpy()
    if len(ll) > DUMP_MAX_VALUES:
        ll = ll[np.sort(np.random.default_rng(0).choice(len(ll), DUMP_MAX_VALUES, replace=False))]
    save_finite(out_dir, 'loglik', ll)
    save_finite(out_dir, 'best_rows', rows.cpu().numpy())


def run_reference(args, rank, world):
    if rank != 0:
        return
    from covest_b200 import workload
    cfg = workload.CONFIGS[args.workload]
    axes = workload_axes(args.workload, world)
    hist = reference_histogram(args.workload)
    cores = os.cpu_count() or 1
    ref = CpuReference(hist, cfg, axes, cores)
    # one step = one bounded sample of the workload: >= 64 lattice points, about 10 s of all cores
    # (BASELINE.md section 3); the size is set once by an untimed probe
    _, _, n = ref.sized_rate(target_s=10.0)
    rates, secs = [], []
    for step in range(args.warmup + args.steps):
        rate, dt = ref.rate(n, seed=5000 + step)
        if step >= args.warmup:
            rates.append(rate)
            secs.append(dt)
    ref.close()
    value = float(np.mean(rates))
    sample = '%d seeded lattice points x %d bins per step (%.1f s), persistent fork pool of %d' % (
        n, len(hist), float(np.mean(secs)), cores)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': float(np.mean(secs) * 1e3),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64 (x87 f80 inside truncated_poisson)',
        'data': 'synthetic', 'config': workload_config(args.workload, world, len(hist), axes),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': ref.kind, 'kind_detail': ref.detail,
                         'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def committed_traffic(kernel, workload_name, n_points):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed
    `ncu --set full` capture of this same command (profiles/, per launch) -- only when this run
    launches the kernel on the batch the capture was taken on; else None."""
    path = os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')
    try:
        with open(path) as f:
            for row in json.load(f):
                if row['kernel'] == kernel and row['workload'] == workload_name and row['points'] == n_points:
                    return {'bytes': row['dram_bytes'], 'source': row['source'],
                            'pipe_fp64_active_pct': row.get('pipe_fp64_active_pct')}
    except (OSError, ValueError, KeyError):
        pass
    return None


def workload_config(name, world, n_bins, axes):
    lens = [len(a) for a in axes]
    from covest_b200 import workload
    c = workload.CONFIGS[name]
    return {'workload': '%s: repeats model k=%d r=%d, lattice %s = %d points x %d bins, %d per rank' % (
        name, c['k'], c['r'], 'x'.join(map(str, lens)), int(np.prod(lens)), n_bins, int(np.prod(lens)) // world),
        'bins': n_bins, 'points_per_rank': int(np.prod(lens)) // world, 'lattice': lens,
        'max_error': 8, 'k_best': K_BEST,
        'points': 'Cartesian lattice, generated on the device from its axes (cvb_lattice_eval)',
        'sharding': 'whole (coverage, error_rate) groups of the lattice dealt round-robin: rank r takes groups r, r+N, ...',
        'l2': 'flushed between timed steps (256 MiB write)'}


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from covest_b200 import parallel, workload
    from covest_b200.models import RepeatsModel

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the library has no CPU path)')
    torch.cuda.set_device(local_rank)
    os.environ['COVEST_B200_DEVICE'] = str(local_rank)
    json_out = sys.stdout
    if world > 1:
        import datetime
        # NCCL prints its version banner on file descriptor 1: everything but the JSON line goes to stderr
        sys.stdout.flush()
        json_out = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank),
                                timeout=datetime.timedelta(seconds=180))
    dev = torch.device('cuda', local_rank)
    stream = torch.cuda.current_stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_device(step, steps, warmup):
        """CUDA-event time of `steps` steps (L2 flushed before each, barrier + synchronize on both
        sides), max over ranks of the total; per-step list of this rank."""
        for _ in range(warmup):
            step()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            flush.fill_(1)
            barrier()
            a.record(stream)
            step()
            b.record(stream)
            barrier()
        ms = [a.elapsed_time(b) for a, b in ev]
        return max_over_ranks(sum(ms)), ms

    def timed_host(step, steps, warmup):
        for _ in range(warmup):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        barrier()
        return max_over_ranks(time.perf_counter() - t0)

    def measure(name, steps, warmup, with_points, dump_dir=None):
        """One workload through every arm of the device path; returns the pieces of a JSON record."""
        cfg = workload.CONFIGS[name]
        hist = reference_histogram(name)
        model = RepeatsModel(cfg['k'], cfg['r'], hist, 0, max_error=8)
        ctx = model.device_context
        if args.path != 'auto':
            ctx.set_path({'prefix': ctx.PATH_FACTORED_PREFIX, 'gemm': ctx.PATH_FACTORED_GEMM,
                          'direct': ctx.PATH_PER_POINT}[args.path])
        n_bins = len(hist)
        axes = workload_axes(name, world)
        total = int(np.prod([len(a) for a in axes]))
        block = int(np.prod([len(a) for a in axes[2:]]))  # whole (c, e) groups, dealt round-robin
        count = total // world
        if args.points:
            count = min(count, args.points)
        count -= count % block
        counted_bins = int(sum(1 for v in hist.values() if v))
        work = workload.lattice_flop(model, axes, count // block, n_bins, counted_bins)
        dev_ll = torch.empty(count, dtype=torch.float64, device=dev)
        dev_rows = torch.empty((K_BEST, 6), dtype=torch.float64, device=dev)
        launches = [0]
        last_rows = [None]

        def step_lattice():  # the headline step: the slice as its axes, everything stays in HBM
            ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, k_best=K_BEST,
                             out_ll=dev_ll, out_rows=dev_rows, stream=stream)
            launches[0] += ctx.last_launches() + (1 if world > 1 else 0)
            last_rows[0] = parallel.merge_topk(parallel.allgather_rows(dev_rows), K_BEST) if world > 1 else dev_rows
            return last_rows[0]

        total_ms, step_ms = timed_device(step_lattice, steps, warmup)
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, dev_ll, last_rows[0])
        n_launch = launches[0] - (launches[0] // (steps + warmup)) * warmup
        value = world * count * n_bins * steps / (total_ms * 1e-3)
        best = step_lattice().cpu().numpy()

        # the kernels of the evaluation alone, CUDA events inside the library on the launching stream
        ctx.set_timing(True)
        kernel_ms, phases = [], []
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, out_ll=dev_ll, stream=stream)
            torch.cuda.synchronize()
            kernel_ms.append(ctx.last_kernel_ms()[0])
            phases.append(ctx.last_path_info())
        ctx.set_timing(False)

        # steps back to back for >= 2 s (no flush: the profile workspace alone is far larger than L2)
        def sustained():
            n = max(steps, int(2200.0 / max(total_ms / steps, 1e-3)))  # total_ms is the max over ranks: the same n everywhere
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(n):
                step_lattice()
            b.record(stream)
            barrier()
            ms = max_over_ranks(a.elapsed_time(b))
            return {'value': world * count * n_bins * n / (ms * 1e-3), 'unit': UNIT, 'steps': n, 'seconds': ms * 1e-3}
        with ClockSampler(local_rank) as clocks:
            sus = sustained()

        # end to end: host buffers, the copies inside the timed region
        def step_host_lattice():
            if world > 1:  # the best rows stay on the device for the all-gather; the values go to host memory
                ll, rows = ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, k_best=K_BEST,
                                            out_rows=dev_rows, stream=stream)
                return ll, parallel.merge_topk(parallel.allgather_rows(rows), K_BEST).cpu().numpy()
            return ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, k_best=K_BEST)
        e2e_steps = max(steps, 30)  # wall-clock timed: enough steps that one hiccup of a rank does not decide it
        e2e_s = timed_host(step_host_lattice, e2e_steps, 3)

        # the call the sharded search makes (grid.lattice_search, CoverageEstimator.compute_coverage_from_lattice):
        # axes in, only the best rows out -- what end to end costs when the caller does not ask for every value
        def step_host_search():
            if world > 1:
                _, rows = ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, k_best=K_BEST,
                                           want_ll=False, out_rows=dev_rows, stream=stream)
                return parallel.merge_topk(parallel.allgather_rows(rows), K_BEST).cpu().numpy()
            return ctx.lattice_eval(axes, first=rank, stride=world, count=count, block=block, k_best=K_BEST,
                                    want_ll=False)[1]
        search_s = timed_host(step_host_search, e2e_steps, 3)
        rec = {
            'cfg': cfg, 'model': model, 'ctx': ctx, 'hist': hist, 'axes': axes, 'count': count, 'block': block,
            'n_bins': n_bins, 'counted_bins': counted_bins, 'work': work, 'value': value, 'total_ms': total_ms,
            'step_ms': step_ms, 'launches': n_launch, 'kernel_ms': kernel_ms, 'phases': phases, 'best': best,
            'sustained': sus, 'clocks': clocks.summary(),
            'e2e': {'value': world * count * n_bins * e2e_steps / e2e_s, 'unit': UNIT, 'steps': e2e_steps,
                    'h2d_bytes_per_step': int(8 * sum(len(a) for a in axes)),
                    'd2h_bytes_per_step': int(count * 8 + K_BEST * 6 * 8),
                    'call': 'cvb_lattice_eval: the candidate lattice handed over as its axes (host), all values '
                            'and the best rows returned to host memory'},
            'e2e_search': {'value': world * count * n_bins * e2e_steps / search_s, 'unit': UNIT, 'steps': e2e_steps,
                           'h2d_bytes_per_step': int(8 * sum(len(a) for a in axes)),
                           'd2h_bytes_per_step': int(K_BEST * 6 * 8),
                           'call': 'cvb_lattice_eval with out_ll = NULL: axes in, the best rows out (what '
                                   'lattice_search / compute_coverage_from_lattice call)'},
        }
        if with_points:
            # the same batch as an explicit point array (the general plan: keys, radix sort, group tables)
            host_pts = workload.lattice_points(axes, first=rank, stride=world, count=count, block=block)
            dev_pts = torch.from_numpy(host_pts).to(dev)

            def step_points():
                ctx.loglik(dev_pts, out=dev_ll, stream=stream)
                rows = ctx.topk(dev_ll, dev_pts, K_BEST, stream=stream)
                if world > 1:
                    rows = parallel.merge_topk(parallel.allgather_rows(rows), K_BEST)
                return rows
            pts_ms, _ = timed_device(step_points, steps, warmup)
            info = ctx.last_path_info()
            rec['explicit_points'] = {'value': world * count * n_bins * steps / (pts_ms * 1e-3), 'unit': UNIT,
                                      'ms_per_step': pts_ms / steps, 'kernel': info['kernel'],
                                      'analytic_plan': info['analytic_plan'],
                                      'note': 'the batch as a point array resident in HBM: cvb_loglik_batch + cvb_topk'}
            pin_pts = torch.from_numpy(host_pts).pin_memory()

            def step_host_points(pts):
                ll, rows = ctx.loglik_topk(pts, K_BEST)
                if world > 1:
                    rows = parallel.merge_topk(parallel.allgather_rows(torch.from_numpy(rows).to(dev)), K_BEST).cpu().numpy()
                return rows
            s_pin = timed_host(lambda: step_host_points(pin_pts.numpy()), steps, 2)
            s_page = timed_host(lambda: step_host_points(host_pts), steps, 2)
            rec['e2e_points'] = {'value': world * count * n_bins * steps / s_pin, 'unit': UNIT,
                                 'pageable_value': world * count * n_bins * steps / s_page,
                                 'h2d_bytes_per_step': int(count * 5 * 8),
                                 'd2h_bytes_per_step': int(count * 8 + K_BEST * 6 * 8),
                                 'call': 'cvb_loglik_topk on an explicit host array (pinned; pageable_value: a plain numpy array)'}
            del dev_pts, pin_pts
        return rec

    def roofline_of(rec, peak_tflops, peak_dmma, name):
        info = rec['phases'][-1]
        km = float(np.mean(rec['kernel_ms']))
        work, n_bins = rec['work'], rec['n_bins']
        factored = info['path'] == 'factored'
        if factored:
            # the kernels after K1 carry the slots of a profile row, not every bin (csrc/factored.h, CvfSlots)
            work = workload.lattice_flop(rec['model'], rec['axes'], rec['count'] // rec['block'], n_bins,
                                         rec['counted_bins'], row_bins=info['row_slots'])
            dom_ms = float(np.mean([p['gemm_ms'] for p in rec['phases']]))
            dominant = info['kernel']
            flop_launch = work['prefix_flop'] if dominant == 'cvf_prefix_kernel' else work['gemm_flop']
        else:
            groups = rec['count'] // rec['block']
            flop_launch = float(n_bins * (workload.FLOP_PER_TERM_BIN * work['sum_terms_per_group'] * groups +
                                          workload.FLOP_PER_BIN * rec['count']))
            dominant, dom_ms = 'cv_loglik_kernel', km
        achieved = flop_launch / (dom_ms * 1e-3) / 1e12
        traffic = committed_traffic(dominant, name, rec['count']) or {}
        terms_sum = work['sum_terms_per_group'] * (rec['count'] // rec['block'])
        roof = {'bound': 'fp64', 'achieved': achieved, 'peak': peak_tflops, 'unit': 'TFLOP/s',
                'frac': achieved / peak_tflops if peak_tflops else None,
                'traffic': traffic.get('bytes'), 'traffic_source': traffic.get('source'),
                'ncu_pipe_fp64_active_pct': traffic.get('pipe_fp64_active_pct'),
                'flop_accounting': 'SURVEY.md section 8(d) / DESIGN.md section 6: 64 flop per (point, bin with a count) '
                                   'for the logarithm and the weighted sum, 6 per (point, slot of a profile row), 2 per '
                                   '(q-run, copy, slot); the logarithm as executed is 9 FP64 instructions -- the pipe '
                                   'utilisation ncu measures is ncu_pipe_fp64_active_pct',
                'kernel': dominant, 'kernel_ms': dom_ms, 'flop_per_launch': flop_launch,
                'mean_terms_per_point': work['mean_terms'],
                'peak_source': 'register-resident DFMA chain measured in this run (cvb_fp64_peak); '
                               'DMMA m8n8k4 chain: %.2f TFLOP/s' % peak_dmma,
                'kernel_share_of_step': dom_ms * len(rec['step_ms']) / rec['total_ms'] if world == 1 else None,
                'survey_accounting': {
                    'primary_flop': float(n_bins * (40.0 * terms_sum + 64.0 * rec['count'])),
                    'secondary_flop': float(n_bins * (4.0 * terms_sum + 64.0 * rec['count'])),
                    'primary_equivalent_tflops': float(n_bins * (40.0 * terms_sum + 64.0 * rec['count'])) / (km * 1e-3) / 1e12,
                    'secondary_equivalent_tflops': float(n_bins * (4.0 * terms_sum + 64.0 * rec['count'])) / (km * 1e-3) / 1e12,
                    'gemm_formulation_flop': work['gemm_flop'] if factored else None,
                    'note': 'SURVEY.md section 8(d): the work of the reference-shaped formulations of the same batch '
                            '(an exp per term and bin / a recurrence) over the time of the whole evaluation here; the '
                            'rates exceed the FP64 peak because the factored formulations do less work for the same values'}}
        phases = ({'path': 'factored', 'kernel': info['kernel'], 'groups': info['groups'], 'q_runs': info['q_runs'],
                   'tiles': info['tiles'], 'analytic_plan': info['analytic_plan'],
                   'refined_points': info['refined_points'],
                   'profile_workspace_bytes': 8 * info['profile_doubles'],
                   'plan_ms': float(np.mean([p['plan_ms'] for p in rec['phases']])),
                   'profile_ms': float(np.mean([p['profile_ms'] for p in rec['phases']])),
                   'kernel_ms': dom_ms, 'evaluation_ms': km, 'profile_flop': work['profile_flop'],
                   'kernel_flop': flop_launch, 'counted_bins': rec['counted_bins'], 'row_slots': info['row_slots'],
                   'mean_copies_per_point': work['mean_copies'],
                   'evaluation_tflops': (work['profile_flop'] + flop_launch) / (km * 1e-3) / 1e12}
                  if factored else {'path': info['path'], 'evaluation_ms': km,
                                    'refined_points': info['refined_points']})
        return roof, phases

    with ClockSampler(local_rank) as clocks:
        main = measure(args.workload, args.steps, args.warmup, with_points=(args.workload == 'cfg3'),
                       dump_dir=args.dump_outputs)
    ctx = main['ctx']
    peak_tflops = ctx.fp64_peak(0) if rank == 0 else None
    peak_dmma = ctx.fp64_peak(1) if rank == 0 else None

    extra = {}
    if args.workload == 'cfg3':
        # seeded uniform-random points of the same box (SURVEY.md section 8(d)): every point has its own
        # (coverage, error rate), nothing to share -- the per-point kernel
        n_rand = min(main['count'], args.points or 1000000)
        rnd = torch.from_numpy(workload.random_box_points(main['cfg']['theta'], n_rand, 31337 + rank)).to(dev)
        rnd_ll = torch.empty(n_rand, dtype=torch.float64, device=dev)

        def step_random():
            ctx.loglik(rnd, out=rnd_ll, stream=stream)
            return ctx.topk(rnd_ll, rnd, K_BEST, stream=stream)
        r_ms, _ = timed_device(step_random, 3, 1)
        info = ctx.last_path_info()
        extra['random_points'] = {'value': world * n_rand * main['n_bins'] * 3 / (r_ms * 1e-3), 'unit': UNIT,
                                  'ms_per_step': r_ms / 3, 'points_per_rank': n_rand, 'kernel': info['kernel'],
                                  'refined_points': info['refined_points'],
                                  'note': 'seeded uniform-random points of the initial_grid box, resident in HBM'}
        # the HBM-bound entry point: per-bin probabilities, 8 B written per point x bin
        n_p = min(100000, main['count'])
        sub = rnd[:n_p].contiguous()
        ctx.probs(sub)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        out_p = ctx.probs(sub, stream=stream)
        b.record(stream)
        torch.cuda.synchronize()
        p_ms = a.elapsed_time(b)
        hbm = None
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                hbm = json.load(f).get('hbm_gbs')
        except (OSError, ValueError):
            pass
        hbm = hbm or 6553.3
        extra['probs_batch'] = {'points': n_p, 'bins': main['n_bins'], 'ms': p_ms,
                                'written_gb_per_s': n_p * main['n_bins'] * 8 / (p_ms * 1e-3) / 1e9,
                                'hbm_peak_gb_per_s': hbm,
                                'frac_of_hbm': n_p * main['n_bins'] * 8 / (p_ms * 1e-3) / 1e9 / hbm,
                                'value': n_p * main['n_bins'] / (p_ms * 1e-3), 'unit': UNIT,
                                'note': 'cvb_probs_batch, device buffers (includes zero-filling the output); compute-bound: '
                                        'the per-point kernel forms every term, the 8 B per point x bin are written once'}
        del out_p, rnd, rnd_ll
        if world == 1 and main['phases'][-1].get('row_slots', 0) < 64 * ((main['n_bins'] + 63) // 64):
            # the same step with every bin carried through K2p (COVEST_B200_ROWS=full, read when a context
            # is created): what the row layout of csrc/factored.h is worth on this histogram
            os.environ['COVEST_B200_ROWS'] = 'full'
            try:
                full = RepeatsModel(main['cfg']['k'], main['cfg']['r'], main['hist'], 0, max_error=8)
                fctx = full.device_context
            finally:
                del os.environ['COVEST_B200_ROWS']
            f_ll = torch.empty(main['count'], dtype=torch.float64, device=dev)
            f_rows = torch.empty((K_BEST, 6), dtype=torch.float64, device=dev)

            def step_full():
                fctx.lattice_eval(main['axes'], count=main['count'], block=main['block'], k_best=K_BEST,
                                  out_ll=f_ll, out_rows=f_rows, stream=stream)
                return f_rows
            f_ms, _ = timed_device(step_full, max(3, args.steps // 2), 2)
            f_steps = max(3, args.steps // 2)
            extra['full_rows'] = {'value': main['count'] * main['n_bins'] * f_steps / (f_ms * 1e-3), 'unit': UNIT,
                                  'ms_per_step': f_ms / f_steps, 'row_slots': fctx.last_path_info()['row_slots'],
                                  'note': 'COVEST_B200_ROWS=full: every line of the histogram in the profile rows, '
                                          'bins without counts carried one by one instead of as 32 sums'}
            full.close()
            del f_ll, f_rows

    cfg5 = None
    if (world == 8 or args.cfg5) and args.workload == 'cfg3' and not args.points and not args.no_cfg5:
        # BASELINE.json configs[4] / the north-star target: 10^8 points x 2000 bins over 8 ranks, per-rank
        # top-64, all-gather, multi-start refinement from the global best rows, second all-gather
        from covest_b200.covest import CoverageEstimator
        main['model'].close()
        torch.cuda.empty_cache()
        c5 = measure('cfg5', max(5, args.steps // 2), 2, with_points=False)
        roof5, phases5 = (None, None)
        if rank == 0:
            roof5, phases5 = roofline_of(c5, peak_tflops, peak_dmma, 'cfg5')
        est = CoverageEstimator(c5['model'], optimizer='lockstep')
        barrier()
        t0 = time.perf_counter()
        x, success, rows = est.compute_coverage_from_lattice(c5['axes'], k_best=K_BEST)
        barrier()
        flow_s = max_over_ranks(time.perf_counter() - t0)
        t0 = time.perf_counter()
        xr, fr, okr, table = est.refine_starts(rows[np.isfinite(rows[:, 0]), 1:])
        barrier()
        refine_s = max_over_ranks(time.perf_counter() - t0)
        if rank == 0:
            cfg5 = {'metric': METRIC, 'value': c5['value'], 'unit': UNIT, 'n_gpus': world, 'steps': len(c5['step_ms']),
                    'ms_per_step': c5['total_ms'] / len(c5['step_ms']),
                    'config': workload_config('cfg5', world, c5['n_bins'], c5['axes']),
                    'e2e': c5['e2e'], 'e2e_search': c5['e2e_search'], 'sustained': c5['sustained'], 'roofline': roof5, 'phases': phases5,
                    'gpu_launches': c5['launches'], 'best_row': [float(v) for v in c5['best'][0]],
                    'refinement': {
                        'flow': 'lattice -> per-rank top-64 -> NCCL all-gather -> merge -> starts dealt round-robin -> '
                                'lock-step Newton refinement on every rank -> all-gather of the refined optima',
                        'flow_seconds': flow_s, 'refine_seconds': refine_s, 'starts': int(len(rows)),
                        'starts_per_rank': int((len(rows) + world - 1) // world),
                        'estimate': [float(v) for v in x], 'success': bool(success),
                        'objective': float(fr), 'best_lattice_loglik': float(rows[0, 0]),
                        'converged_starts': int(np.sum(table[:, 1] > 0)),
                        'launches': est.launches, 'evaluations': est.evaluations}}
        c5['model'].close()

    if rank == 0:
        roof, phases = roofline_of(main, peak_tflops, peak_dmma, args.workload)
        line = {
            'metric': METRIC, 'value': main['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': main['total_ms'] / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args.workload, world, main['n_bins'], main['axes']),
            'e2e': main['e2e'], 'e2e_search': main['e2e_search'], 'gpu_launches': main['launches'], 'clocks': clocks.summary(),
            'sustained': dict(main['sustained'], clocks=main['clocks']),
            'roofline': roof, 'phases': phases, 'best_row': [float(v) for v in main['best'][0]],
        }
        for key in ('explicit_points', 'e2e_points'):
            if key in main:
                line[key] = main[key]
        line.update(extra)
        if cfg5 is not None:
            line['cfg5'] = cfg5
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            ref = CpuReference({j: int(v) for j, v in main['hist'].items()}, main['cfg'], main['axes'], cores)
            rate, dt, n_cpu = ref.sized_rate(target_s=15.0)
            ref.close()
            line['cpu_baseline'] = {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': ref.kind,
                                    'kind_detail': ref.detail,
                                    'sample': '%d seeded lattice points x %d bins in %.1f s, persistent fork pool' % (
                                        n_cpu, main['n_bins'], dt)}
            try:  # BASELINE.json's second figure: covest end-to-end wall time
                line['covest_e2e'] = covest_end_to_end(cores)
            except Exception as exc:  # never lose the throughput line over the extra figure
                line['covest_e2e'] = {'error': repr(exc)}
        print(json.dumps(line), file=json_out, flush=True)
    barrier()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='cfg3', choices=['cfg3', 'cfg4', 'cfg5'])
    ap.add_argument('--points', type=int, default=0, help='cap the points per rank (development)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-cfg5', action='store_true', help='at --gpus 8: skip the cfg5 sub-record')
    ap.add_argument('--cfg5', action='store_true',
                    help='add the cfg5 sub-record at any number of GPUs (12.5e6 points x 2000 bins per rank)')
    ap.add_argument('--path', default='auto', choices=['auto', 'prefix', 'gemm', 'direct'],
                    help='evaluation path of the device arm (development; auto = what a user gets)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the values and best rows of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
