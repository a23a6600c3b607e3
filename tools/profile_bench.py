#!/usr/bin/env python
"""Cost of profile likelihoods on one GPU; prints one JSON object.

  lattice   the cfg3 lattice (40 x 25 x 10 x 10 x 10 = 10^6 points, 1000-bin histogram), device buffers:
            cvb_lattice_eval with k_best = 1, and cvb_lattice_profile with keep masks coverage (40
            segments) and (coverage, error_rate) (1000 segments), in alternation after warm-up, CUDA
            events around each call; median and spread in ms
  cli       wall time of `covest <cfg2 fixture> -m repeat -k 21 -r 100 -sf 1 --polish`, without and with
            --ci 0.95 (tests/golden/e2e_golden.json, the cfg2 repeats histogram)

The card's name and power limit are read in the same run and reported with the numbers.

    python tools/profile_bench.py [--reps 40] [--warmup 5]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from covest_b200 import workload  # noqa: E402
from covest_b200.models import RepeatsModel  # noqa: E402


def card():
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        out['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except Exception as exc:  # the numbers stand without it, marked as such
        out['power_limit_and_max_sm_clock'] = 'not read: %s' % exc
    return out


def lattice(reps, warmup):
    cfg = workload.CONFIGS['cfg3']
    model = RepeatsModel(cfg['k'], cfg['r'], workload.synthetic_histogram('cfg3'), 0, max_error=8)
    ctx = model.device_context
    axes = workload.lattice_axes(cfg['theta'], n_c=40, n_e=25)
    dev = torch.device('cuda', ctx.device)
    best = torch.empty((1, 6), dtype=torch.float64, device=dev)
    prof = {1: torch.empty((40, 6), dtype=torch.float64, device=dev),
            3: torch.empty((1000, 6), dtype=torch.float64, device=dev)}
    calls = {'lattice_eval_k1': lambda: ctx.lattice_eval(axes, want_ll=False, k_best=1, out_rows=best),
             'lattice_profile_c': lambda: ctx.lattice_profile(axes, 1, out_rows=prof[1]),
             'lattice_profile_ce': lambda: ctx.lattice_profile(axes, 3, out_rows=prof[3])}
    times = {k: [] for k in calls}
    for rep in range(warmup + reps):
        for name, call in calls.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            call()
            b.record()
            torch.cuda.synchronize()
            if rep >= warmup:
                times[name].append(a.elapsed_time(b))
    # the rows of the profile against the top-1 of the evaluation: the best segment is the best point
    top = best.cpu().numpy()[0]
    rows = prof[3].cpu().numpy()
    assert rows[int(np.argmax(rows[:, 0]))].tolist() == top.tolist()
    out = {k: {'median_ms': float(np.median(v)), 'min_ms': float(np.min(v)), 'max_ms': float(np.max(v))}
           for k, v in times.items()}
    base = out['lattice_eval_k1']['median_ms']
    for k in ('lattice_profile_c', 'lattice_profile_ce'):
        out[k]['over_eval'] = out[k]['median_ms'] / base - 1.0
    out['points'] = int(np.prod([len(a) for a in axes]))
    return out


def cli_wall():
    from covest_b200 import covest as cli
    with open(os.path.join(ROOT, 'tests', 'golden', 'e2e_golden.json')) as f:
        g = json.load(f)['cfg2_repeats']
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, 'cfg2.hist')
        with open(path, 'w') as f:
            f.write(''.join('%d %d\n' % (j, h) for j, h in g['hist']))
        cwd = os.getcwd()
        os.chdir(tmp)
        try:
            base = [path, '-m', 'repeat', '-k', '21', '-r', '100', '-sf', '1', '--polish', '--seed', '1']
            for name, argv in (('warm_up', base), ('polish', base), ('polish_ci95', base + ['--ci', '0.95'])):
                t0 = time.perf_counter()
                with contextlib.redirect_stdout(io.StringIO()) as buf:
                    cli.run(argv)
                out[name + '_s'] = time.perf_counter() - t0
                if name == 'polish_ci95':
                    import yaml
                    rep = yaml.safe_load(buf.getvalue())
                    out['report'] = {k: rep[k] for k in rep if k.endswith('_ci') or k in ('ci_flags', 'coverage',
                                                                                         'genome_size')}
        finally:
            os.chdir(cwd)
    out.pop('warm_up_s')
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    p.add_argument('--reps', type=int, default=40)
    p.add_argument('--warmup', type=int, default=5)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('profile_bench.py measures on a CUDA device; none is visible')
    print(json.dumps({'card': card(), 'lattice': lattice(args.reps, args.warmup), 'cli': cli_wall()}, indent=1))


if __name__ == '__main__':
    main()
