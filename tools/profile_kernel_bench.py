#!/usr/bin/env python
"""Time of the profile kernel (K1, cvf_profile_kernel) alone on the benchmark's lattices; prints one JSON object.

  cfg3       bench.py's headline lattice (10^6 points, 1000 bins); no tail: K1 runs on the row tables, 2 rows per
             group (NA = 2)
  cfg3_full  the same with COVEST_B200_ROWS=full: every line of the histogram, NA = 8
  cfg3_na4   the same lattice on cfg3's histogram with a count of 1 in every empty bin up to 384: six lines with
             counts, row tables with NA = 4 (no benchmark workload runs at NA = 4)
  cfg4       10^5 points, 5000 bins: the full tables stay (NA = 8, five blocks of groups)
  cfg5       12.5 * 10^6 points, 2000 bins: row tables, NA = 2

tests/test_row_tables_host.py pins the NA of cfg3, cfg4 and cfg5.  Each call is one cvb_lattice_eval of the whole
lattice with the library's CUDA events on (set_timing); `profile_ms` of cvb_last_path_info is K1 plus the tile-order
kernel of the lattice (a few microseconds).  A 256 MiB buffer is overwritten before every call, so that no call finds the
previous one's profiles in L2.  Median, min and max over --reps calls after --warmup; `kernel_ms` is the prefix
kernel (K2p) of the same calls, which K1's changes must leave alone.  The card's name, power limit and max SM
clock are read in the same run and reported with the numbers.

    python tools/profile_kernel_bench.py [--reps 20] [--warmup 3] [--workloads cfg3,cfg3_full,cfg3_na4,cfg4,cfg5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import reference_histogram, workload_axes  # noqa: E402
from covest_b200 import workload  # noqa: E402
from covest_b200.models import RepeatsModel  # noqa: E402

WORKLOADS = {'cfg3': ('cfg3', None), 'cfg3_full': ('cfg3', 'full'), 'cfg3_na4': ('cfg3', None), 'cfg4': ('cfg4', None),
             'cfg5': ('cfg5', None)}


def card():
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        out['power_limit_and_max_sm_clock'] = q.stdout.strip() or q.stderr.strip()
    except Exception as exc:  # the numbers stand without it, marked as such
        out['power_limit_and_max_sm_clock'] = 'not read: %s' % exc
    return out


def time_k1(label, reps, warmup, flush):
    name, rows = WORKLOADS[label]
    cfg = workload.CONFIGS[name]
    hist = reference_histogram(name)
    if label == 'cfg3_na4':
        hist = {j: h or (1 if j <= 384 else 0) for j, h in hist.items()}
    if rows:
        os.environ['COVEST_B200_ROWS'] = rows  # read when the context is created
    try:
        model = RepeatsModel(cfg['k'], cfg['r'], hist, 0, max_error=8)
        ctx = model.device_context
    finally:
        os.environ.pop('COVEST_B200_ROWS', None)
    axes = workload_axes(name, 1)
    count = int(np.prod([len(a) for a in axes]))
    block = int(np.prod([len(a) for a in axes[2:]]))
    ll = torch.empty(count, dtype=torch.float64, device=torch.device('cuda', ctx.device))
    ctx.set_timing(True)
    k1, k2p = [], []
    for rep in range(warmup + reps):
        flush.fill_(rep & 0xff)
        torch.cuda.synchronize()
        ctx.lattice_eval(axes, count=count, block=block, out_ll=ll)
        torch.cuda.synchronize()
        info = ctx.last_path_info()
        if rep >= warmup:
            k1.append(info['profile_ms'])
            k2p.append(info['gemm_ms'])
    ctx.set_timing(False)
    model.close()
    assert info['kernel'] == 'cvf_prefix_kernel', info
    return {'profile_ms': float(np.median(k1)), 'profile_ms_min': float(np.min(k1)),
            'profile_ms_max': float(np.max(k1)), 'kernel_ms': float(np.median(k2p)), 'items': info['items'],
            'row_slots': info['row_slots'], 'points': count}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default=','.join(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('profile_kernel_bench.py measures on a GPU; none is visible')
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    out = {'card': card(), 'reps': args.reps, 'warmup': args.warmup, 'workloads': {}}
    for label in args.workloads.split(','):
        out['workloads'][label] = time_k1(label, args.reps, args.warmup, flush)
    print(json.dumps(out))


if __name__ == '__main__':
    main()
