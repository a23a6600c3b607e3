"""Compare two `bench.py --dump-outputs DIR` directories, e.g. the outputs of two builds on one workload.

    python tools/compare_dumps.py DIR_A DIR_B [--rtol 1e-12]

For loglik and best_rows it checks that the non-finite masks (<name>_nonfinite.npy) are identical and
reports the largest relative difference of the finite values; for best_rows it also checks that the
parameter columns (every column after the log-likelihood) are equal, i.e. both builds picked the same
points in the same order.  Prints one JSON line; the exit code is 1 when a check fails or a relative
difference exceeds --rtol.
"""
import argparse
import json
import os
import sys

import numpy as np


def load(d, name):
    return np.load(os.path.join(d, name + '.npy')), np.load(os.path.join(d, name + '_nonfinite.npy'))


def max_rel(a, b):
    with np.errstate(divide='ignore', invalid='ignore'):
        rel = np.abs(a - b) / np.abs(b)
    rel[a == b] = 0.0
    return float(rel.max()) if rel.size else 0.0


def compare(dir_a, dir_b, rtol):
    out, ok = {}, True
    for name in ('loglik', 'best_rows'):
        a, ka = load(dir_a, name)
        b, kb = load(dir_b, name)
        rec = {'shape_equal': a.shape == b.shape}
        if rec['shape_equal']:
            rec['nonfinite_equal'] = bool(np.array_equal(ka, kb))
            fin = (ka == 0) & (kb == 0)
            rec['finite'] = int(fin.sum())
            rec['max_rel_diff'] = max_rel(a[fin], b[fin])
            ok = ok and rec['nonfinite_equal'] and rec['max_rel_diff'] <= rtol
            if name == 'best_rows':
                rec['params_equal'] = bool(np.array_equal(a[:, 1:], b[:, 1:]) and np.array_equal(ka[:, 1:], kb[:, 1:]))
                ok = ok and rec['params_equal']
        ok = ok and rec['shape_equal']
        out[name] = rec
    out['ok'] = ok
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('dir_a')
    ap.add_argument('dir_b')
    ap.add_argument('--rtol', type=float, default=1e-12, help='largest accepted relative difference of finite values')
    args = ap.parse_args()
    res = compare(args.dir_a, args.dir_b, args.rtol)
    print(json.dumps(res))
    return 0 if res['ok'] else 1


if __name__ == '__main__':
    sys.exit(main())
