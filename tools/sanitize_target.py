#!/usr/bin/env python
"""Small batches through every kernel of the library, for compute-sanitizer (memcheck, racecheck,
synccheck, initcheck): the per-point kernel (basic and repeats, with per-bin probabilities), the plan
kernels (general and from lattice axes), the profile kernel, the prefix kernel (with and without a
tail), the GEMM path, the term-by-term re-evaluation, the three top-K selections and the row merge.

    compute-sanitizer --tool racecheck python tools/sanitize_target.py
    compute-sanitizer --tool initcheck python tools/sanitize_target.py

(initcheck reads of device memory never written; tests/test_gpu_poison.py covers the same ground
where the tool cannot run.)
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from covest_b200 import parallel, workload  # noqa: E402
from covest_b200.models import BasicModel, RepeatsModel  # noqa: E402
from tests.helpers import case_hist, load_case  # noqa: E402

case = load_case('cfg2_repeats')
hist = case_hist(case)
done = []
basic = BasicModel(21, 100, hist, 0, max_error=8)
ll = basic.loglikelihood_batch(np.array(load_case('cfg1_basic')['points'][:64]))
p = basic.probabilities_batch(np.array([[10, .03], [25, .01]]))
basic.close()
done.append('basic')

for tail in (0, 1234):
    model = RepeatsModel(21, 100, hist, tail, max_error=8)
    ctx = model.device_context
    axes = [np.geomspace(10, 90, 5), np.geomspace(.01, .09, 3), np.linspace(.3, 1, 5), np.linspace(0, 1, 5),
            np.linspace(.02, 1, 11)]
    pts = workload.lattice_points(axes)
    a, rows = ctx.lattice_eval(axes, k_best=8)                     # plan from the axes, prefix kernel
    assert ctx.last_path_info()['kernel'] == 'cvf_prefix_kernel'
    b = ctx.loglik(pts)                                            # general plan (sort), prefix kernel
    ctx.set_path(ctx.PATH_FACTORED_GEMM)
    c = ctx.loglik(pts)
    ctx.set_path(ctx.PATH_PER_POINT)
    d = ctx.loglik(pts[:600])
    ctx.set_path(ctx.PATH_TERM_BY_TERM)
    e = ctx.loglik(pts[:300])
    ctx.set_path(ctx.PATH_AUTO)
    assert np.array_equal(a, b, equal_nan=True)
    fin = np.isfinite(d)
    assert np.max(np.abs(c[:600][fin] - d[fin]) / np.abs(d[fin])) < 1e-10
    fin = np.isfinite(e)
    assert np.max(np.abs(e[fin] - d[:300][fin]) / np.abs(d[:300][fin])) < 1e-10
    probs = ctx.probs(pts[:16], clip=True)
    big = np.tile(b, 12)[:40000]                                   # radix selection needs >= 32768 values
    ctx.topk(big, np.tile(pts, (12, 1))[:40000], 16)
    ctx.topk(b[:5000], pts[:5000], 8)
    model.close()
    done.append('repeats tail=%s' % tail)

import torch  # noqa: E402
rows = torch.from_numpy(np.random.default_rng(1).normal(size=(128, 6))).cuda()
parallel.merge_topk(rows, 16)
torch.cuda.synchronize()
done.append('merge')
print('sanitize target ok:', '; '.join(done))
