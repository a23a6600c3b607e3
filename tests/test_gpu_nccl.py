"""The multi-GPU flow on real devices: world size 2 over NCCL (needs two GPUs; skipped otherwise).
tests/test_parallel_gloo.py covers the same host logic on CPU over gloo."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_lattice_and_refinement_over_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    out = str(tmp_path / 'out.json')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
           '--master-addr', '127.0.0.1', '--master-port', '29544',
           os.path.join(ROOT, 'tests', 'nccl_worker.py'), out]
    subprocess.run(cmd, check=True, timeout=600, cwd=ROOT, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    with open(out) as f:
        res = json.load(f)
    assert res['world'] == 2 and res['backend'] == 'nccl'
    assert res['rows_equal_single_rank']      # sharding does not change the global best rows ...
    assert res['rows2_equal']
    assert res['x'] == res['single_x']        # ... nor the refined optimum
    assert res['ok'] and res['refined_ll'] >= res['best_lattice_ll']
    assert res['per_rank'][0] == res['per_rank'][1]   # every rank holds the same answers
