"""The profile kernel (K1, cvf_profile_kernel in csrc/factored.cu) at every rows-per-group NA and CTA size.

K1 has one instantiation per NA, each with its own warps per CTA (16 for NA <= 4, 12 for NA = 8), and the
launch takes fewer when the group records of a long histogram and the working sets of a large S leave no
room.  Whatever the CTA size, each work item (a group and 16 copy numbers) must come out the same, so the
values may not depend on which warp ran which item.

For histograms whose row tables (no tail: the tables K1 runs on) have NA = 1, 2, 4 and 8, and S = 1, 8, 17
and 32, and for a 14 400-key histogram on its full tables (NA = 8, 15 blocks of group records) at S = 32,
where 11 warps fit instead of 12:
- the lattice values of the prefix and GEMM paths are bit-identical between a default context and one with
  COVEST_B200_PROFILE_MIB=1, whose small profile workspace splits K1 into many launches over a few groups
  each, so that the warps meet the items in another order;
- a sample matches the oracle (1e-9).
The NA is that of the row tables the host builds for the histogram (csrc/cvtables.h, the tool of
tests/test_row_tables_host.py), and `row_slots` shows that the batched path ran on those row tables.
"""
import subprocess

import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests import test_gpu_counted_rows as rows
from tests import test_row_tables_host
from tests.helpers import rel_err_ll

pytestmark = pytest.mark.gpu

LL_RTOL = 1e-9
NA_OF = {'line0': 1, 'lines013': 2, 'lines0to5': 4, 'lines0to8': 8}
CASES = [(name, S) for name in NA_OF for S in (1, 8, 17, 32)]


@pytest.fixture(scope='module')
def row_tables_na(tmp_path_factory):
    d = tmp_path_factory.mktemp('profile_geometry')
    src, exe = d / 'tables.cpp', d / 'tables'
    src.write_text(test_row_tables_host.SOURCE)
    subprocess.check_call(['g++', '-O1', '-std=gnu++17', '-ffp-contract=off', '-I', test_row_tables_host.CSRC,
                           str(src), '-o', str(exe)])

    def na(hist):
        out = subprocess.run([str(exe)], input=''.join('%d %r\n' % (j, float(v)) for j, v in hist.items()),
                             capture_output=True, text=True, check=True).stdout
        return {f[0]: int(f[1]) for f in (line.split() for line in out.splitlines())}['rows']
    return na


def _axes(name):
    """16 x 4 (coverage, error rate) groups: 1 MiB holds the profiles of at most 16 of them"""
    _, cov, err, q = rows.HISTS[name]
    return [np.linspace(cov[0], cov[1], 16), np.linspace(err[0], err[1], 4), np.array([0.4, 0.8]),
            np.array([0.0, 0.3, 0.7]), np.asarray(q)]


def _long_hist():
    """14 400 keys, counts in lines 0 .. 8 as in 'lines0to8'"""
    rng = np.random.default_rng(11)
    return {j: (int(rng.integers(1, 10 ** 6 // j + 2)) if j <= 576 else 0) for j in range(1, 14401)}


def _lattice(ctx, path, axes):
    ctx.set_path(path)
    ll, _ = ctx.lattice_eval(axes)
    return ll, ctx.last_path_info(), ctx.last_launches()


def _check(hist, S, k, r, axes, row_slots, env=()):
    pts = rows._grid(axes)
    pick = np.random.default_rng(S).choice(len(pts), 24, replace=False)
    want = orc.Model('repeats', k, r, hist, 0, max_error=S).loglik_batch(pts[pick], threads=8)
    with rows._context(hist, S, k, r, env=env) as whole, \
            rows._context(hist, S, k, r, env=env + (('COVEST_B200_PROFILE_MIB', '1'),)) as split:
        for path in (whole.PATH_FACTORED_PREFIX, whole.PATH_FACTORED_GEMM):
            a, ia, na_ = _lattice(whole, path, axes)
            b, ib, nb_ = _lattice(split, path, axes)
            assert ia['path'] == 'factored' and ia['row_slots'] == row_slots
            assert nb_ >= na_ + 6, (path, na_, nb_)  # three or more group ranges, each with its K1 launch
            assert np.isfinite(a).sum() >= len(pts) // 2
            assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), path
            assert np.array_equal(np.isinf(a[pick]), np.isinf(want)), path
            assert rel_err_ll(a[pick], want).max() <= LL_RTOL, (path, float(rel_err_ll(a[pick], want).max()))


@pytest.mark.parametrize('name,S', CASES, ids=['%s-S%d' % c for c in CASES])
def test_profiles_do_not_depend_on_the_cta_size_or_the_launch_split(row_tables_na, name, S):
    hist = rows._hist(name)
    assert row_tables_na(hist) == NA_OF[name]
    k, r = rows._kr(name, S)
    _check(hist, S, k, r, _axes(name), 64 * rows._counted_lines(hist) + 32)


def test_a_cta_with_fewer_warps_than_its_instantiation_gives_the_same_values():
    """COVEST_B200_ROWS=full keeps K1 on the full tables: 15 blocks of 8 groups of 8 rows take 15 KB of group
    records, and a warp at S = 32 takes 18 240 bytes (working set and an NA = 8 stage), so 11 of K1's 12
    warps fit the 227 KB of a CTA"""
    hist = _long_hist()
    _, cov, err, q = rows.HISTS['lines0to8']
    axes = [np.linspace(cov[0], cov[1], 8), np.array(err), np.array([0.4, 0.8]), np.array([0.3, 0.7]), np.asarray(q[:3])]
    _check(hist, 32, 31, 100, axes, 64 * 240, env=(('COVEST_B200_ROWS', 'full'),))  # every line of the tables
