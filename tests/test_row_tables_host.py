"""The row tables of a histogram without a tail (covest_b200/csrc/cvtables.h, cv_build_row_tables), built on
the host: which histograms get them and their shape.

tests/test_gpu_counted_rows.py runs the device on these histograms; this pins the shapes its comments state
(rows per group NA 1, 2, 4 and 8), and that the second histogram of each of its pairs runs on full tables
that are the first one's row tables plus one group: the premise of its bit-identity test.
"""
import os
import subprocess

import numpy as np
import pytest

from tests import test_gpu_counted_rows as rows

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'covest_b200', 'csrc')
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

SOURCE = r'''
#include <cstdio>
#include <vector>
#include "cvtables.h"
static void show(const char *what, const CvHostTables &T)
{
    printf("%s %d %d %d %zu", what, T.na, T.n_groups, T.n_blocks, T.slot_h.size() / 64);
    for (int i = 0; i < T.n_groups * CV_GD; i++)
        printf(" %a", T.grp[i]);
    printf("\n");
}
int main()
{
    std::vector<int> j;
    std::vector<double> h;
    int a;
    double b;
    while (scanf("%d %lf", &a, &b) == 2) {
        j.push_back(a);
        h.push_back(b);
    }
    CvHostTables T, R;
    if (!cv_build_tables((int)j.size(), j.data(), h.data(), T).empty())
        return 1;
    show("full", T);
    if (cv_build_row_tables(T, j.data(), h.data(), R))
        show("rows", R);
    return 0;
}
'''


@pytest.fixture(scope='module')
def tables_tool(tmp_path_factory):
    d = tmp_path_factory.mktemp('row_tables')
    src, exe = d / 'tables.cpp', d / 'tables'
    src.write_text(SOURCE)
    subprocess.check_call(['g++', '-O1', '-std=gnu++17', '-ffp-contract=off', '-I', CSRC, str(src), '-o', str(exe)])

    def run(hist):
        out = subprocess.run([str(exe)], input=''.join('%d %r\n' % (j, float(v)) for j, v in hist.items()),
                             capture_output=True, text=True, check=True).stdout
        tables = {}
        for line in out.splitlines():
            f = line.split()
            tables[f[0]] = {'na': int(f[1]), 'groups': int(f[2]), 'blocks': int(f[3]), 'lines': int(f[4]), 'grp': f[5:]}
        return tables
    return run


# rows per group of the row tables, None: the full tables stay
EXPECTED_NA = {'line0': 1, 'line1': 1, 'last_line': 1, 'lines013': 2, 'lines0to5': 4, 'lines025': 2, 'sparse_keys': 4,
               'lines0to8': 8, 'cfg4': None, 'all_zero': None}


def test_every_histogram_of_the_device_test_is_stated():
    assert set(EXPECTED_NA) == set(rows.HISTS)


@pytest.mark.parametrize('name', sorted(EXPECTED_NA))
def test_row_tables_of_the_device_test_histograms(tables_tool, name):
    t = tables_tool(rows._hist(name))
    if EXPECTED_NA[name] is None:
        assert 'rows' not in t
        return
    r = t['rows']
    assert r['na'] == EXPECTED_NA[name] and r['blocks'] == 1 and r['lines'] < t['full']['lines']
    assert t['full']['na'] == 8


@pytest.mark.parametrize('name', rows.PAIRS)
def test_the_second_histogram_of_a_pair_runs_on_the_first_ones_row_tables(tables_tool, name):
    a = tables_tool(rows._hist(name))['rows']
    b = tables_tool(rows._counted_keys_only(rows._hist(name), rows._line))
    assert 'rows' not in b
    full = b['full']
    assert (full['na'], full['blocks'], full['lines']) == (a['na'], a['blocks'], a['lines'])
    assert full['groups'] in (a['groups'], a['groups'] + 1)
    assert full['grp'][:len(a['grp'])] == a['grp']


@pytest.mark.parametrize('name,na,lines', [('cfg3', 2, 4), ('cfg5', 2, 4), ('cfg4', None, None)])
def test_row_tables_of_the_benchmark_histograms(tables_tool, name, na, lines):
    z = np.load(os.path.join(GOLDEN, 'big_%s.npz' % name))
    t = tables_tool(dict(zip(z['hist_j'].tolist(), z['hist_h'].tolist())))
    if na is None:
        assert 'rows' not in t   # three blocks of row tables: the full tables stay (cvtables.h)
    else:
        assert (t['rows']['na'], t['rows']['lines']) == (na, lines)
