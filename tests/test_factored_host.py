"""Host decisions of the batched path's driver (covest_b200/csrc/factored.h), built on the host: the geometry of
the prefix kernel per row length, and the cut of a plan's groups into ranges whose profiles fit the workspace.
"""
import os
import subprocess

import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'covest_b200', 'csrc')

SOURCE = r'''
#include <cstdio>
#include <vector>
#include "factored.h"
int main(int argc, char **argv)
{
    if (argc > 1) { /* the geometry for 1 .. 48 half-lines */
        for (int h = 1; h <= 48; h++) {
            const CvfPrefixGeometry g = cvf_prefix_geometry(h);
            printf("%d %d\n", g.nw, g.sl);
        }
        return 0;
    }
    size_t w_limit;
    int n;
    if (scanf("%zu %d", &w_limit, &n) != 2)
        return 1;
    std::vector<int> tile(n + 1), item(n + 1), achunk(n + 1);
    std::vector<long long> woff(n + 1);
    for (int g = 0; g <= n; g++)
        if (scanf("%d %d %d %lld", &tile[g], &item[g], &achunk[g], &woff[g]) != 4)
            return 1;
    for (const CvfRange &r : cvf_group_ranges(tile, item, achunk, woff, w_limit))
        printf("%d %d %d %d %d %d %lld %lld %lld %lld\n", r.g0, r.g1, r.tile0, r.tile1, r.item0, r.item1, r.w0, r.w1,
               r.a0, r.a1);
    return 0;
}
'''

# (warps, slots per thread) of the prefix kernel for rows of 1 .. 48 half-lines
GEOMETRY = [(1, 3), (1, 3), (1, 3), (1, 4), (2, 3), (2, 3), (2, 4), (2, 4),
            (3, 3), (3, 4), (3, 4), (3, 4), (4, 4), (4, 4), (4, 4), (4, 4),
            (6, 3), (6, 3), (6, 4), (6, 4), (6, 4), (6, 4), (6, 4), (6, 4)] + [(8, 4)] * 24


@pytest.fixture(scope='module')
def tool(tmp_path_factory):
    d = tmp_path_factory.mktemp('factored_host')
    src, exe = d / 'factored.cpp', d / 'factored'
    src.write_text(SOURCE)
    subprocess.check_call(['g++', '-O1', '-std=gnu++17', '-ffp-contract=off', '-I', CSRC, '-I', '/usr/local/cuda/include',
                           str(src), '-o', str(exe)])
    return str(exe)


def test_prefix_geometry(tool):
    out = subprocess.run([tool, 'geometry'], capture_output=True, text=True, check=True).stdout
    assert [tuple(map(int, line.split())) for line in out.splitlines()] == GEOMETRY


def _prefix(counts):
    out = [0]
    for c in counts:
        out.append(out[-1] + c)
    return out


def _reference_cuts(woff, w_limit):
    """The group boundaries: a range grows while its profiles fit w_limit, and holds at least one group."""
    n, cut, g0 = len(woff) - 1, [0], 0
    while g0 < n:
        g1 = g0 + 1
        while g1 < n and woff[g1 + 1] - woff[g0] <= w_limit:
            g1 += 1
        cut.append(g1)
        g0 = g1
    return cut


# (profile doubles per group, w_limit, the boundaries): equal groups, a limit exactly at a boundary, one group
# larger than the limit, a group alone between larger ones
CASES = [
    ([1024] * 8, 4096, [0, 4, 8]),
    ([1024] * 8, 4095, [0, 3, 6, 8]),
    ([1024] * 7, 1024, [0, 1, 2, 3, 4, 5, 6, 7]),
    ([512, 512, 9000, 512, 256, 256, 2048], 2048, [0, 2, 3, 6, 7]),
    ([3000, 100, 3000, 100, 100], 2048, [0, 1, 2, 3, 5]),
    ([16384], 1024, [0, 1]),
]


@pytest.mark.parametrize('w,w_limit,cuts', CASES)
def test_group_ranges(tool, w, w_limit, cuts):
    n = len(w)
    woff = _prefix(w)
    tile, item, achunk = _prefix([g % 3 + 1 for g in range(n)]), _prefix([2 * g + 1 for g in range(n)]), \
        _prefix([g % 2 for g in range(n)])
    stdin = '%d %d\n' % (w_limit, n) + ''.join('%d %d %d %d\n' % t for t in zip(tile, item, achunk, woff))
    out = subprocess.run([tool], input=stdin, capture_output=True, text=True, check=True).stdout
    ranges = [tuple(map(int, line.split())) for line in out.splitlines()]
    assert _reference_cuts(woff, w_limit) == cuts
    assert [r[0] for r in ranges] + [ranges[-1][1]] == cuts
    for g0, g1, t0, t1, i0, i1, w0, w1, a0, a1 in ranges:
        assert (t0, t1, i0, i1, w0, w1, a0, a1) == (tile[g0], tile[g1], item[g0], item[g1], woff[g0], woff[g1],
                                                    achunk[g0], achunk[g1])
        assert w1 - w0 <= w_limit or g1 - g0 == 1
