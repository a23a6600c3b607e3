"""Device scratch that a kernel reads without having written it in the same call, and output elements
that no kernel writes.

Contexts made with COVEST_B200_POISON=nan (bytes 0xFF: every double a NaN) or =finite (bytes 0x7F:
every double ~1.4e306) fill the double scratch of each call before its first kernel: the profile
workspace and copy-weight tiles of the factored path, the prefix kernel's partials, the term-by-term
accumulators, the staging of values and probabilities, and the top-K value buffers.  A stale read then
shows: a NaN survives a multiplication by an exact zero, and a huge finite value gets past the checks
that a NaN would send down another path (a NaN probability is re-evaluated term by term).

A. Poisoned and clean contexts give the same values, bit for bit, on every path, histogram shape,
   number of error classes and last chunk of the profile kernel; a sample is checked against the oracle.
B. Every element of every output is written and nothing around it: outputs are pre-filled with a
   sentinel NaN and framed by guard zones, host and device buffers alike.
C. A sequence of calls in one poisoned context, which grows, shrinks and re-plans its workspaces,
   gives what a fresh clean context gives for each call.

What this cannot see: shared memory, registers, and the index and count buffers (plan tables, marked
points, work counters, top-K indices and radix scratch, the lattice template), which are not poisoned
because a poisoned index could fault.  Part C covers the plan tables and the template instead.
"""
import contextlib
import ctypes
import functools

import numpy as np
import pytest

from oracle import covest_oracle as orc
from tests.helpers import context_for
from tests import test_gpu_rows
from tests.test_gpu_error_classes import LL_RTOL, _assert_close, _gate, _hist

pytestmark = pytest.mark.gpu

POISONS = ('nan', 'finite')
POISON_BITS = {'nan': 0xFFFFFFFFFFFFFFFF, 'finite': 0x7F7F7F7F7F7F7F7F}
THRESHOLD = 1e-8  # orc.Model's default, the cut-off threshold of models.py:183


@functools.lru_cache(maxsize=None)
def _histogram(name):
    """(hist, tail): a histogram of tests/test_gpu_error_classes.py, or 'sparse700', the 700 keys of
    tests/test_gpu_rows.py with a tail of 5000.  There the lines without counts travel as one line whose
    first half holds their sums (csrc/factored.h, CvfSlots), and with a tail every slot of a row enters
    the mass, the second half of that line too."""
    if name == 'sparse700':
        return test_gpu_rows.sparse_hist(), test_gpu_rows.TAIL
    return _hist(name)


@contextlib.contextmanager
def _context(m, poison=None, env=()):
    """A device context for the oracle model `m`, made with COVEST_B200_POISON=poison (None: clean,
    also when the variable is set around the test run) and the other variables of `env`, which the
    library reads when the context is created."""
    with pytest.MonkeyPatch.context() as mp:
        for k, v in env:
            mp.setenv(k, v)
        if poison:
            mp.setenv('COVEST_B200_POISON', poison)
        else:
            mp.delenv('COVEST_B200_POISON', raising=False)
        ctx = context_for(m)
    try:
        yield ctx
    finally:
        ctx.close()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _assert_same(got, want, what):
    """Bit for bit, except that NaNs compare as NaNs."""
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    differ = (nan_g != nan_w) | (~nan_w & (_bits(got) != _bits(want)))
    if differ.any():
        i = np.flatnonzero(differ)
        raise AssertionError('%s: %d of %d values differ from the clean context, first at %s: %r instead of %r'
                             % (what, len(i), len(got), i[:8].tolist(), got[i[:4]].tolist(), want[i[:4]].tolist()))


# ---- the points ----------------------------------------------------------------------------------
def _grid(axes):
    return np.ascontiguousarray(np.array(np.meshgrid(*axes, indexing='ij')).reshape(len(axes), -1).T)


def _lattice_axes(name, small):
    """Repeats lattice: q down to 0.05 (cut-offs of up to ~300 copies, many 16-copy chunks).  The large
    one has 2112 points or more, so that the automatic choice takes the factored path (from 2048 points,
    include/covest_b200.h); the small one serves the slow term-by-term path.  e = 0.3 on the 15-bin
    histogram gives the classes up to ~16 a weight (tests/test_gpu_error_classes.py)."""
    errs = [0.004, 0.03] + ([0.3] if name == 'e05_repeats' else [])
    if small:
        return (np.array([20.0, 40.0]), np.array(errs), np.array([0.3, 0.65, 1.0]), np.array([0.0, 0.5, 1.0]),
                np.array([0.05, 0.1, 0.2, 0.4, 0.7, 1.0]))
    return (np.array([15.0, 20.0, 30.0, 40.0]), np.array(errs + [0.01]), np.array([0.3, 0.5, 0.75, 1.0]),
            np.array([0.0, 0.3, 0.7, 1.0]), np.array([0.05, 0.08, 0.1, 0.15, 0.2, 0.3, 0.4, 0.55, 0.7, 0.85, 1.0]))


def _cutoff(q1, q2, q, top, thr=THRESHOLD):
    """O_thr of models.py:185-191 (oracle/covest_oracle.py py_probs): copies o < O_thr enter."""
    two = (1 - q1) * q2
    many = (1 - q1) * (1 - q2) * q
    for o in range(1, top):
        b = q1 if o == 1 else two if o == 2 else many * (1 - q) ** (o - 3)
        if b <= thr:
            return o
    return top


# largest cut-off of a group: its largest copy number O_thr - 1 is 1, 16, 17, 20, 21, 24, 31, 32, 48, 63,
# i.e. 0, 1, 4, 5, 8 and 15 mod 16, where the profile kernel's last 16-copy chunk of the group ends
CUT_TARGETS = (2, 17, 18, 21, 22, 25, 32, 33, 49, 64)
CUT_RESIDUES = {0, 1, 4, 5, 8, 15}
_Q_GRID = np.round(np.linspace(0.02, 0.98, 961), 6)


@functools.lru_cache(maxsize=None)
def _cut_points(top):
    """One (coverage, error rate) group per target cut-off, 12 points each: one at the target (q1 = q2 =
    0.5, q in the middle of the q that give it), 11 with smaller cut-offs; the groups of target 2 have
    q1 = 1 (no second copy: b(2) = 0).  Returns (points, largest cut-off of each group)."""
    rng = np.random.default_rng(5)
    cut_of_q = np.array([_cutoff(0.5, 0.5, q, top) for q in _Q_GRID])
    rows, cuts = [], []
    for g, target in enumerate(CUT_TARGETS):
        c, e = 15.0 + 2.5 * g, (0.01, 0.02)[g % 2]
        if target == 2:
            group = [[c, e, 1.0, q2, q] for q2, q in rng.uniform(0, 1, (12, 2))]
        else:
            qs = _Q_GRID[cut_of_q == target]
            assert len(qs), target
            smaller = _Q_GRID[cut_of_q < target]
            group = [[c, e, 0.5, 0.5, qs[len(qs) // 2]]] + [[c, e, 0.5, 0.5, q] for q in rng.choice(smaller, 11)]
        rng.shuffle(group)
        rows += group
        cuts.append(max(_cutoff(p[2], p[3], p[4], top) for p in group))
    assert cuts == list(CUT_TARGETS)
    return np.ascontiguousarray(rows), tuple(cuts)


def test_cut_points_end_the_last_chunk_at_every_residue():
    for top in (max(_histogram('cfg2_repeats')[0]), max(_histogram('cfg3_repeats_dense1000')[0])):
        _, cuts = _cut_points(top)
        assert {(c - 1) % 16 for c in cuts} >= CUT_RESIDUES


def _nan_first_points(name):
    """A group of 16 points with NaN coverage first, then the small lattice as explicit points: K1
    writes NaN profiles for that group, which a later group must not read."""
    axes = _lattice_axes(name, True)
    rng = np.random.default_rng(9)
    bad = np.column_stack([np.full(16, np.nan), np.full(16, 0.02), rng.uniform(.3, 1, 16), rng.uniform(0, 1, 16),
                           rng.uniform(.05, 1, 16)])
    return np.ascontiguousarray(np.vstack([bad, _grid(axes)]))


def _basic_axes():
    return (np.geomspace(5.0, 60.0, 12), np.geomspace(1e-3, 0.3, 8))


# ---- part A: poisoned = clean ---------------------------------------------------------------------
PATHS = {'auto': 0, 'per_point': 1, 'gemm': 3, 'prefix': 4, 'term_by_term': 5}
# histogram -> (k, r).  Rows per group NA: e05 1, cfg2 2, dense400 4, cfg3 8, trim120 1 with a tail of 175.
# cfg4 (k = 31, r = 150) runs the prefix kernel's 8 x 4 geometry in several passes.  sparse700 has a tail
# and a line of sums, whose second half only the GEMM reads (its mass sums whole lines).
HISTS = {
    'e05_repeats': (21, 100), 'cfg2_repeats': (21, 100), 'dense400': (21, 100), 'cfg3_repeats_dense1000': (21, 100),
    'cfg2_repeats_trim120': (21, 100), 'cfg4_repeats_k31': (31, 150), 'sparse700': (21, 100)}


def _cases():
    """(histogram, k, r, S, kind, path, points, environment)"""
    out = []
    for name, (k, r) in HISTS.items():
        for path in PATHS:
            if name == 'sparse700' and path == 'term_by_term':
                continue
            out.append((name, k, r, 8, 'repeats', path, 'small' if path == 'term_by_term' else 'lattice', ()))
    out += [('e05_basic', 21, 100, 8, 'basic', 'per_point', 'basic', ()),
            ('e05_basic', 21, 100, 8, 'basic', 'auto', 'basic', ())]
    # S = 1, 8, 12, 17: 8, 4, 2, 1 copies per tile of the profile kernel; 32: the last S of the factored
    # path; 33: the per-point fallback.  S <= k + 1.
    for name in ('cfg2_repeats', 'cfg3_repeats_dense1000'):
        for S in (1, 12, 17, 32, 33):
            for path in ('gemm', 'prefix', 'per_point'):
                out.append((name, max(21, S - 1), 100, S, 'repeats', path, 'lattice', ()))
        for S in (1, 8, 12, 17, 32):
            for path in ('gemm', 'prefix') + (('auto',) if S == 8 else ()):
                out.append((name, max(21, S - 1), 100, S, 'repeats', path, 'cuts', ()))
    for path in ('gemm', 'prefix', 'per_point'):
        out.append(('cfg2_repeats', 21, 100, 8, 'repeats', path, 'nan_first', ()))
    for path in ('gemm', 'prefix'):
        out.append(('cfg3_repeats_dense1000', 21, 100, 8, 'repeats', path, 'lattice', (('COVEST_B200_PROFILE_MIB', '1'),)))
        out.append(('cfg3_repeats_dense1000', 21, 100, 8, 'repeats', path, 'nan_first', (('COVEST_B200_PROFILE_MIB', '1'),)))
    for path in ('gemm', 'prefix'):
        out.append(('cfg2_repeats', 21, 100, 8, 'repeats', path, 'lattice', (('COVEST_B200_ROWS', 'full'),)))
    return out


CASES = _cases()


def _case_id(case):
    name, k, r, S, kind, path, pts, env = case
    return '%s-S%d-k%d-%s-%s%s' % (name, S, k, path, pts, ''.join('-%s=%s' % (a[12:].lower(), b) for a, b in env))


@functools.lru_cache(maxsize=None)
def _oracle(kind, name, k, r, S):
    hist, tail = _histogram(name)
    return orc.Model(kind, k, r, hist, tail, max_error=S)


def _points(name, pts_kind):
    """(lattice axes or None, the explicit points of the case)."""
    if pts_kind == 'basic':
        return _basic_axes(), _grid(_basic_axes())
    if pts_kind in ('lattice', 'small'):
        axes = test_gpu_rows.axes() if name == 'sparse700' else _lattice_axes(name, pts_kind == 'small')
        return axes, _grid(axes)
    if pts_kind == 'cuts':
        return None, _cut_points(max(_histogram(name)[0]))[0]
    return None, _nan_first_points(name)


def _evaluate(ctx, name, path, pts_kind):
    """Values of the case's points: lattice_eval (when the points are a lattice), then loglik of the
    explicit points, one array."""
    ctx.set_path(PATHS[path])
    axes, pts = _points(name, pts_kind)
    by_axes = [] if axes is None else list(ctx.lattice_eval(axes)[0])
    return np.concatenate([np.array(by_axes, dtype=np.float64), ctx.loglik(pts)])


@functools.lru_cache(maxsize=None)
def _oracle_sample(kind, name, k, r, S, pts_kind):
    """Up to 64 points of the case with finite parameters, inside the reference's numeric domain, and
    the oracle's values there; `at` indexes the explicit points."""
    m = _oracle(kind, name, k, r, S)
    pts = _points(name, pts_kind)[1]
    ok = np.flatnonzero(np.isfinite(pts).all(axis=1))
    at = np.sort(np.random.default_rng(3).choice(ok, min(64, len(ok)), replace=False))
    want = m.loglik_batch(pts[at], threads=8)
    inside = ~(np.isnan(want) | np.isposinf(want))
    return at[inside], want[inside]


@pytest.mark.parametrize('case', CASES, ids=_case_id)
def test_poisoned_scratch_gives_the_clean_values(case):
    name, k, r, S, kind, path, pts_kind, env = case
    m = _oracle(kind, name, k, r, S)
    pts = _points(name, pts_kind)[1]
    with _context(m, None, env) as ctx:
        clean = _evaluate(ctx, name, path, pts_kind)
        info = ctx.last_path_info()
    if S <= 32 and path in ('gemm', 'prefix'):
        assert info['kernel'] == ('cvf_gemm_kernel' if path == 'gemm' else 'cvf_prefix_kernel')
    if path == 'auto' and kind == 'repeats' and len(pts) >= 2048:
        assert info['path'] == 'factored'
    for poison in POISONS:
        with _context(m, poison, env) as ctx:
            got = _evaluate(ctx, name, path, pts_kind)
        _assert_same(got, clean, (path, poison))
    # anchored to the reference: a sample of the explicit points' values
    at, want = _oracle_sample(kind, name, k, r, S, pts_kind)
    assert len(at) >= 8
    ll = clean[len(clean) - len(pts):][at]
    _assert_close(ll, want, _gate(m, pts[at], want, LL_RTOL), (path, 'oracle'))
    if pts_kind == 'nan_first':
        assert np.isnan(clean[:16]).all() and not np.isnan(clean[16:]).any()


# ---- part B: every output element written, nothing around it ----------------------------------------
SENTINEL = 0x7FF4DEADBEEF0001  # a NaN payload no arithmetic produces
GUARD_BITS = 0x7FF4DEADBEEF0002
GUARD = 64


class Framed:
    """n doubles pre-filled with SENTINEL, with GUARD elements of GUARD_BITS before and after; `ptr` is
    the address of the first of the n (host memory, or device memory when `device`)."""

    def __init__(self, n, device):
        import torch
        self.n = int(n)
        bits = np.full(self.n + 2 * GUARD, GUARD_BITS, dtype=np.uint64)
        bits[GUARD:GUARD + self.n] = SENTINEL
        self.device = device
        if device:
            self.buf = torch.from_numpy(bits.view(np.int64)).cuda()
            self.ptr = ctypes.c_void_p(self.buf.data_ptr() + 8 * GUARD)
        else:
            self.buf = bits.view(np.float64)
            self.ptr = ctypes.c_void_p(self.buf.ctypes.data + 8 * GUARD)

    def values(self, poison=None):
        """The n values, after checking that each was written and that the guards are intact."""
        import torch
        if self.device:
            torch.cuda.synchronize()
            bits = self.buf.cpu().numpy().view(np.uint64)
        else:
            bits = self.buf.view(np.uint64)
        guards = np.concatenate([bits[:GUARD], bits[GUARD + self.n:]])
        assert np.all(guards == GUARD_BITS), 'a guard element was overwritten'
        inner = bits[GUARD:GUARD + self.n]
        left = np.flatnonzero(inner == SENTINEL)
        assert not len(left), '%d of %d elements were never written, first at %s' % (len(left), self.n, left[:8].tolist())
        if poison:
            stale = np.flatnonzero(inner == POISON_BITS[poison])
            assert not len(stale), '%d of %d elements hold the poison, first at %s' % (len(stale), self.n, stale[:8].tolist())
        return inner.view(np.float64).copy()


def _dev(a, device):
    """`a` as float64 in host memory, or in device memory when `device` (the caller keeps the tensor
    alive for as long as the library may read it)."""
    if not device:
        return np.ascontiguousarray(a, dtype=np.float64)
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _p(a):
    return ctypes.c_void_p(a.data_ptr() if hasattr(a, 'data_ptr') else a.ctypes.data)


def _ok(ctx, rc):
    assert rc == 0, ctx._lib.cvb_last_error(ctx._ctx).decode()


def _check_rows(rows, ll_all, n, K, n_param):
    """Rows of a top-K: best first, (-inf, NaN...) beyond the batch (include/covest_b200.h)."""
    rows = rows.reshape(K, 1 + n_param)
    real = min(n, K)
    if n:
        best = np.sort(np.where(np.isnan(ll_all), -np.inf, ll_all))[::-1][:real]
        assert np.array_equal(np.where(np.isnan(rows[:real, 0]), -np.inf, rows[:real, 0]), best)
    assert np.all(rows[real:, 0] == -np.inf) and np.isnan(rows[real:, 1:]).all()


@pytest.mark.parametrize('device', [False, True], ids=['host', 'device'])
@pytest.mark.parametrize('poison', POISONS)
def test_every_output_element_is_written(poison, device):
    m = _oracle('repeats', 'cfg2_repeats', 21, 100, 8)
    mb = _oracle('basic', 'e05_basic', 21, 100, 8)
    big = _grid(_lattice_axes('cfg2_repeats', False))            # 2112 points: factored under auto
    with _context(m, poison) as ctx, _context(mb, poison) as ctxb:
        lib, c = ctx._lib, ctx._ctx
        # loglik_batch: the factored path, the per-point kernel, a batch below the automatic threshold
        for path, pts in ((0, big), (1, big), (0, big[:37])):
            ctx.set_path(path)
            out = Framed(len(pts), device)
            src = _dev(pts, device)
            _ok(ctx, lib.cvb_loglik_batch(c, len(pts), _p(src), out.ptr, None))
            assert not np.isnan(out.values(poison)).any()
        # probs_batch on both models, with and without the log-likelihoods, clipped and not
        for cx, mm, pts in ((ctx, m, big[::7]), (ctxb, mb, _grid(_basic_axes())[::3])):
            for clip in (0, 1):
                for with_ll in (False, True):
                    outp = Framed(len(pts) * len(mm.bin_j), device)
                    outl = Framed(len(pts), device) if with_ll else None
                    src = _dev(pts, device)
                    _ok(cx, cx._lib.cvb_probs_batch(cx._ctx, len(pts), _p(src), clip, outp.ptr,
                                                    outl.ptr if outl else None, None))
                    outp.values(poison)
                    if outl:
                        outl.values(poison)
        # lattice_eval: slices of the lattice, with and without rows
        axes = _lattice_axes('cfg2_repeats', False)
        lens = np.array([len(a) for a in axes], dtype=np.int32)
        vals = np.concatenate(axes)
        total = int(np.prod(lens))
        M = int(np.prod(lens[2:]))
        whole = np.array(ctx.lattice_eval(axes)[0])
        for first, stride, block, count, K in ((0, 1, 1, total, 0), (5, 3, 1, 300, 40), (1, 2, 7, 250, 0),
                                               (0, 1, M, 2 * M, 10), (2, 1, M, M, 3 * M), (0, 1, 1, 0, 5),
                                               (17, 1, 1, 20, 64)):
            for path in (0, 1):
                ctx.set_path(path)
                out = Framed(count, device)
                rows = Framed(K * 6, device) if K else None
                _ok(ctx, lib.cvb_lattice_eval(c, lens.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                              vals.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), first, stride,
                                              block, count, out.ptr, K, rows.ptr if rows else None, None))
                got = out.values(poison)
                i = np.arange(count)
                idx = (first + (i // block) * stride) * block + i % block
                assert np.array_equal(np.isnan(got), np.isnan(whole[idx]))
                if rows:
                    _check_rows(rows.values(poison), got, count, K, 5)
        # loglik_topk and topk: small batches, radix selection (n >= 32768, K <= 1024), the sort (K > 1024), K > n
        ctx.set_path(0)
        rng = np.random.default_rng(11)
        many = np.tile(big, (16, 1))[:33000].copy()
        many[:, 0] *= rng.uniform(0.9, 1.1, len(many))
        for pts, K in ((big[:300], 20), (big[:300], 400), (many, 64), (many, 1500)):
            for want_ll in (True, False):
                out = Framed(len(pts), device) if want_ll else None
                rows = Framed(K * 6, device)
                src = _dev(pts, device)
                _ok(ctx, lib.cvb_loglik_topk(c, len(pts), _p(src), out.ptr if out else None, K,
                                             rows.ptr, None))
                r = rows.values(poison)
                if out:
                    _check_rows(r, out.values(poison), len(pts), K, 5)
        for n, K in ((1000, 10), (1000, 1001), (40000, 100), (40000, 2000), (0, 3)):
            llv = rng.normal(-1e5, 10, n)
            llv[::97] = -np.inf
            llv[5::101] = np.nan
            pts = rng.uniform(0, 1, (n, 5))
            rows = Framed(K * 6, device)
            src_ll, src_pts = _dev(llv if n else np.zeros(1), device), _dev(pts if n else np.zeros(5), device)
            _ok(ctx, lib.cvb_topk(c, n, _p(src_ll), _p(src_pts), K, rows.ptr, None))
            _check_rows(rows.values(poison), llv, n, K, 5)
    if device:  # merge_rows takes device buffers only
        import torch
        for n_rows, k_best in ((100, 10), (100, 150), (2048, 2048), (0, 4)):
            src = np.column_stack([np.random.default_rng(n_rows).normal(0, 1, n_rows), np.zeros((n_rows, 5))])
            rows = _dev(src if n_rows else np.zeros((1, 6)), True)
            out = Framed(k_best * 6, True)
            assert ctx._lib.cvb_merge_rows(_p(rows), n_rows, 6, k_best, out.ptr, None) == 0
            torch.cuda.synchronize()
            _check_rows(out.values(), src[:, 0], n_rows, k_best, 5)


# ---- part C: one poisoned context, a sequence of calls ----------------------------------------------
def _sequence():
    """Calls that grow, shrink and change the workspaces: a large lattice, a small one, explicit points
    of another grouping, a lattice whose q axes differ in one value (the template cache key), the
    per-point kernel and probability staging (probs, clip = 0), the first lattice again."""
    big = _lattice_axes('cfg3_repeats_dense1000', False)
    small = _lattice_axes('cfg3_repeats_dense1000', True)
    shifted = big[:4] + (np.where(big[4] == 0.2, 0.25, big[4]),)
    cuts = _cut_points(max(_histogram('cfg3_repeats_dense1000')[0]))[0]
    return [('lattice', big), ('lattice', small), ('loglik', cuts), ('lattice', shifted),
            ('probs', cuts[::5]), ('lattice', big)]


def _call(ctx, what, arg):
    if what == 'lattice':
        ll, rows = ctx.lattice_eval(arg, k_best=8)
        return np.concatenate([np.array(ll), rows.ravel()])
    if what == 'loglik':
        return np.array(ctx.loglik(arg))
    p, ll = ctx.probs(arg, clip=False, with_loglik=True)
    return np.concatenate([p.ravel(), ll])


@pytest.mark.parametrize('path', ['auto', 'gemm', 'prefix'])
@pytest.mark.parametrize('poison', POISONS)
def test_a_sequence_of_calls_in_one_poisoned_context(poison, path):
    m = _oracle('repeats', 'cfg3_repeats_dense1000', 21, 100, 8)
    seq = _sequence()
    with _context(m, poison) as ctx:
        ctx.set_path(PATHS[path])
        got = [_call(ctx, what, arg) for what, arg in seq]
    for i, (what, arg) in enumerate(seq):
        with _context(m) as fresh:
            fresh.set_path(PATHS[path])
            _assert_same(got[i], _call(fresh, what, arg), (i, what, poison))


def test_an_unknown_poison_is_an_error():
    from covest_b200.engine import DeviceError
    m = _oracle('repeats', 'e05_repeats', 21, 100, 8)
    with pytest.raises(DeviceError, match='COVEST_B200_POISON'):
        with _context(m, 'zero'):
            pass
