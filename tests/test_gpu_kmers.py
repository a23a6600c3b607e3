"""The device k-mer counter (csrc/kmers.cu, cvb_kmer_*, covest_b200/kmers.py) against the numpy canonical
counter of tests/kmer_helpers.py, and `covest` on the histogram of simulated reads.  Needs a B200."""
import ctypes
import io
import os
import subprocess
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest
import yaml

from covest_b200 import _capi, data, kmers
from tests import kmer_helpers as kh

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mixed_stream(seed, poly_a=3_000_000):
    """Reads of length < k, = k and long, N runs, lowercase, IUPAC codes, and a poly-A block (one slot
    takes millions of adds), as records of a compacted block."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b'ACGT', dtype=np.uint8)
    recs = []
    for n in list(range(0, 40)) + [1000] * 50 + [20000] * 5:
        r = rng.choice(acgt, n)
        if n > 100:
            r[rng.integers(0, n, n // 200)] = ord('N')
            low = rng.random(n) < 0.1
            r[low] |= 0x20
            r[rng.integers(0, n, 3)] = ord('R')
            r[50:70] = ord('N')
        recs.append(r.tobytes())
    recs.append(b'A' * poly_a)
    recs.append(b'acgtNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNNacgt' * 100)
    return recs


def _join(recs):
    return b''.join(kh.SEP + r for r in recs)


def _oracle(stream, k):
    keys, counts = kh.numpy_counts(stream, k)
    stats = [len(keys), int(counts.sum()), int(counts.max()) if len(counts) else 0, 0]
    return kh.hist_of_counts(counts), stats, keys, counts


def _hist_dict(dense):
    return {int(j) + 1: int(dense[j]) for j in np.flatnonzero(dense)}


def _stream_parts(recs, n_parts):
    cut = np.linspace(0, len(recs), n_parts + 1).astype(int)
    return [_join(recs[a:b]) for a, b in zip(cut[:-1], cut[1:])]


@pytest.mark.parametrize('k', [1, 2, 11, 16, 21, 31])
def test_histogram_and_stats_equal_the_oracle(k):
    import torch
    recs = _mixed_stream(k)
    stream = _join(recs)
    want_hist, want_stats, _, counts = _oracle(stream, k)
    cap = 1 << 20
    # host buffer, one call
    with kmers.KmerCounter(k, cap) as kc:
        kc.count(np.frombuffer(stream, dtype=np.uint8))
        st = kc.stats()
        assert st.tolist() == want_stats
        assert _hist_dict(kc.histogram(st[2])) == want_hist
        # fewer bins: the last one takes every larger count
        nb = 5
        dense = kc.histogram(nb)
        assert dense[:nb - 1].tolist() == [want_hist.get(j, 0) for j in range(1, nb)]
        assert int(dense[-1]) == int(np.sum(counts >= nb))
    # device buffer on an explicit stream, cut at read boundaries into parts
    s = torch.cuda.Stream()
    with kmers.KmerCounter(k, cap) as kc:
        parts = [torch.frombuffer(bytearray(p), dtype=torch.uint8).cuda() for p in _stream_parts(recs, 7)]
        torch.cuda.synchronize()
        for t in parts:  # kept alive until the stream is done with them
            kc.count(t, stream=s)
        out = torch.full((4,), -7, dtype=torch.int64, device='cuda')
        torch.cuda.synchronize()
        kc.stats(out=out, stream=s)
        s.synchronize()
        assert out.cpu().tolist() == want_stats
        dh = torch.full((want_stats[2],), -7, dtype=torch.int64, device='cuda')
        torch.cuda.synchronize()
        kc.histogram(want_stats[2], out=dh, stream=s)
        s.synchronize()
        assert _hist_dict(dh.cpu().numpy()) == want_hist
    # host buffers cut into parts: bytes, and a CPU torch tensor
    with kmers.KmerCounter(k, cap) as kc:
        for i, part in enumerate(_stream_parts(recs, 3)):
            kc.count(torch.frombuffer(bytearray(part), dtype=torch.uint8) if i == 1 else part)
        assert kc.stats().tolist() == want_stats


@pytest.mark.parametrize('k', [5, 21, 31])
def test_host_staging_parts_equal_one_device_call(k):
    """A host buffer of ~150 MB goes through the pinned staging in three parts, each repeating the k - 1
    bytes before it: the table must equal that of the same bytes counted from device memory in one call."""
    import torch
    rng = np.random.default_rng(k)
    n = 150_000_000
    seq = np.frombuffer(b'ACGTACGTACGTACGTacgtN', dtype=np.uint8)[rng.integers(0, 21, n, dtype=np.uint8)]
    with kmers.KmerCounter(k, 1 << 28) as a, kmers.KmerCounter(k, 1 << 28) as b:
        a.count(seq)
        b.count(torch.from_numpy(seq).cuda())
        torch.cuda.synchronize()
        sa, sb = a.stats(), b.stats()
        assert sa.tolist() == sb.tolist()
        valid = np.concatenate(([0], np.cumsum((seq | 0x20) == ord('n'))))  # windows without an N
        assert sa[1] == int(np.sum(valid[k:] - valid[:-k] == 0))
        assert np.array_equal(a.histogram(sa[2]), b.histogram(sb[2]))


def test_clear_and_reuse_equal_a_fresh_table():
    recs = _mixed_stream(5, poly_a=1000)
    one, two = _join(recs[:60]), _join(recs[60:])
    with kmers.KmerCounter(21, 1 << 18) as kc, kmers.KmerCounter(21, 1 << 18) as fresh:
        kc.count(one)
        kc.histogram(kc.stats()[2])
        kc.clear()
        assert kc.stats().tolist() == [0, 0, 0, 0]
        kc.count(two)
        fresh.count(two)
        assert kc.stats().tolist() == fresh.stats().tolist()
        m = int(fresh.stats()[2])
        assert np.array_equal(kc.histogram(m), fresh.histogram(m))


@pytest.mark.parametrize('k', [11, 21])
def test_parts_sum_to_the_whole(k):
    recs = _mixed_stream(100 + k, poly_a=100000)
    stream = _join(recs)
    want_hist, want_stats, keys, counts = _oracle(stream, k)
    for n_parts in (1, 2, 3, 8):
        part = kh.part_of(keys, n_parts)
        total = np.zeros(want_stats[2], dtype=np.int64)
        distinct = 0
        for p in range(n_parts):
            with kmers.KmerCounter(k, 1 << 18, part=p, n_parts=n_parts) as kc:
                kc.count(stream)
                st = kc.stats()
                mine = part == p
                assert st[0] == int(mine.sum()) and st[1] == int(counts[mine].sum())
                dense = kc.histogram(want_stats[2])
                assert _hist_dict(dense) == kh.hist_of_counts(counts[mine])
                total += dense
                distinct += int(st[0])
        assert _hist_dict(total) == want_hist and distinct == want_stats[0]


def _distinct_stream(n_kmers, k, seed):
    rng = np.random.default_rng(seed)
    s = np.frombuffer(b'ACGT', dtype=np.uint8)[rng.integers(0, 4, n_kmers + k - 1)].tobytes()
    _, counts = kh.numpy_counts(s, k)
    assert len(counts) == n_kmers and counts.max() == 1  # every canonical k-mer once
    return s


def test_overflow_is_an_error_with_the_dropped_count(tmp_path):
    cap = 1024
    limit = cap - cap // 8
    lib = _capi.load()
    # just under the limit: every k-mer fits
    s = _distinct_stream(limit, 31, 1)
    with kmers.KmerCounter(31, cap) as kc:
        kc.count(s)
        assert kc.stats().tolist() == [limit, limit, 1, 0]
        assert _hist_dict(kc.histogram(1)) == {1: limit}
    # over it: cvb_kmer_histogram returns CVB_ENOMEM and names the count
    n = 3000
    s = _distinct_stream(n, 31, 2)
    with kmers.KmerCounter(31, cap) as kc:
        kc.count(s)
        distinct, total, mx, dropped = kc.stats().tolist()
        assert distinct <= limit and dropped == n - distinct and dropped >= n - limit and total == distinct
        out = np.full(4, 123, dtype=np.int64)
        rc = lib.cvb_kmer_histogram(kc._t, 4, out.ctypes.data_as(ctypes.c_void_p), None)
        assert rc == -3
        assert ('%d k-mers were dropped' % dropped) in lib.cvb_kmer_last_error(kc._t).decode()
        assert out.tolist() == [123] * 4  # left as it was
        with pytest.raises(kmers.KmerTableFull) as err:
            kc.histogram(4)
        assert err.value.dropped == dropped
    # the CLI exits with the count and what to do about it
    reads = tmp_path / 'r.fa'
    kh.write_fasta(str(reads), [s])
    gib = cap * kmers.SLOT_BYTES / float(1 << 30)
    with pytest.raises(SystemExit) as err:
        kmers.run([str(reads), '-k', '31', '-o', str(tmp_path / 'x.hist'), '--table-gib', repr(gib)])
    msg = str(err.value.code)
    assert 'k-mers did not fit' in msg and '--table-gib' in msg and 'more GPUs' in msg
    assert int(msg.split()[1]) >= n - limit
    assert not (tmp_path / 'x.hist').exists()


def test_every_output_is_written():
    """As the poison tests of the likelihood calls: outputs pre-filled with a sentinel and framed by guards;
    every element written, no guard changed -- host and device buffers."""
    import torch
    lib = _capi.load()
    stream = _join(_mixed_stream(9, poly_a=5000))
    G, SENT = 64, -0x5A5A5A5A5A5A5A5A
    with kmers.KmerCounter(21, 1 << 18) as kc:
        kc.count(stream)
        _, _, mx, _ = kc.stats().tolist()
        for n_bins in (1, 2, mx, mx + 3, 5000):
            for dev in (False, True):
                buf = np.full(n_bins + 2 * G, SENT, dtype=np.int64)
                if dev:
                    tb = torch.from_numpy(buf).cuda()
                    torch.cuda.synchronize()
                    ptr = ctypes.c_void_p(tb.data_ptr() + 8 * G)
                else:
                    ptr = ctypes.c_void_p(buf.ctypes.data + 8 * G)
                assert lib.cvb_kmer_histogram(kc._t, n_bins, ptr, None) == 0
                if dev:
                    torch.cuda.synchronize()
                    buf = tb.cpu().numpy()
                assert np.all(buf[:G] == SENT) and np.all(buf[G + n_bins:] == SENT)
                assert np.all(buf[G:G + n_bins] != SENT) and np.all(buf[G:G + n_bins] >= 0)
        for dev in (False, True):
            buf = np.full(4 + 2 * G, SENT, dtype=np.int64)
            if dev:
                tb = torch.from_numpy(buf).cuda()
                torch.cuda.synchronize()
                ptr = ctypes.c_void_p(tb.data_ptr() + 8 * G)
            else:
                ptr = ctypes.c_void_p(buf.ctypes.data + 8 * G)
            assert lib.cvb_kmer_stats(kc._t, ptr, None) == 0
            if dev:
                torch.cuda.synchronize()
                buf = tb.cpu().numpy()
            assert np.all(buf[:G] == SENT) and np.all(buf[G + 4:] == SENT)
            assert buf[G:G + 4].tolist() == kc.stats().tolist()


def test_bad_arguments_are_refused():
    lib = _capi.load()
    t = ctypes.c_void_p()
    for args in ((0, 1024, 0, 1), (32, 1024, 0, 1), (21, 1000, 0, 1), (21, 0, 0, 1), (21, 1024, 2, 2),
                 (21, 1024, -1, 2), (21, 1024, 0, 0)):
        assert lib.cvb_kmer_table_create(args[0], args[1], args[2], args[3], 0, ctypes.byref(t)) == -1, args
        assert not t.value
    with pytest.raises(ValueError):
        kmers.KmerCounter(21, 1000)


# ---- end to end: simulated reads -> device histogram -> covest ----------------------------------------
GENOME, READ_LEN, COVERAGE, ERROR, K = 1_000_000, 100, 10, 0.01, 21
# Tolerances from the errors observed on a B200 (DESIGN.md section 11), each with a 5x margin.  Input,
# counting and estimate are deterministic for the seeds below, so the margin covers changes of the
# estimator's numerics, not run-to-run noise.
SIZE_RTOL_BASIC, COV_RTOL_BASIC = 0.005, 0.005     # observed: genome size -0.10 %, coverage +0.10 %
SIZE_RTOL_REPEAT, COV_RTOL_REPEAT = 0.012, 0.012   # observed: genome size +0.24 %, coverage -0.24 %


def _simulated_hist(tmp_path, repeats=(), seed=2024):
    genome, reads = kh.simulate(GENOME, READ_LEN, COVERAGE, ERROR, seed, repeats=repeats)
    fq = tmp_path / 'sim.fq'
    kh.write_fastq(str(fq), reads)
    out = tmp_path / 'sim.hist'
    hist, st = kmers.run([str(fq), '-k', str(K), '-o', str(out)])
    assert st['reads'] == len(reads) and st['bases'] == len(reads) * READ_LEN
    assert st['total'] == len(reads) * (READ_LEN - K + 1)
    h2, meta = data.load_histogram(str(out))
    assert h2 == hist and list(h2) == sorted(h2)
    assert meta['k'] == str(K) and meta['reads'] == str(len(reads)) and float(meta['mean_read_length']) == READ_LEN
    return out


def _covest(path, *extra):
    from covest_b200 import covest as cli
    buf = io.StringIO()
    cwd = os.getcwd()
    os.chdir(os.path.dirname(str(path)))
    try:
        with redirect_stdout(buf):
            cli.run([str(path), '-k', str(K), '-r', str(READ_LEN), '--polish', '--seed', '1'] + list(extra))
    finally:
        os.chdir(cwd)
    return yaml.safe_load(buf.getvalue())


def test_covest_recovers_the_simulated_genome(tmp_path):
    out = _covest(_simulated_hist(tmp_path))
    size_err = out['genome_size'] / GENOME - 1
    cov_err = out['coverage'] / COVERAGE - 1
    print('basic model: genome_size %d (rel. error %+.4f), coverage %.4f (%+.4f), error_rate %.5f' % (
        out['genome_size'], size_err, out['coverage'], cov_err, out['error_rate']))
    assert abs(size_err) <= SIZE_RTOL_BASIC and abs(cov_err) <= COV_RTOL_BASIC


# low-copy repeat families (8.5 % of the genome): 20 of 1000 bases in 2 copies, 20 of 500 in 3, 10 of 300 in 5
REPEATS = ((1000, 2),) * 20 + ((500, 3),) * 20 + ((300, 5),) * 10


def test_covest_repeat_model_on_planted_repeats(tmp_path):
    out = _covest(_simulated_hist(tmp_path, repeats=REPEATS, seed=77), '-m', 'repeat')
    size_err = out['genome_size'] / GENOME - 1
    cov_err = out['coverage'] / COVERAGE - 1
    print('repeats model: genome_size %d (rel. error %+.4f), coverage %.4f (%+.4f), q1 %.3f q2 %.3f q %.3f' % (
        out['genome_size'], size_err, out['coverage'], cov_err, out['q1'], out['q2'], out['q']))
    assert abs(size_err) <= SIZE_RTOL_REPEAT and abs(cov_err) <= COV_RTOL_REPEAT


def test_two_gpus_give_the_histogram_of_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    _, reads = kh.simulate(200_000, READ_LEN, COVERAGE, ERROR, 5)
    fq = tmp_path / 'sim.fq'
    kh.write_fastq(str(fq), reads)
    one = tmp_path / 'one.hist'
    kmers.run([str(fq), '-k', str(K), '-o', str(one)])
    two = tmp_path / 'two.hist'
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
           '--master-addr', '127.0.0.1', '--master-port', '29545', '-m', 'covest_b200.kmers',
           str(fq), '-k', str(K), '-o', str(two)]
    subprocess.run(cmd, check=True, timeout=600, cwd=ROOT, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    assert two.read_text() == one.read_text()
