"""The host side of the k-mer counter (covest_b200/kmers.py) and the references the device tests use:
the block reader against a naive per-record parse at every block size, the numpy canonical counter
against a dict of strings, the read simulator, and argument checks.  No GPU needed."""
import os

import numpy as np
import pytest

from covest_b200 import kmers
from tests import kmer_helpers as kh


def _records(rng, n, lo, hi, alphabet=b'ACGT'):
    a = np.frombuffer(alphabet, dtype=np.uint8)
    return [bytes(rng.choice(a, int(rng.integers(lo, hi + 1))).tolist()) for _ in range(n)]


def _stream(path, block_bytes):
    blocks = list(kmers.read_blocks(path, block_bytes))
    seq = b''.join(bytes(b.seq) for b in blocks)
    return seq, sum(b.reads for b in blocks), sum(b.bases for b in blocks)


READ_CASES = {
    'fasta': dict(kind='fasta'),
    'fasta_wrapped': dict(kind='fasta', width=7),
    'fasta_crlf_wrapped': dict(kind='fasta', width=5, crlf=True),
    'fasta_gz': dict(kind='fasta', width=11, gz=True),
    'fastq': dict(kind='fastq'),
    'fastq_crlf': dict(kind='fastq', crlf=True),
    'fastq_gz': dict(kind='fastq', gz=True),
}


@pytest.mark.parametrize('name', sorted(READ_CASES))
def test_reader_equals_naive_parse_at_every_block_size(tmp_path, name):
    case = dict(READ_CASES[name])
    kind = case.pop('kind')
    rng = np.random.default_rng(len(name))
    recs = _records(rng, 9, 0, 23, b'ACGTacgtNNRY')  # lowercase, N, IUPAC codes, empty records, short reads
    recs[3] = b''
    recs[5] = b'NNNNNNNN'
    path = str(tmp_path / ('r.' + kind + ('.gz' if case.get('gz') else '')))
    (kh.write_fasta if kind == 'fasta' else kh.write_fastq)(path, recs, **case)
    want = kh.naive_compact(path)
    assert want == b''.join(kh.SEP + r for r in recs)
    size = os.path.getsize(path) if not case.get('gz') else 400
    for bs in list(range(1, size + 2)) + [1 << 20]:
        got, reads, bases = _stream(path, bs)
        assert got == want, bs
        assert reads == len(recs) and bases == sum(map(len, recs)), bs


def test_reader_skips_blank_lines_and_reads_many_records(tmp_path):
    rng = np.random.default_rng(3)
    recs = _records(rng, 500, 1, 150)
    path = str(tmp_path / 'big.fa')
    kh.write_fasta(path, recs, width=60)
    with open(path, 'ab') as f:
        f.write(b'\n\n')
    for bs in (64, 1000, 4099, 1 << 20):
        assert _stream(path, bs)[0] == b''.join(kh.SEP + r for r in recs)


def test_malformed_fastq_raises(tmp_path):
    path = tmp_path / 'bad.fq'
    path.write_bytes(b'@r1\nACGT\n+\nIIII\n@r2\nACGT\nIIII\n+\n')
    for bs in (3, 1 << 20):
        with pytest.raises(ValueError, match=r'line 3 of record 2'):
            list(kmers.read_blocks(str(path), bs))
    path.write_bytes(b'@r1\nACGT\n+\nIIII\n@r2\nACGT\n')
    with pytest.raises(ValueError, match='incomplete'):
        list(kmers.read_blocks(str(path)))
    path.write_bytes(b'ACGT\n')
    with pytest.raises(ValueError, match='neither FASTA'):
        list(kmers.read_blocks(str(path)))


@pytest.mark.parametrize('k', range(1, 32))
def test_numpy_counter_equals_dict_counter(k):
    rng = np.random.default_rng(k)
    stream = b''.join(kh.SEP + r for r in _records(rng, 12, 0, 90, b'ACGTacgtN'))
    if k % 2 == 0:  # palindromic k-mers: a k-mer equal to its own reverse complement counts once per window
        half = bytes(rng.choice(np.frombuffer(b'ACGT', dtype=np.uint8), k // 2).tolist())
        pal = half + half.translate(bytes.maketrans(b'ACGT', b'TGCA'))[::-1]
        stream += kh.SEP + pal * 3 + kh.SEP + pal
    want = kh.dict_counts(stream, k)
    keys, counts = kh.numpy_counts(stream, k)
    assert {int(a): int(b) for a, b in zip(keys, counts)} == {kh.pack(s): c for s, c in want.items()}
    assert sorted(want.values()) == sorted(counts.tolist())


def test_partition_of_keys_is_a_split():
    keys = np.arange(100000, dtype=np.uint64) * np.uint64(2654435761)
    for n in (1, 2, 3, 8):
        p = kh.part_of(keys, n)
        assert p.max() < n
        if n > 1:
            assert np.all(np.bincount(p.astype(np.int64), minlength=n) > 100000 / n * 0.9)


def test_simulator_is_deterministic():
    a = kh.simulate(5000, 100, 10, 0.01, seed=7, repeats=((300, 4),))
    b = kh.simulate(5000, 100, 10, 0.01, seed=7, repeats=((300, 4),))
    c = kh.simulate(5000, 100, 10, 0.01, seed=8, repeats=((300, 4),))
    assert a == b and a != c
    genome, reads = a
    assert len(genome) == 5000 and len(reads) == 500 and all(len(r) == 100 for r in reads)
    assert sum(a != b for r, s in zip(reads, kh.simulate(5000, 100, 10, 0.0, seed=7, repeats=((300, 4),))[1])
               for a, b in zip(r, s)) in range(300, 700)  # ~1% of 50000 bases substituted
    # error-free reads come from the genome on either strand
    genome, clean = kh.simulate(5000, 100, 10, 0.0, seed=7)
    rc = genome.translate(bytes.maketrans(b'ACGT', b'TGCA'))[::-1]
    assert all(r in genome or r in rc for r in clean)
    assert any(r not in genome for r in clean) and any(r in genome for r in clean)


def test_validation(tmp_path):
    for bad in (0, 32, -1, 1.5, True, '21'):
        with pytest.raises(ValueError):
            kmers.check_k(bad)
    assert kmers.check_k(31) == 31
    for bad in (0, -1, float('nan'), float('inf'), 'x', 1e-9):
        with pytest.raises(ValueError):
            kmers.capacity_for_gib(bad)
    assert kmers.capacity_for_gib(1) == 1 << 26
    assert kmers.capacity_for_gib(1.5) == 1 << 26
    with pytest.raises(FileNotFoundError):
        kmers.count_kmers([str(tmp_path / 'missing.fq')], 21)
    with pytest.raises(ValueError):
        kmers.count_kmers([str(tmp_path / 'missing.fq')], 40)
    reads = tmp_path / 'r.fa'
    reads.write_bytes(b'>r\nACGT\n')
    for argv in ([str(tmp_path / 'missing.fq'), '-k', '21', '-o', 'x'],
                 [str(reads), '-k', '32', '-o', 'x'],
                 [str(reads), '-k', '21', '-o', 'x', '--table-gib', '0'],
                 [str(reads), '-k', '21', '-o', 'x', '--table-gib', 'nan']):
        with pytest.raises(SystemExit) as err:
            kmers.run(argv)
        assert err.value.code == 2


def test_default_capacity(tmp_path):
    p = tmp_path / 'r.fa'
    p.write_bytes(b'A' * 100000)
    free = 1 << 40
    assert kmers.default_capacity([str(p)], 1, free) == 1 << 17   # 125000 slots -> 2^17
    assert kmers.default_capacity([str(p)], 4, free) == 1 << 15   # a quarter per part
    assert kmers.default_capacity([str(p)], 1, 1 << 20) == 1 << 15  # half the free memory, 16 B a slot
    g = tmp_path / 'r.fa.gz'
    g.write_bytes(b'')
    assert kmers.default_capacity([str(g)], 1, 1 << 30) == 1 << 25
    tiny = tmp_path / 't.fa'
    tiny.write_bytes(b'>r\nAC\n')
    assert kmers.default_capacity([str(tiny)], 1, free) == kmers.MIN_CAPACITY
