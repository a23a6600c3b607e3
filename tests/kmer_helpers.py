"""Host references for the k-mer counter (covest_b200/kmers.py, csrc/kmers.cu): a naive per-record
reader, a numpy canonical counter, a plain dict-of-strings counter, the hash partition, and a seeded
read simulator (SURVEY.md section 8(d): uniform genome, reads of length r at coverage c, substitutions
at rate e, random strand, optional planted repeats)."""
import gzip

import numpy as np

SEP = b'\n'
_COMP = bytes.maketrans(b'ACGTacgt', b'TGCAtgca')


# ---- reading -------------------------------------------------------------------------------------
def naive_compact(path):
    """SEP + sequence of every record, read line by line: the stream read_blocks must produce."""
    opener = gzip.open if path.endswith('.gz') else open
    with opener(path, 'rb') as f:
        lines = [ln[:-1] if ln.endswith(b'\r') else ln for ln in f.read().split(b'\n')]
    while lines and not lines[-1].strip():
        lines.pop()
    while lines and not lines[0].strip():
        lines.pop(0)
    out = []
    if lines and lines[0].startswith(b'@'):
        assert len(lines) % 4 == 0
        for i in range(0, len(lines), 4):
            assert lines[i].startswith(b'@') and lines[i + 2].startswith(b'+')
            out.append(SEP + lines[i + 1])
    else:
        for ln in lines:
            if ln.startswith(b'>'):
                out.append(SEP)
            else:
                out.append(ln)
    return b''.join(out)


def write_fasta(path, records, width=None, crlf=False, gz=False):
    nl = b'\r\n' if crlf else b'\n'
    parts = []
    for i, seq in enumerate(records):
        parts.append(b'>read%d some description' % i + nl)
        if width:
            for j in range(0, len(seq), width):
                parts.append(seq[j:j + width] + nl)
        elif seq or not width:
            parts.append(seq + nl)
    data = b''.join(parts)
    with (gzip.open if gz else open)(path, 'wb') as f:
        f.write(data)


def write_fastq(path, records, crlf=False, gz=False):
    nl = b'\r\n' if crlf else b'\n'
    rng = np.random.default_rng(len(records))
    parts = []
    for i, seq in enumerate(records):
        # quality strings made of letters a base could be, and of '@' / '+', so that a reader that let
        # them through or split records on them would be seen
        qual = bytes(rng.choice(np.frombuffer(b'ACGT@+I#', dtype=np.uint8), len(seq)).tolist())
        parts.append(b'@read%d' % i + nl + seq + nl + b'+' + nl + qual + nl)
    with (gzip.open if gz else open)(path, 'wb') as f:
        f.write(b''.join(parts))


# ---- counting ------------------------------------------------------------------------------------
def _codes(stream):
    b = np.frombuffer(bytes(stream), dtype=np.uint8) | 0x20
    code = np.full(256, 4, dtype=np.uint8)
    for i, ch in enumerate(b'acgt'):
        code[ch] = i
    return code[b]


def canonical_keys(stream, k):
    """Packed canonical keys (uint64) of every window of k bases of a byte stream: pack, reverse
    complement, minimum."""
    c = _codes(stream)
    n = len(c) - k + 1
    if n <= 0:
        return np.zeros(0, dtype=np.uint64)
    bad = np.concatenate(([0], np.cumsum(c > 3)))
    ok = bad[k:] - bad[:-k] == 0
    fwd = np.zeros(n, dtype=np.uint64)
    rev = np.zeros(n, dtype=np.uint64)
    c64 = np.minimum(c, 3).astype(np.uint64)
    for i in range(k):
        w = c64[i:i + n]
        fwd = (fwd << np.uint64(2)) | w
        rev = rev | ((np.uint64(3) - w) << np.uint64(2 * i))
    return np.minimum(fwd, rev)[ok]


def numpy_counts(stream, k):
    """(keys, counts) of the canonical k-mers of a stream, keys ascending (np.unique)."""
    return np.unique(canonical_keys(stream, k), return_counts=True)


def hist_of_counts(counts):
    j, h = np.unique(counts, return_counts=True)
    return {int(a): int(b) for a, b in zip(j, h)}


def dict_counts(stream, k):
    """Canonical k-mer counts by strings: every window of ACGT letters, min(k-mer, reverse complement)."""
    out = {}
    for rec in bytes(stream).upper().replace(SEP, b'N').split(b'N'):
        for i in range(len(rec) - k + 1):
            w = rec[i:i + k]
            if w.strip(b'ACGT'):
                continue
            rc = w.translate(_COMP)[::-1]
            key = min(w, rc)
            out[key] = out.get(key, 0) + 1
    return out


def pack(s):
    v = 0
    for ch in s:
        v = v * 4 + b'ACGT'.index(ch)
    return v


def fmix64(h):
    h = np.asarray(h, dtype=np.uint64).copy()
    h ^= h >> np.uint64(33)
    h *= np.uint64(0xff51afd7ed558ccd)
    h ^= h >> np.uint64(33)
    h *= np.uint64(0xc4ceb9fe1a85ec53)
    h ^= h >> np.uint64(33)
    return h


def part_of(keys, n_parts):
    """The part of each key in a table split n_parts ways (kmers.cu cvk_insert)."""
    return ((fmix64(keys) >> np.uint64(40)) * np.uint64(n_parts)) >> np.uint64(24)


# ---- simulation ----------------------------------------------------------------------------------
def simulate(genome_len, read_len, coverage, error_rate, seed, repeats=()):
    """(genome, reads): a uniform random genome of genome_len bases, in which each (length, copies) of
    `repeats` plants `copies` copies of one random segment at random places; round(coverage * G / r)
    reads of length r from uniform positions on a random strand, each base substituted with probability
    error_rate by one of the three others.  Deterministic in `seed`."""
    rng = np.random.default_rng(seed)
    genome = rng.integers(0, 4, genome_len, dtype=np.uint8)
    for length, copies in repeats:
        seg = rng.integers(0, 4, length, dtype=np.uint8)
        for pos in rng.integers(0, genome_len - length + 1, copies):
            genome[pos:pos + length] = seg
    n_reads = int(round(coverage * genome_len / read_len))
    starts = rng.integers(0, genome_len - read_len + 1, n_reads)
    reads = genome[starts[:, None] + np.arange(read_len)[None, :]]
    flip = rng.random(n_reads) < 0.5
    reads[flip] = 3 - reads[flip, ::-1]
    err = rng.random(reads.shape) < error_rate
    reads[err] = (reads[err] + rng.integers(1, 4, int(err.sum()), dtype=np.uint8)) % 4
    letters = np.frombuffer(b'ACGT', dtype=np.uint8)
    return letters[genome].tobytes(), [letters[r].tobytes() for r in reads]
