"""Canonical k-mer counting on the device: FASTA/FASTQ reads -> the abundance histogram `covest` reads.

    python -m covest_b200.kmers READS... -k 21 -o reads.hist [--table-gib G]

The host reads each file in blocks and compacts every block with numpy into the sequence bytes of its
records, one separator byte before each record (headers and quality lines never reach the device);
the device counts the canonical k-mers of the block in an open-addressed hash table
(csrc/kmers.cu, cvb_kmer_* in include/covest_b200.h) and finally sums the table into the histogram.
Under torch.distributed rank r holds part r of the k-mers, every rank reads every file, and the
per-part histograms are summed over the ranks (DESIGN.md section 11).  The reference's counter is
bin/kmer_hist.py; this one needs no Biopython.
"""
import argparse
import ctypes
import gzip
import math
import os
import sys
from collections import namedtuple

import numpy as np

from . import _capi, parallel
from .engine import DeviceError, _ptr, _stream_ptr, default_device

K_MAX = 31
SLOT_BYTES = 16
BLOCK_BYTES = 64 << 20  # bytes of a file read at a time
LOAD = 0.8              # default table: at most this many slots per input byte of a part
MIN_CAPACITY = 1 << 10
SEP = 0x0A              # the byte before every record of a compacted block (not a base: ends k-mers)
_NL, _CR, _GT, _AT, _PLUS = 0x0A, 0x0D, ord('>'), ord('@'), ord('+')

Block = namedtuple('Block', ('seq', 'reads', 'bases'))


class KmerTableFull(DeviceError):
    """The table (of some rank) dropped k-mers: its histogram would be wrong."""

    def __init__(self, dropped):
        self.dropped = int(dropped)
        super().__init__('the k-mer table is full: %d k-mers were dropped' % self.dropped)


def check_k(k):
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= k <= K_MAX:
        raise ValueError('k must be an integer in [1, %d], not %r' % (K_MAX, k))
    return int(k)


def capacity_for_gib(table_gib):
    """Slots of a table of at most `table_gib` GiB: the largest power of two that fits."""
    try:
        g = float(table_gib)
    except (TypeError, ValueError):
        raise ValueError('table size must be a number of GiB, not %r' % (table_gib,))
    if not math.isfinite(g) or g * (1 << 30) < SLOT_BYTES:
        raise ValueError('table size must be a finite number of GiB that holds a slot, not %r' % (table_gib,))
    slots = int(g * (1 << 30)) // SLOT_BYTES
    return 1 << (slots.bit_length() - 1)


def default_capacity(paths, n_parts, free_bytes):
    """The default table of a run over `paths`: capacity_for_bytes of their size, or of the device's free
    memory alone for compressed input, whose size is not known up front."""
    if any(p.endswith('.gz') for p in paths):
        return capacity_for_bytes(None, n_parts, free_bytes)
    return capacity_for_bytes(sum(os.path.getsize(p) for p in paths), n_parts, free_bytes)


def capacity_for_bytes(n_bytes, n_parts, free_bytes):
    """The smallest power of two of at least n_bytes / n_parts / LOAD slots (at least MIN_CAPACITY), capped
    at the largest power of two of slots that fits half of free_bytes; the cap when n_bytes is None."""
    cap = max(1, int(free_bytes) // 2 // SLOT_BYTES)
    cap = 1 << (cap.bit_length() - 1)
    if n_bytes is None:
        return cap
    need = math.ceil(n_bytes / max(1, n_parts) / LOAD)
    want = 1 << max(0, need - 1).bit_length()
    return min(max(want, MIN_CAPACITY), cap)


# ---- reading -------------------------------------------------------------------------------------
def _line_starts(nl):
    starts = np.empty_like(nl)
    if len(nl):
        starts[0] = 0
        starts[1:] = nl[:-1] + 1
    return starts


def _segments(bounds, first):
    """A bool mask of bounds[-1] bytes: the segments [bounds[i], bounds[i + 1]) alternate between
    `first` and its negation (np.repeat: one fill per segment, no pass of a running sum)."""
    pattern = np.zeros(len(bounds) - 1, dtype=bool)
    pattern[0 if first else 1::2] = True
    return np.repeat(pattern, np.diff(bounds))


def _compact_fasta(b):
    """A writable uint8 block of whole FASTA records ending in a newline -> (compacted, records)."""
    nl = np.flatnonzero(b == _NL)
    starts = _line_starts(nl)
    is_hdr = b[starts] == _GT
    hdr, hdr_end = starts[is_hdr], nl[is_hdr]
    bounds = np.empty(2 * len(hdr) + 2, dtype=np.int64)  # drop what follows '>' up to and with the newline
    bounds[0], bounds[1:-1:2], bounds[2:-1:2], bounds[-1] = 0, hdr + 1, hdr_end + 1, len(b)
    keep = _segments(bounds, True)
    keep &= b != _NL
    cr = nl[(nl > 0)]
    keep[cr[b[cr - 1] == _CR] - 1] = False  # CRLF line endings
    b[hdr] = SEP
    return b[keep], len(hdr)


def _compact_fastq(b, nl, where, first=0):
    """A writable uint8 block of whole 4-line FASTQ records, the first being record `first` of its file
    (counted from 0) -> (compacted, records)."""
    starts = _line_starts(nl)
    hs, ss, ps = starts[0::4], starts[1::4], starts[2::4]
    bad = np.flatnonzero(b[hs] != _AT)
    if len(bad):
        raise ValueError('%s: record %d does not start with @' % (where, first + bad[0] + 1))
    bad = np.flatnonzero(b[ps] != _PLUS)
    if len(bad):
        raise ValueError('%s: line 3 of record %d does not start with +' % (where, first + bad[0] + 1))
    se = nl[1::4].copy()
    se -= (se > ss) & (b[np.maximum(se - 1, 0)] == _CR)
    # per record: keep the header's first byte (made the separator) and the sequence line
    bounds = np.empty(4 * len(hs) + 1, dtype=np.int64)
    bounds[0:-1:4], bounds[1:-1:4], bounds[2:-1:4], bounds[3:-1:4] = hs, hs + 1, ss, se
    bounds[-1] = len(b)
    keep = _segments(bounds, True)
    b[hs] = SEP
    return b[keep], len(hs)


def _open(path):
    return gzip.open(path, 'rb') if path.endswith('.gz') else open(path, 'rb')


def read_blocks(path, block_bytes=BLOCK_BYTES):
    """The records of a FASTA (single-line or wrapped) or 4-line FASTQ file, plain or .gz, as compacted
    blocks: Block(seq = uint8 array of SEP + sequence per record, reads, bases).  A block holds whole
    records only; a record cut by the end of a read is carried over to the next block (a record longer
    than block_bytes makes a block of its own).  Wrapped FASTA lines are joined, CR before a newline is
    dropped, and so are headers and quality lines."""
    fmt = None
    buf = bytearray()
    done = 0  # records yielded
    with _open(path) as f:
        eof = False
        while not eof:
            chunk = f.read(block_bytes)
            eof = not chunk
            buf += chunk
            if fmt is None:
                lead = len(buf) - len(buf.lstrip())
                if lead:
                    del buf[:lead]
                if not buf:
                    continue
                fmt = {_GT: 'fasta', _AT: 'fastq'}.get(buf[0])
                if fmt is None:
                    raise ValueError('%s: neither FASTA (>) nor FASTQ (@)' % path)
            if eof:
                buf = bytearray(buf.rstrip())
                if not buf:
                    break
                buf += b'\n'
            if fmt == 'fasta':
                cut = len(buf) if eof else buf.rfind(b'\n>') + 1
                if cut <= 0:
                    continue
                b = np.frombuffer(buf, dtype=np.uint8, count=cut).copy()
                seq, reads = _compact_fasta(b)
            else:
                nl = np.flatnonzero(np.frombuffer(buf, dtype=np.uint8) == _NL)  # no view outlives the line
                n_rec = len(nl) // 4
                if eof and len(nl) % 4:
                    raise ValueError('%s: the last record is incomplete (%d lines)' % (path, len(nl) % 4))
                if n_rec == 0:
                    continue
                cut = int(nl[4 * n_rec - 1]) + 1
                b = np.frombuffer(buf, dtype=np.uint8, count=cut).copy()
                seq, reads = _compact_fastq(b, nl[:4 * n_rec], path, done)
            del buf[:cut]
            done += reads
            yield Block(seq, reads, len(seq) - reads)


# ---- the device table ----------------------------------------------------------------------------
class KmerCounter:
    """One device k-mer table (cvb_kmer_table): holds part `part` of `n_parts` of the canonical k-mers."""

    def __init__(self, k, capacity, part=0, n_parts=1, device=None):
        self._lib = _capi.load()
        self._t = ctypes.c_void_p()
        self.k = check_k(k)
        self.capacity = int(capacity)
        self.device = default_device() if device is None else int(device)
        rc = self._lib.cvb_kmer_table_create(self.k, self.capacity, int(part), int(n_parts), self.device,
                                             ctypes.byref(self._t))
        if rc != _capi.CVB_OK:
            msg = self._lib.cvb_kmer_last_error(None).decode()
            self._t = ctypes.c_void_p()
            raise (ValueError if rc == -1 else DeviceError)('cvb_kmer_table_create failed (%d): %s' % (rc, msg))

    def _check(self, rc, what):
        if rc != _capi.CVB_OK:
            raise DeviceError('%s failed (%d): %s' % (what, rc, self._lib.cvb_kmer_last_error(self._t).decode()))

    def close(self):
        if getattr(self, '_t', None) is not None and self._t.value:
            self._lib.cvb_kmer_table_destroy(self._t)
            self._t = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def clear(self, stream=None):
        self._check(self._lib.cvb_kmer_clear(self._t, _stream_ptr(stream)), 'cvb_kmer_clear')

    def count(self, seq, stream=None):
        """Counts the k-mers of `seq`: bytes, a uint8 numpy array or a uint8 torch tensor (a CUDA one in
        place, a CPU one through its numpy view)."""
        if isinstance(seq, (bytes, bytearray, memoryview)):
            seq = np.frombuffer(seq, dtype=np.uint8)
        if hasattr(seq, 'data_ptr') and not seq.is_cuda:
            import torch
            if seq.dtype != torch.uint8:
                raise ValueError('sequence tensors must be uint8')
            seq = seq.contiguous().numpy()
        if hasattr(seq, 'data_ptr'):
            import torch
            if seq.dtype != torch.uint8 or not seq.is_contiguous():
                raise ValueError('sequence tensors must be contiguous uint8')
            n = seq.numel()
        else:
            seq = np.ascontiguousarray(seq, dtype=np.uint8)
            n = seq.size
        self._check(self._lib.cvb_kmer_count(self._t, _ptr(seq) if n else None, n, _stream_ptr(stream, seq)),
                    'cvb_kmer_count')

    def stats(self, out=None, stream=None):
        """[distinct, total, max_count, dropped] (int64) of this table."""
        if out is None:
            out = np.zeros(4, dtype=np.int64)
        self._check(self._lib.cvb_kmer_stats(self._t, _ptr(out), _stream_ptr(stream, out)), 'cvb_kmer_stats')
        return out

    def histogram(self, n_bins, out=None, stream=None):
        """int64 array h with h[j - 1] = k-mers seen j times (above n_bins: the last entry).  Raises
        KmerTableFull when the table dropped k-mers."""
        if out is None:
            out = np.zeros(int(n_bins), dtype=np.int64)
        rc = self._lib.cvb_kmer_histogram(self._t, int(n_bins), _ptr(out), _stream_ptr(stream, out))
        if rc == -3:
            raise KmerTableFull(self.stats()[3])
        self._check(rc, 'cvb_kmer_histogram')
        return out


def _allreduce_int64(values, op, device):
    """Element-wise SUM or MAX of an int64 vector over the ranks (NCCL: on `device`; gloo: on the host)."""
    values = np.ascontiguousarray(values, dtype=np.int64)
    rank, w = parallel.world()
    if w == 1:
        return values
    import torch
    dist = parallel._dist()
    t = torch.from_numpy(values.copy())
    if dist.get_backend() == 'nccl':
        t = t.to(torch.device('cuda', device))
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == 'max' else dist.ReduceOp.SUM)
    return t.cpu().numpy()


def count_kmers(paths, k, table_gib=None, device=None, block_bytes=BLOCK_BYTES):
    """The canonical k-mer histogram of the reads in `paths` -> (hist, stats).  hist: {abundance: number
    of distinct k-mers} with only the abundances that occur, ascending; stats: reads, bases, distinct,
    total (k-mers counted) and max_count.  Under torch.distributed every rank reads every file, counts
    its part of the k-mers, and returns the global result.  Raises KmerTableFull (on every rank) when a
    table dropped k-mers: a larger table_gib, or more ranks, holds them."""
    k = check_k(k)
    paths = [os.fspath(p) for p in ([paths] if isinstance(paths, (str, os.PathLike)) else paths)]
    for p in paths:
        if not os.path.isfile(p):
            raise FileNotFoundError('reads file not found: %s' % p)
    capacity = None if table_gib is None else capacity_for_gib(table_gib)
    rank, w = parallel.world()
    device = default_device() if device is None else int(device)
    if capacity is None:
        import torch
        free, _ = torch.cuda.mem_get_info(device)
        capacity = default_capacity(paths, w, free)
    reads = bases = 0
    with KmerCounter(k, capacity, part=rank, n_parts=w, device=device) as kc:
        for p in paths:
            for blk in read_blocks(p, block_bytes):
                kc.count(blk.seq)
                reads += blk.reads
                bases += blk.bases
        distinct, total, max_count, dropped = kc.stats()
        distinct, total, dropped = _allreduce_int64([distinct, total, dropped], 'sum', device)
        max_count = int(_allreduce_int64([max_count], 'max', device)[0])
        if dropped:
            raise KmerTableFull(dropped)
        dense = _allreduce_int64(kc.histogram(max(max_count, 1)), 'sum', device)
    hist = {int(j) + 1: int(dense[j]) for j in np.flatnonzero(dense)}
    return hist, {'reads': reads, 'bases': bases, 'distinct': int(distinct), 'total': int(total),
                  'max_count': max_count}


# ---- command line --------------------------------------------------------------------------------
def build_parser():
    p = argparse.ArgumentParser(prog='python -m covest_b200.kmers',
                                description='Count canonical k-mers of FASTA/FASTQ reads (plain or .gz) on the '
                                            'GPU and write the abundance histogram covest reads.')
    p.add_argument('reads', nargs='+', help='FASTA or FASTQ files')
    p.add_argument('-k', '--kmer-size', type=int, required=True, help='k-mer size, 1 to %d' % K_MAX)
    p.add_argument('-o', '--output', required=True, help='histogram file to write')
    p.add_argument('--table-gib', type=float, default=None,
                   help='hash table size per GPU in GiB (default: from the input size, at most half of '
                        'the free device memory)')
    return p


def run(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    try:
        check_k(args.kmer_size)
        if args.table_gib is not None:
            capacity_for_gib(args.table_gib)
    except ValueError as exc:
        parser.error(str(exc))
    for p in args.reads:
        if not os.path.isfile(p):
            parser.error('reads file not found: %s' % p)
    own_group = False
    if int(os.environ.get('WORLD_SIZE', '1')) > 1 and parallel.world()[1] == 1:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        own_group = True
    try:
        try:
            hist, st = count_kmers(args.reads, args.kmer_size, args.table_gib)
        except KmerTableFull as exc:
            sys.exit('error: %d k-mers did not fit the table and were dropped; give a larger --table-gib '
                     'or count on more GPUs' % exc.dropped)
        if parallel.world()[0] == 0:
            from .data import save_histogram
            meta = {'tool': 'covest_b200.kmers', 'k': args.kmer_size, 'reads': st['reads'], 'bases': st['bases'],
                    'mean_read_length': '%.2f' % (st['bases'] / st['reads'] if st['reads'] else 0.0)}
            save_histogram(hist, args.output, meta)
        return hist, st
    finally:
        if own_group:
            parallel._dist().destroy_process_group()


if __name__ == '__main__':
    run()
