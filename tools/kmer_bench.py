"""Throughput of the k-mer counter (covest_b200/kmers.py, csrc/kmers.cu), one leg at a time:

  device   canonical k-mer inserts per second from device buffers: >= 10^9 simulated read bases (reads of
           150 from a random genome of 10^8 bases, no errors), timed with CUDA events around the counting
           calls only, once with a 4 GiB table (2^28 slots, 32x the 126 MB L2, 37 % full) and once at the
           default table size for that input (2^31 slots, 32 GiB, 5 % full);
  parse    host block reader (read_blocks) on a plain and a gzip FASTQ file, MB of file per second;
  file     python -m covest_b200.kmers on the plain and the gzip file, wall time to the .hist;
  cpu      the numpy canonical counter of tests/kmer_helpers.py (pack, reverse complement, np.unique), the
           baseline: numpy runs it on one host core (the core count is reported beside it);
  ceiling  one 32-byte sector read and written back per insert at 7.7 TB/s (data sheet, 1000 W).

    python tools/kmer_bench.py [--bases 1e9] [--file-mb 600] [--json OUT]

Prints one JSON line (GPU name and power limit included).  Files go to a temporary directory."""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from covest_b200 import kmers  # noqa: E402

K = 21
READ = 150
LETTERS = np.frombuffer(b'ACGT', dtype=np.uint8)


def gpu_facts():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(',')]
        return name, limit
    except Exception as exc:  # the measurement still stands; say what is missing
        return 'unknown (%s)' % exc, 'unknown'


def device_reads(total_bases, genome_len, seed):
    """Chunks (CUDA uint8 tensors, ~10^8 bytes each) of reads of READ bases from a random genome, each
    read preceded by a separator byte."""
    import torch
    g = torch.Generator(device='cuda').manual_seed(seed)
    letters = torch.tensor(list(b'ACGT'), dtype=torch.uint8, device='cuda')
    genome = letters[torch.randint(0, 4, (genome_len,), device='cuda', generator=g)]
    per_chunk = 100_000_000 // (READ + 1)
    chunks, left = [], total_bases // READ
    ar = torch.arange(READ, device='cuda')
    while left > 0:
        n = min(per_chunk, left)
        starts = torch.randint(0, genome_len - READ, (n, 1), device='cuda', generator=g)
        rec = torch.empty((n, READ + 1), dtype=torch.uint8, device='cuda')
        rec[:, 0] = 10
        rec[:, 1:] = genome[starts + ar]
        chunks.append(rec.reshape(-1))
        left -= n
    del genome
    torch.cuda.synchronize()
    return chunks


def time_device(chunks, capacity):
    import torch
    with kmers.KmerCounter(K, capacity) as kc:
        kc.count(chunks[0][:1 << 20])  # first launch
        torch.cuda.synchronize()
        best = None
        for _ in range(2):
            kc.clear()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for c in chunks:
                kc.count(c)
            b.record()
            b.synchronize()
            ms = a.elapsed_time(b)
            best = ms if best is None else min(best, ms)
        st = kc.stats()
        kc.histogram(int(st[2]))  # raises if anything was dropped
    return {'capacity': capacity, 'table_gib': capacity * kmers.SLOT_BYTES / 2 ** 30, 'ms': best,
            'inserts': int(st[1]), 'distinct': int(st[0]), 'inserts_per_s': st[1] / (best * 1e-3),
            'load': int(st[0]) / capacity}


def write_fastq(path, n_reads, genome_len, seed):
    rng = np.random.default_rng(seed)
    genome = rng.integers(0, 4, genome_len, dtype=np.uint8)
    head, mid = np.frombuffer(b'@read\n', np.uint8), np.frombuffer(b'\n+\n', np.uint8)
    width = len(head) + READ + len(mid) + READ + 1
    with open(path, 'wb') as f:
        for lo in range(0, n_reads, 500_000):
            n = min(500_000, n_reads - lo)
            rec = np.empty((n, width), dtype=np.uint8)
            rec[:, :6] = head
            starts = rng.integers(0, genome_len - READ, n)
            codes = genome[starts[:, None] + np.arange(READ)]
            flip = rng.random(n) < 0.5
            codes[flip] = 3 - codes[flip, ::-1]  # reverse strand
            seq = LETTERS[codes]
            rec[:, 6:6 + READ] = seq
            rec[:, 6 + READ:9 + READ] = mid
            rec[:, 9 + READ:-1] = ord('I')
            rec[:, -1] = 10
            f.write(rec.tobytes())


def time_parse(path):
    t0 = time.perf_counter()
    bases = 0
    for blk in kmers.read_blocks(path):
        bases += blk.bases
    s = time.perf_counter() - t0
    return {'file_mb': os.path.getsize(path) / 1e6, 's': s, 'file_mb_per_s': os.path.getsize(path) / 1e6 / s,
            'bases_per_s': bases / s}


def time_file(path, out):
    t0 = time.perf_counter()
    hist, st = kmers.run([path, '-k', str(K), '-o', out])
    s = time.perf_counter() - t0
    return {'s': s, 'bases': st['bases'], 'bases_per_s': st['bases'] / s, 'distinct': st['distinct']}


def time_cpu(n_bases, seed):
    from tests.kmer_helpers import numpy_counts
    rng = np.random.default_rng(seed)
    stream = LETTERS[rng.integers(0, 4, n_bases, dtype=np.uint8)].tobytes()
    t0 = time.perf_counter()
    keys, counts = numpy_counts(stream, K)
    s = time.perf_counter() - t0
    return {'bases': n_bases, 's': s, 'inserts_per_s': int(counts.sum()) / s, 'host_cores': os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--bases', type=float, default=1e9)
    ap.add_argument('--genome', type=float, default=1e8)
    ap.add_argument('--file-mb', type=float, default=600)
    ap.add_argument('--gz-mb', type=float, default=150)
    ap.add_argument('--cpu-bases', type=float, default=2e7)
    ap.add_argument('--json', default=None)
    args = ap.parse_args()
    import torch
    name, limit = gpu_facts()
    res = {'gpu': name, 'power_limit': limit, 'k': K, 'read_length': READ}
    chunks = device_reads(int(args.bases), int(args.genome), 1)
    res['device_4gib_table'] = time_device(chunks, 1 << 28)  # 32x the L2, 8x smaller than the default
    free, _ = torch.cuda.mem_get_info()
    cap = kmers.capacity_for_bytes(int(args.bases * (READ + 1) / READ), 1, free)  # the default for these bytes
    res['device_default_table'] = time_device(chunks, cap)
    del chunks
    torch.cuda.empty_cache()
    res['ceiling_inserts_per_s'] = 7.7e12 / 64  # a 32-byte sector read and written back per insert
    tmp = tempfile.mkdtemp(prefix='kmer_bench_')
    try:
        fq = os.path.join(tmp, 'reads.fq')
        width = 6 + 2 * READ + 4
        write_fastq(fq, int(args.file_mb * 1e6 / width), 10_000_000, 2)
        gz = fq + '.gz'
        with open(fq, 'rb') as src, gzip.open(gz, 'wb', compresslevel=1) as dst:
            dst.write(src.read(int(args.gz_mb * 1e6) // width * width))
        res['parse_plain'] = time_parse(fq)
        res['parse_gz'] = time_parse(gz)
        res['file_plain'] = time_file(fq, os.path.join(tmp, 'plain.hist'))
        res['file_gz'] = time_file(gz, os.path.join(tmp, 'gz.hist'))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    res['cpu_numpy'] = time_cpu(int(args.cpu_bases), 3)
    line = json.dumps(res)
    print(line)
    if args.json:
        with open(args.json, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
