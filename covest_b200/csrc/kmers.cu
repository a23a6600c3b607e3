/*
 * kmers.cu -- canonical k-mer counting on the device (DESIGN.md section 11).
 *
 * The table is open-addressed with linear probing over a power-of-two number of 16-byte slots
 * (kmers.h CvkSlot).  A key is the 2-bit packed canonical k-mer -- the smaller of the k-mer and its
 * reverse complement, `jellyfish count -C` -- and picks its first slot by the low bits of fmix64(key).
 * The top 24 bits of the same hash pick the key's part of a partitioned table (part / n_parts), so the
 * part depends on the key alone and never on the capacity.
 *
 * A new key first reserves a unit of the occupancy counter, then claims an empty slot with atomicCAS;
 * the count is raised with atomicAdd.  A reservation is only given while fewer than `limit` are held,
 * so at least capacity / 8 slots (at least one) stay empty and every probe ends.  A key that gets no
 * reservation is counted in CVK_DROPPED and not inserted; the histogram refuses to report a table that
 * dropped anything.
 */
#include <cooperative_groups.h>

#include "kmers.h"

namespace cg = cooperative_groups;

#define CVK_BLOCK 256
#define CVK_RUN 60 /* window end positions per thread: 15 words, an odd stride, so the shared reads do not conflict */
#define CVK_SPAN (CVK_BLOCK * CVK_RUN)
#define CVK_HALO 32 /* >= k - 1 bytes staged before a block's span */
#define CVK_SMEM_BINS 2048 /* counts up to this go to per-block shared bins */

__device__ __forceinline__ unsigned long long cvk_fmix64(unsigned long long h)
{
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return h;
}

/* 2-bit code of a byte: A/a 0, C/c 1, G/g 2, T/t 3, anything else 4 (breaks k-mers) */
__device__ __forceinline__ unsigned char cvk_code_of(unsigned int b)
{
    switch (b | 0x20u) {
    case 'a': return 0;
    case 'c': return 1;
    case 'g': return 2;
    case 't': return 3;
    default: return 4;
    }
}

__device__ __forceinline__ void cvk_insert(const CvkTable &t, unsigned long long key)
{
    const unsigned long long h = cvk_fmix64(key);
    if (t.n_parts > 1 && (unsigned int)(((h >> 40) * t.n_parts) >> 24) != t.part)
        return;
    unsigned long long i = h & t.mask;
    bool reserved = false;
    for (;;) {
        const unsigned long long cur = *(volatile const unsigned long long *)&t.slots[i].key;
        if (cur == key) {
            atomicAdd(&t.slots[i].count, 1ull);
            break;
        }
        if (cur == CVK_EMPTY) {
            if (!reserved) { /* warp-aggregated: one atomic on the counter per group of lanes here */
                cg::coalesced_group g = cg::coalesced_threads();
                unsigned long long base = 0;
                if (g.thread_rank() == 0)
                    base = atomicAdd(&t.state[CVK_OCCUPIED], (unsigned long long)g.size());
                base = g.shfl(base, 0) + g.thread_rank();
                if (base >= t.limit) { /* full: give the unit back, count the k-mer as dropped */
                    atomicAdd(&t.state[CVK_OCCUPIED], ~0ull);
                    atomicAdd(&t.state[CVK_DROPPED], 1ull);
                    return;
                }
                reserved = true;
            }
            const unsigned long long prev = atomicCAS(&t.slots[i].key, CVK_EMPTY, key);
            if (prev == CVK_EMPTY || prev == key) {
                atomicAdd(&t.slots[i].count, 1ull);
                if (prev == key) /* another thread claimed the slot for the same key */
                    break;
                return;
            }
            /* another key took the slot: keep the reservation and probe on */
        }
        i = (i + 1) & t.mask;
    }
    if (reserved)
        atomicAdd(&t.state[CVK_OCCUPIED], ~0ull);
}

/* A block takes spans of CVK_SPAN window end positions; its bytes, with the k - 1 before the span,
 * are staged through shared memory by consecutive threads.  Thread t walks end positions
 * [t * CVK_RUN, (t + 1) * CVK_RUN) of the span with rolling forward and reverse-complement codes,
 * after warming up over the k - 1 bytes before its run.  Bytes outside [0, n) read as 'N'. */
__global__ void __launch_bounds__(CVK_BLOCK) cvk_count_kernel(CvkTable t, const unsigned char *__restrict__ seq,
                                                              long long n)
{
    __shared__ unsigned char code[256];
    __shared__ unsigned char buf[CVK_HALO + CVK_SPAN];
    code[threadIdx.x] = cvk_code_of(threadIdx.x);
    const int k = t.k;
    const int shift = 2 * (k - 1);
    const unsigned long long kmask = (1ull << (2 * k)) - 1;
    for (long long base = (long long)blockIdx.x * CVK_SPAN; base < n; base += (long long)gridDim.x * CVK_SPAN) {
        __syncthreads();
        const long long lo = base - CVK_HALO; /* buf[i] holds seq[lo + i] */
        for (int i = threadIdx.x; i < CVK_HALO + CVK_SPAN; i += CVK_BLOCK) {
            const long long g = lo + i;
            buf[i] = (g >= 0 && g < n) ? seq[g] : (unsigned char)'N';
        }
        __syncthreads();
        const int first = CVK_HALO + threadIdx.x * CVK_RUN - (k - 1);
        unsigned long long fwd = 0, rev = 0;
        int valid = 0;
        for (int i = 0; i < CVK_RUN + k - 1; i++) {
            const unsigned int c = code[buf[first + i]];
            if (c > 3) {
                valid = 0;
                continue;
            }
            fwd = ((fwd << 2) | c) & kmask;
            rev = (rev >> 2) | ((unsigned long long)(3 - c) << shift);
            if (++valid >= k)
                cvk_insert(t, fwd < rev ? fwd : rev);
        }
    }
}

__global__ void cvk_clear_kernel(CvkTable t)
{
    const unsigned long long cap = t.mask + 1;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < cap;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        CvkSlot s;
        s.key = CVK_EMPTY;
        s.count = 0;
        t.slots[i] = s;
    }
    if (blockIdx.x == 0 && threadIdx.x < CVK_STATE_WORDS)
        t.state[threadIdx.x] = 0;
}

__global__ void __launch_bounds__(CVK_BLOCK) cvk_stats_kernel(CvkTable t)
{
    const unsigned long long cap = t.mask + 1;
    unsigned long long distinct = 0, total = 0, mx = 0;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < cap;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const CvkSlot s = t.slots[i];
        if (s.key != CVK_EMPTY) {
            distinct++;
            total += s.count;
            mx = s.count > mx ? s.count : mx;
        }
    }
    for (int o = 16; o; o >>= 1) {
        distinct += __shfl_xor_sync(0xffffffffu, distinct, o);
        total += __shfl_xor_sync(0xffffffffu, total, o);
        const unsigned long long m = __shfl_xor_sync(0xffffffffu, mx, o);
        mx = m > mx ? m : mx;
    }
    if ((threadIdx.x & 31) == 0 && distinct) {
        atomicAdd(&t.state[CVK_DISTINCT], distinct);
        atomicAdd(&t.state[CVK_TOTAL], total);
        atomicMax(&t.state[CVK_MAX], mx);
    }
}

/* Occupied slots by count: counts up to CVK_SMEM_BINS (nearly all of them) into per-block shared bins,
 * flushed once per block; larger counts straight to global atomics.  Integer sums: deterministic. */
__global__ void __launch_bounds__(CVK_BLOCK) cvk_histogram_kernel(CvkTable t, long long n_bins,
                                                                  unsigned long long *hist)
{
    __shared__ unsigned long long bins[CVK_SMEM_BINS];
    const long long nb = n_bins < CVK_SMEM_BINS ? n_bins : CVK_SMEM_BINS;
    for (int i = threadIdx.x; i < nb; i += CVK_BLOCK)
        bins[i] = 0;
    __syncthreads();
    const unsigned long long cap = t.mask + 1;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < cap;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const CvkSlot s = t.slots[i];
        if (s.key == CVK_EMPTY || s.count == 0)
            continue;
        const long long b = (s.count < (unsigned long long)n_bins ? (long long)s.count : n_bins) - 1;
        if (b < nb)
            atomicAdd(&bins[b], 1ull);
        else
            atomicAdd(&hist[b], 1ull);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nb; i += CVK_BLOCK)
        if (bins[i])
            atomicAdd(&hist[i], bins[i]);
}

static int cvk_slot_blocks(const CvkTable &t, int n_sm)
{
    const unsigned long long want = (t.mask + 1 + CVK_BLOCK - 1) / CVK_BLOCK;
    const unsigned long long cap = (unsigned long long)n_sm * 8;
    return (int)(want < cap ? (want ? want : 1) : cap);
}

cudaError_t cvk_launch_clear(const CvkTable &t, int n_sm, cudaStream_t s)
{
    cvk_clear_kernel<<<cvk_slot_blocks(t, n_sm), CVK_BLOCK, 0, s>>>(t);
    return cudaGetLastError();
}

cudaError_t cvk_launch_count(const CvkTable &t, const unsigned char *seq, long long n, int n_sm, cudaStream_t s)
{
    if (n <= 0)
        return cudaSuccess;
    const long long spans = (n + CVK_SPAN - 1) / CVK_SPAN;
    const long long cap = (long long)n_sm * 8;
    cvk_count_kernel<<<(int)(spans < cap ? spans : cap), CVK_BLOCK, 0, s>>>(t, seq, n);
    return cudaGetLastError();
}

cudaError_t cvk_launch_stats(const CvkTable &t, int n_sm, cudaStream_t s)
{
    cvk_stats_kernel<<<cvk_slot_blocks(t, n_sm), CVK_BLOCK, 0, s>>>(t);
    return cudaGetLastError();
}

cudaError_t cvk_launch_histogram(const CvkTable &t, long long n_bins, long long *hist, int n_sm, cudaStream_t s)
{
    cvk_histogram_kernel<<<cvk_slot_blocks(t, n_sm), CVK_BLOCK, 0, s>>>(t, n_bins, (unsigned long long *)hist);
    return cudaGetLastError();
}
