/*
 * kmers.h -- launch interface between the C ABI (capi.cu) and the k-mer counting kernels (kmers.cu).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define CVK_EMPTY (~0ull) /* key of an empty slot: a packed k-mer with k <= 31 never sets the top two bits */

/* One slot of the open-addressed table: 16 bytes, so that an insert touches one 32-byte sector.  The
 * count takes the 8 bytes a 32-bit count would leave as padding: no input can wrap it. */
struct __align__(16) CvkSlot {
    unsigned long long key;   /* 2-bit packed canonical k-mer (A=0 C=1 G=2 T=3, first base most significant) */
    unsigned long long count;
};

/* The device words of a table.  The first four are what cvb_kmer_stats returns, in its order. */
enum { CVK_DISTINCT = 0, CVK_TOTAL = 1, CVK_MAX = 2, CVK_DROPPED = 3, CVK_OCCUPIED = 4, CVK_STATE_WORDS = 5 };

struct CvkTable {
    CvkSlot *slots;
    unsigned long long mask;  /* capacity - 1 */
    unsigned long long limit; /* most slots the table may occupy: capacity - max(1, capacity / 8) */
    unsigned int part, n_parts;
    int k;
    unsigned long long *state; /* CVK_STATE_WORDS device words */
};

/* every slot empty with count 0, and every state word 0 */
cudaError_t cvk_launch_clear(const CvkTable &t, int n_sm, cudaStream_t s);
/* inserts every window of k valid bases that lies inside seq[0, n) (device bytes) */
cudaError_t cvk_launch_count(const CvkTable &t, const unsigned char *seq, long long n, int n_sm, cudaStream_t s);
/* state[CVK_DISTINCT], [CVK_TOTAL], [CVK_MAX] from the slots */
cudaError_t cvk_launch_stats(const CvkTable &t, int n_sm, cudaStream_t s);
/* hist[j - 1] += number of occupied slots with count j (counts above n_bins: the last bin); hist is
 * n_bins device int64 words the caller zeroed */
cudaError_t cvk_launch_histogram(const CvkTable &t, long long n_bins, long long *hist, int n_sm, cudaStream_t s);
