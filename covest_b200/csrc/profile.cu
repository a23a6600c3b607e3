/*
 * profile.cu -- the best point of every segment of a lattice slice (cvb_lattice_profile).
 *
 * A segment is the set of slice points that share the digits of the kept axes; its number is the
 * mixed-radix number of those digits in axis order, the last kept axis fastest.  The best point
 * of a segment is the one cv_topk_select / the radix paths of topk.cu would rank first: larger
 * value first, NaN as -inf, -0 tied with +0, ties to the lower lattice index.
 *
 * Segments are not contiguous in the slice (a profile of the error rate alone takes every
 * len(q1) * len(q2) * len(q)-th run), so nothing here assumes they are.  Four launches, none of
 * whose results depends on the order in which threads run:
 *   cv_prof_init    keys of every segment to 0 ("no point"), indices to the maximum;
 *   cv_prof_max     each warp reduces the order-preserving keys (topk.cu cv_topk_keys) of its lanes
 *                   per segment (a labeled partition: __match_any_sync) and one lane per segment
 *                   atomicMax-es the key of its segment;
 *   cv_prof_argmin  each point whose key equals its segment's maximum offers its lattice index to an
 *                   atomicMin; within a warp the lowest lane of a segment offers it, since the
 *                   lattice index grows with the slice index;
 *   cv_prof_gather  the rows (value, axis values...): the value decoded from the key, as the radix
 *                   top-K reports it; (-inf, NaN...) for a segment without a point.
 * Reading 8 bytes a point twice next to an evaluation of ~1000 bins a point, it is kept apart from
 * the evaluation kernels.
 */
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>

#include "kernels.h"

namespace cg = cooperative_groups;

#define CV_PROF_THREADS 256
#define CV_PROF_NONE 0xffffffffffffffffULL /* the index of a segment without a point, a lane without a point */

__device__ __forceinline__ unsigned long long cv_prof_key(double v)
{
    if (v != v)
        v = -INFINITY;
    if (v == 0.0)
        v = 0.0; /* -0.0 and +0.0 tie */
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL); /* never 0: -inf maps to 0x000fff... */
}

__device__ __forceinline__ double cv_prof_value(unsigned long long key)
{
    const unsigned long long b = (key >> 63) ? (key & 0x7fffffffffffffffULL) : ~key;
    return __longlong_as_double((long long)b);
}

/* lattice index of slice point i (kdevice.h cv_lattice_point) */
__device__ __forceinline__ long long cv_prof_index(const CvLattice &lat, long long i)
{
    if (lat.block > 1) {
        const long long run = i / lat.block;
        return (lat.first + run * lat.stride) * lat.block + (i - run * lat.block);
    }
    return lat.first + i * lat.stride;
}

/* segment of lattice index idx: its kept digits, mixed radix, the last kept axis fastest */
__device__ __forceinline__ long long cv_prof_segment(const CvLattice &lat, long long idx, unsigned int keep)
{
    long long seg = 0, mult = 1;
#pragma unroll
    for (int a = CV_MAX_PARAMS - 1; a >= 0; a--) {
        if (a < lat.n_axes) {
            const long long n = lat.len[a];
            const long long q = idx / n;
            if (keep & (1u << a)) {
                seg += (idx - q * n) * mult;
                mult *= n;
            }
            idx = q;
        }
    }
    return seg;
}

__global__ void __launch_bounds__(CV_PROF_THREADS)
cv_prof_init(long long n_seg, unsigned long long *__restrict__ key, unsigned long long *__restrict__ best)
{
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < n_seg;
         s += (long long)gridDim.x * blockDim.x) {
        key[s] = 0ULL;
        best[s] = CV_PROF_NONE;
    }
}

__global__ void __launch_bounds__(CV_PROF_THREADS)
cv_prof_max(const __grid_constant__ CvLattice lat, unsigned int keep, const double *__restrict__ ll, long long n,
            unsigned long long *__restrict__ key)
{
    const cg::thread_block_tile<32> warp = cg::tiled_partition<32>(cg::this_thread_block());
    const long long step = (long long)gridDim.x * blockDim.x;
    /* the loop bound is the same for the 32 lanes of a warp: every lane takes part in the partition */
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += step) {
        const long long i = base + warp.thread_rank();
        const bool have = i < n;
        const unsigned long long seg =
            have ? (unsigned long long)cv_prof_segment(lat, cv_prof_index(lat, i), keep) : CV_PROF_NONE;
        const unsigned long long k = have ? cv_prof_key(ll[i]) : 0ULL;
        const cg::coalesced_group same = cg::labeled_partition(warp, seg);
        const unsigned long long m = cg::reduce(same, k, cg::greater<unsigned long long>());
        if (have && same.thread_rank() == 0)
            atomicMax(key + seg, m);
    }
}

__global__ void __launch_bounds__(CV_PROF_THREADS)
cv_prof_argmin(const __grid_constant__ CvLattice lat, unsigned int keep, const double *__restrict__ ll, long long n,
               const unsigned long long *__restrict__ key, unsigned long long *__restrict__ best)
{
    const cg::thread_block_tile<32> warp = cg::tiled_partition<32>(cg::this_thread_block());
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += step) {
        const long long i = base + warp.thread_rank();
        unsigned long long seg = CV_PROF_NONE;
        long long idx = 0;
        if (i < n) {
            idx = cv_prof_index(lat, i);
            const unsigned long long s = (unsigned long long)cv_prof_segment(lat, idx, keep);
            if (cv_prof_key(ll[i]) == key[s])
                seg = s;
        }
        const cg::coalesced_group same = cg::labeled_partition(warp, seg);
        if (seg != CV_PROF_NONE && same.thread_rank() == 0) /* the lowest lane: the lowest lattice index */
            atomicMin(best + seg, (unsigned long long)idx);
    }
}

__global__ void __launch_bounds__(CV_PROF_THREADS)
cv_prof_gather(const __grid_constant__ CvLattice lat, long long n_seg, const unsigned long long *__restrict__ key,
               const unsigned long long *__restrict__ best, double *__restrict__ out_rows)
{
    const int np = lat.n_axes;
    for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < n_seg;
         s += (long long)gridDim.x * blockDim.x) {
        double *o = out_rows + s * (1 + np);
        const unsigned long long b = best[s];
        if (b == CV_PROF_NONE) {
            o[0] = -INFINITY;
            for (int a = 0; a < np; a++)
                o[1 + a] = NAN;
            continue;
        }
        o[0] = cv_prof_value(key[s]);
        long long idx = (long long)b;
        for (int a = np - 1; a >= 0; a--) {
            const long long len = lat.len[a];
            const long long q = idx / len;
            o[1 + a] = lat.axis[a][(int)(idx - q * len)];
            idx = q;
        }
    }
}

static unsigned int cv_prof_grid(long long n, int n_sm)
{
    long long blocks = (n + CV_PROF_THREADS - 1) / CV_PROF_THREADS;
    const long long cap = (long long)n_sm * 8;
    return (unsigned int)(blocks < 1 ? 1 : blocks > cap ? cap : blocks);
}

cudaError_t cv_launch_lattice_profile(const CvLattice &lat, unsigned int keep_mask, const double *ll, long long n,
                                      long long n_seg, unsigned long long *seg_key, unsigned long long *seg_best,
                                      double *out_rows, int n_sm, cudaStream_t stream)
{
    const unsigned int gs = cv_prof_grid(n_seg, n_sm);
    cv_prof_init<<<gs, CV_PROF_THREADS, 0, stream>>>(n_seg, seg_key, seg_best);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return e;
    if (n > 0) {
        const unsigned int gp = cv_prof_grid(n, n_sm);
        cv_prof_max<<<gp, CV_PROF_THREADS, 0, stream>>>(lat, keep_mask, ll, n, seg_key);
        if ((e = cudaGetLastError()) != cudaSuccess)
            return e;
        cv_prof_argmin<<<gp, CV_PROF_THREADS, 0, stream>>>(lat, keep_mask, ll, n, seg_key, seg_best);
        if ((e = cudaGetLastError()) != cudaSuccess)
            return e;
    }
    cv_prof_gather<<<gs, CV_PROF_THREADS, 0, stream>>>(lat, n_seg, seg_key, seg_best, out_rows);
    return cudaGetLastError();
}
