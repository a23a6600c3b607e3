/*
 * factored.cu -- batched evaluation of the repeats model as profiles x copy weights (factored.h).
 *
 *   cvf_point_keys      K0: per point clip, cut-off O_thr, sort key ((c, e) hash | q | O_thr)
 *   cvf_heads / cvf_group_starts / cvf_group_counts / cvf_group_scan / cvf_tile_table
 *                       groups (equal (c, e)), q-runs (equal q inside a group) and tiles from the
 *                       sorted keys -- the plan of an explicit point array
 *   cvf_lattice_fill / cvf_lattice_order
 *                       the same tables for a lattice handed over as its axes: from a template of
 *                       one group computed on the host (cvf_lattice_template), no sort, nothing
 *                       read back
 *   cvf_profile_kernel  K1: one warp per (group, 16 copy numbers): profiles over all bins; a row
 *                       keeps the 64-bin lines that hold a count, the others leave as 32 sums
 *                       (factored.h, CvfSlots: they enter the result through the mass only)
 *   cvf_prefix_kernel   K2p: one CTA per tile of up to four q-runs: running sums over the copy
 *                       numbers, per point the three-term combination + epilogue (the default for
 *                       batches whose points share q, as lattices do); warps per CTA and slots per
 *                       thread are template parameters picked to cover a row in one pass
 *   cvf_weights_kernel, cvf_gemm_kernel   K1b, K2: one CTA per tile of 128 points: copy weights and
 *                       FP64 tensor-core GEMM + epilogue (batches that share (c, e) but not q)
 *
 * cub's device radix sort and prefix sums order the keys and lay out the group tables (plumbing);
 * every likelihood flop is in the hand-written kernels of this file and of cvpoint.h.
 *
 * Reference lines are relative to /root/reference.
 */
#include "factored.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cstring>
#include <vector>

#include "kdevice.h"

#define CVF_M 128       /* points per tile of K2 */
#define CVF_NS 64       /* bins (slots) per N-step of K2 */
#define CVF_KC 16       /* copy numbers per K-chunk */
#define CVF_THREADS 256
#define CVF_OBITS 20    /* bits of O_thr in the sort key */
#define CVF_TILE_DOUBLES (CVF_KC * CVF_NS)

/* device view of the plan of one batch */
struct CvfPlan {
    unsigned long long *keys, *keys_alt;
    unsigned int *idx, *idx_alt; /* after the sort: point index by sorted position (in idx_sorted) */
    const unsigned int *idx_sorted;
    int *othr;       /* by ORIGINAL point index */
    int *head, *gid; /* by sorted position */
    unsigned long long *flags2; /* by sorted position: head | head2 << 32, then their running sums (gid | rid << 32) */
    int *head2, *rid; /* q-runs: points of a group that also share q (prefix path); rid = running count */
    int *g_omax;      /* [n + 1] per group: the largest O_thr of its points */
    int *r_start;     /* [n + 1] sorted position of the first point of a q-run */
    int *g_rfirst;    /* [n + 1] per group: index of its first q-run */
    int *g_start;    /* [n + 1] sorted position of the first point of a group */
    int *tile_start; /* [n + 1] counts, then exclusive prefix */
    int *item_start;
    long long *w_off;
    int *a_start;    /* [n + 1] per group: K-chunks of copy weights of all its tiles, then prefix */
    /* per tile of K2 (filled by cvf_tile_table once the number of tiles is known) */
    int *t_first, *t_cnt, *t_nkc, *t_aoff, *t_group;
    int *t_key, *t_key_alt, *t_order, *t_order_alt; /* tiles by descending number of K-chunks */
    const int *t_sorted;
    long long *header; /* n_groups, tiles, items, profile doubles, weight chunks, q-runs */
    int obits;         /* bits of O_thr in the sort key: enough for max(hist) + padding */
    int tile_points;   /* points per tile of K2 (the prefix kernel's tiles are whole q-runs) */
    int prefix;        /* 1: sorted by (c, e), q, O_thr and tiled for the prefix kernel */
};

/* slots a copy takes in a term tile of the profile kernel: S rounded up to a multiple of 4 */
__host__ __device__ __forceinline__ int cvf_copy_slots(int n_err) { return (n_err + 3) & ~3; }
/* copies per tile: the largest power of two that fits 32 lanes */
__host__ __device__ __forceinline__ int cvf_copies_per_tile(int n_err)
{
    int c = 32 / cvf_copy_slots(n_err);
    return c >= 8 ? 8 : c >= 4 ? 4 : c >= 2 ? 2 : 1;
}

bool cvf_supported(const CvModelDesc &m)
{
    return m.model_kind == 1 && m.n_err <= 32 && m.max_bin < (1 << CVF_OBITS) - CV_COPY_PAD;
}

__device__ __forceinline__ unsigned int cvf_hash(double c, double e)
{
    unsigned long long x = (unsigned long long)__double_as_longlong(c) * 0x9E3779B97F4A7C15ULL;
    x ^= (unsigned long long)__double_as_longlong(e) + 0xD6E8FEB86659FD93ULL + (x << 6) + (x >> 2);
    x ^= x >> 32;
    x *= 0xD6E8FEB86659FD93ULL;
    x ^= x >> 29;
    return (unsigned int)x;
}

/* K0 */
__global__ void __launch_bounds__(256)
cvf_point_keys(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
               const double *__restrict__ params, long long n, int clip, CvfPlan pl)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    double row[CV_MAX_PARAMS];
    cvf_raw_row(m, lat, params, i, row);
    const double c = cvf_clipped(m, row, clip, 0), e = cvf_clipped(m, row, clip, 1);
    const double q1 = cvf_clipped(m, row, clip, 2), q2 = cvf_clipped(m, row, clip, 3),
                 q = cvf_clipped(m, row, clip, 4);
    const double two = cv_mul(cv_sub(1.0, q1), q2);                          /* models.py:195 */
    const double many = cv_mul(cv_mul(cv_sub(1.0, q1), cv_sub(1.0, q2)), q); /* models.py:196 */
    const double base = cv_sub(1.0, q);
    const int othr = cvf_cutoff(m, q1, two, many, base);
    pl.othr[i] = othr;
    pl.idx[i] = (unsigned int)i;
    /* (c, e) hash | q hash (prefix path only) | O_thr: one sort makes groups of equal (c, e), inside
     * them runs of equal q, inside those ascending cut-offs */
    unsigned long long key = ((unsigned long long)cvf_hash(c, e) << 32) | (unsigned long long)othr;
    if (pl.prefix) { /* q in the bits above O_thr: runs of a group in ascending q, so that neighbours
                        need about the same number of copies; q-values closer than the key's
                        resolution share a key and merely interleave (more, shorter runs) */
        const int qbits = 32 - pl.obits;
        const double qc = q > 0.0 ? (q < 1.0 ? q : 1.0) : 0.0; /* NaN -> 0 */
        const unsigned long long qk = (unsigned long long)(qc * (double)((1u << qbits) - 1u));
        key |= qk << pl.obits;
    }
    pl.keys[i] = key;
}

/* head[i] = 1 when sorted position i opens a group: its (c, e) differs from the position before */
__global__ void __launch_bounds__(256)
cvf_heads(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
          const double *__restrict__ params, long long n, int clip, CvfPlan pl)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    int h = 1, h2 = 1;
    if (i > 0) {
        double a[CV_MAX_PARAMS], b[CV_MAX_PARAMS];
        cvf_raw_row(m, lat, params, pl.idx_sorted[i], a);
        cvf_raw_row(m, lat, params, pl.idx_sorted[i - 1], b);
        const long long c0 = __double_as_longlong(cvf_clipped(m, a, clip, 0));
        const long long c1 = __double_as_longlong(cvf_clipped(m, b, clip, 0));
        const long long e0 = __double_as_longlong(cvf_clipped(m, a, clip, 1));
        const long long e1 = __double_as_longlong(cvf_clipped(m, b, clip, 1));
        h = (c0 != c1) || (e0 != e1);
        h2 = h || (pl.prefix && __double_as_longlong(cvf_clipped(m, a, clip, 4)) !=
                                    __double_as_longlong(cvf_clipped(m, b, clip, 4)));
    }
    pl.head[i] = h;
    pl.head2[i] = h2;
    pl.flags2[i] = (unsigned long long)h | ((unsigned long long)h2 << 32);
}

__global__ void __launch_bounds__(256) cvf_group_starts(long long n, CvfPlan pl)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const unsigned long long both = pl.flags2[i]; /* running sums of head and head2 in one scan */
    const int gid = (int)(both & 0xffffffffULL), rid = (int)(both >> 32);
    pl.rid[i] = rid;
    if (pl.head[i]) {
        pl.g_start[gid - 1] = (int)i;
        pl.g_rfirst[gid - 1] = rid - 1;
    }
    if (pl.head2[i])
        pl.r_start[rid - 1] = (int)i;
    if (i == n - 1) {
        pl.header[0] = gid;
        pl.header[5] = rid;
        pl.g_start[gid] = (int)n;
        pl.g_rfirst[gid] = rid;
        pl.r_start[rid] = (int)n;
    }
    /* cut-offs ascend inside a q-run: its last point holds the run's maximum */
    if (i == n - 1 || pl.head2[i + 1])
        atomicMax(pl.g_omax + (gid - 1), pl.othr[pl.idx_sorted[i]]);
}

/* Tiles of the prefix kernel of group g: up to CVF_NQ consecutive whole q-runs with at most
 * CVF_PB points together (one batch of the kernel), or one longer run alone, cut every CVF_PSPLIT
 * points.  emit(first sorted position, points, first run, runs). */
#define CVF_NQ 4   /* q-runs whose running sums a thread of the prefix kernel holds */
#define CVF_PB 512 /* points per batch of the prefix kernel */
#define CVF_PSPLIT 2048
template <class F>
__device__ __forceinline__ int cvf_prefix_tiles(const CvfPlan &pl, int g, F emit)
{
    const int r1 = pl.g_rfirst[g + 1];
    int r = pl.g_rfirst[g], tiles = 0;
    while (r < r1) {
        const int first = pl.r_start[r], rfirst = r;
        int end = first, runs = 0;
        while (r < r1 && runs < CVF_NQ) {
            const int re = pl.r_start[r + 1];
            if (runs > 0 && re - first > CVF_PB)
                break;
            end = re;
            r++;
            runs++;
        }
        for (int p = first; p < end; p += CVF_PSPLIT, tiles++)
            emit(tiles, p, min(CVF_PSPLIT, end - p), rfirst, runs);
    }
    return tiles;
}

/* per group: tiles of K2, items of K1, doubles of its profiles; zeros past the last group so that
 * the exclusive prefix sums end in the totals */
__global__ void __launch_bounds__(256) cvf_group_counts(long long n, int slots_padded, CvfPlan pl)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g > n)
        return;
    const long long ng = pl.header[0];
    int tiles = 0, items = 0, achunks = 0;
    long long w = 0;
    if (g < ng) {
        const int a = pl.g_start[g], b = pl.g_start[g + 1];
        const int tp = pl.tile_points;
        const int omax = max(pl.g_omax[g] - 1, 0);
        tiles = pl.prefix ? cvf_prefix_tiles(pl, (int)g, [](int, int, int, int, int) {}) : (b - a + tp - 1) / tp;
        items = (omax + CVF_KC - 1) / CVF_KC;
        w = (long long)items * CVF_KC * slots_padded;
        if (!pl.prefix)
            for (int p = a; p < b; p += tp) { /* K-chunks of every tile of K2: its last point has the most copies */
                const int last = min(p + tp, b) - 1;
                const int kmax = max(pl.othr[pl.idx_sorted[last]] - 1, 0);
                achunks += (kmax + CVF_KC - 1) / CVF_KC;
            }
    }
    pl.tile_start[g] = tiles;
    pl.item_start[g] = items;
    pl.w_off[g] = w;
    pl.a_start[g] = achunks;
}

/* The exclusive prefix sums of the four per-group counts (tiles, items, profile doubles, weight
 * chunks) over the n_groups + 1 entries that exist -- the host does not know n_groups yet, a scan
 * per array over all n + 1 slots costs eight launches -- and the totals into the header.  One CTA,
 * 1024 groups per round. */
__global__ void __launch_bounds__(1024) cvf_group_scan(CvfPlan pl)
{
    typedef cub::BlockScan<long long, 1024> Scan;
    __shared__ typename Scan::TempStorage tmp;
    const int ng = (int)pl.header[0];
    long long run_t = 0, run_i = 0, run_w = 0, run_a = 0;
    for (int g0 = 0; g0 <= ng; g0 += 1024) {
        const int g = g0 + threadIdx.x;
        const bool in = g <= ng;
        const long long t = in ? pl.tile_start[g] : 0, it = in ? pl.item_start[g] : 0, w = in ? pl.w_off[g] : 0,
                        a = in ? pl.a_start[g] : 0;
        long long et, ei, ew, ea, tt, ti, tw, ta;
        Scan(tmp).ExclusiveSum(t, et, tt);
        __syncthreads();
        Scan(tmp).ExclusiveSum(it, ei, ti);
        __syncthreads();
        Scan(tmp).ExclusiveSum(w, ew, tw);
        __syncthreads();
        Scan(tmp).ExclusiveSum(a, ea, ta);
        __syncthreads();
        if (in) {
            pl.tile_start[g] = (int)(run_t + et);
            pl.item_start[g] = (int)(run_i + ei);
            pl.w_off[g] = run_w + ew;
            pl.a_start[g] = (int)(run_a + ea);
        }
        run_t += tt;
        run_i += ti;
        run_w += tw;
        run_a += ta;
    }
    if (threadIdx.x == 0) { /* entry ng of the counts is 0: the exclusive sums there are the totals */
        pl.header[1] = run_t;
        pl.header[2] = run_i;
        pl.header[3] = run_w;
        pl.header[4] = run_a;
    }
}

/* one thread per group: the records of its tiles */
__global__ void __launch_bounds__(128) cvf_tile_table(int n_groups, CvfPlan pl)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups)
        return;
    const int a = pl.g_start[g], b = pl.g_start[g + 1];
    const int tile0 = pl.tile_start[g];
    if (pl.prefix) {
        cvf_prefix_tiles(pl, g, [&](int t, int first, int cnt, int rfirst, int runs) {
            const int tile = tile0 + t;
            int kmax = 0; /* cut-offs ascend inside a q-run: the last points hold the maxima */
            for (int r = rfirst; r < rfirst + runs; r++) {
                const int last = min(pl.r_start[r + 1], first + cnt) - 1;
                if (last >= first)
                    kmax = max(kmax, pl.othr[pl.idx_sorted[last]] - 1);
            }
            pl.t_first[tile] = first;
            pl.t_cnt[tile] = cnt;
            pl.t_nkc[tile] = (kmax + CVF_KC - 1) / CVF_KC;
            pl.t_aoff[tile] = 0;
            pl.t_group[tile] = g;
            pl.t_key[tile] = 4 * cnt + 3 * kmax; /* about the cost: the costly tiles start first */
            pl.t_order[tile] = tile;
        });
        return;
    }
    const int tp = pl.tile_points;
    int tile = tile0, aoff = pl.a_start[g];
    for (int p = a; p < b; p += tp, tile++) {
        const int cnt = min(tp, b - p);
        const int kmax = max(pl.othr[pl.idx_sorted[p + cnt - 1]] - 1, 0); /* cut-offs ascend along the group */
        const int nkc = (kmax + CVF_KC - 1) / CVF_KC;
        pl.t_first[tile] = p;
        pl.t_cnt[tile] = cnt;
        pl.t_nkc[tile] = nkc;
        pl.t_aoff[tile] = aoff;
        pl.t_group[tile] = g;
        pl.t_key[tile] = nkc; /* the long tiles start first */
        pl.t_order[tile] = tile;
        aoff += nkc;
    }
}

/* ------------------------------------------------------------------------------------------- */
/* The plan of a lattice, from its axes                                                          */
/* ------------------------------------------------------------------------------------------- */
/* A Cartesian lattice handed over as axes (cvb_lattice_eval; what grid.py's rounds and initial
 * boxes are) needs no sort: its groups are the (c, e) index pairs, its q-runs the values of the q
 * axis, and the cut-off O_thr (models.py:185-191) depends on (q1, q2, q) only -- |q1| |q2| |q|
 * values for the whole batch instead of one per point.  The host evaluates those once per set of
 * axes (the *template* of a group: its points by (q ascending, O_thr ascending, lattice order),
 * their cut-offs, its tiles and their order by cost), the template travels to the device (a few
 * KB, only when the axes changed), and one kernel writes the same tables the sort-based plan
 * produces.  Every size is known on the host: no device -> host round trip, nothing blocks. */
struct CvfLatticeDev { /* device copies of the template */
    const int *perm;   /* [M] lattice offset inside the group of the point at sorted offset t */
    const int *othr;   /* [M] its cut-off */
    const int *tt_first, *tt_cnt, *tt_kmax, *tt_order; /* [nT] tiles of a group; by descending cost */
};

__global__ void __launch_bounds__(256)
cvf_lattice_fill(CvfPlan pl, CvfLatticeDev T, int G, int M, int R, int nq, int nT, int omax, int items,
                 long long wpg)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n = (long long)G * M;
    if (p < n) {
        const int g = (int)(p / M), t = (int)(p - (long long)g * M);
        const unsigned int idx = (unsigned int)((long long)g * M + T.perm[t]);
        pl.idx[p] = idx;
        pl.othr[idx] = T.othr[t];
        const int run = t / R;
        pl.head[p] = t == 0;
        pl.head2[p] = t - run * R == 0;
        pl.rid[p] = g * nq + run + 1;
    }
    if (p <= G) { /* per group; entry G closes the prefix tables */
        pl.g_start[p] = (int)(p * M);
        pl.g_rfirst[p] = (int)(p * nq);
        pl.g_omax[p] = p < G ? omax + 1 : 0;
        pl.item_start[p] = (int)(p * items);
        pl.w_off[p] = p * wpg;
        pl.tile_start[p] = (int)(p * nT);
        pl.a_start[p] = 0;
    }
    if (p <= (long long)G * nq)
        pl.r_start[p] = (int)(p * R);
    if (p < (long long)G * nT) {
        const int g = (int)(p / nT), tt = (int)(p - (long long)g * nT);
        const int kmax = T.tt_kmax[tt];
        pl.t_first[p] = g * M + T.tt_first[tt];
        pl.t_cnt[p] = T.tt_cnt[tt];
        pl.t_nkc[p] = (kmax + CVF_KC - 1) / CVF_KC;
        pl.t_aoff[p] = 0;
        pl.t_group[p] = g;
    }
    if (p == 0) {
        pl.header[0] = G;
        pl.header[1] = (long long)G * nT;
        pl.header[2] = (long long)G * items;
        pl.header[3] = (long long)G * wpg;
        pl.header[4] = 0;
        pl.header[5] = (long long)G * nq;
    }
}

/* The order in which the CTAs draw the tiles of the groups g0 .. g1 - 1 (every group has the same
 * tiles): by descending cost over the whole range, i.e. first every group's costliest tile -- the
 * ones that stream the long copy series of the smallest q -- then the next ...  Group by group
 * (inside a group by descending cost, so that the HBM traffic of the long series spreads over the
 * whole kernel) measured cfg3 1.50 ms against 1.44 ms -- its costly tiles finishing last leave SMs
 * idle at the end -- and cfg5 27.4 against 27.8 ms. */
__global__ void __launch_bounds__(256)
cvf_lattice_order(CvfLatticeDev T, int g0, int g1, int nT, int *__restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int ng = g1 - g0;
    if (i >= (long long)ng * nT)
        return;
    const int k = (int)(i / ng);
    const int g = g0 + (int)(i - (long long)k * ng);
    out[i] = g * nT + T.tt_order[k];
}

/* largest g in [0, n) with start[g] <= x (start ascending, start[0] <= x), for a whole warp at once:
 * 32 probes per round, two or three dependent loads instead of log2(n) */
__device__ __forceinline__ int cvf_find_warp(const int *__restrict__ start, int n, int x, int lane)
{
    int lo = 0, hi = n;
    while (hi - lo > 1) {
        const int step = (hi - lo + 31) >> 5;
        const int p = lo + (lane + 1) * step;
        const bool ok = p < hi && __ldg(start + p) <= x;
        const int cnt = __popc(__ballot_sync(CV_FULL_MASK, ok)); /* probes ascend: the first cnt are <= x */
        const int nlo = lo + cnt * step;
        hi = min(nlo + step, hi);
        lo = nlo;
    }
    return lo;
}

/* ------------------------------------------------------------------------------------------- */
/* K1: profiles                                                                                 */
/* ------------------------------------------------------------------------------------------- */
/* Layout of the profiles of a group in HBM: one ROW per copy number, [copy][line][pair L][2]: a
 * row holds all (padded) slots of the histogram in lines of 64 slots (one N-step of K2), and inside
 * a line pair L = 8 * (row of the N-step) + column % 8 holds the slots with columns c and c + 8 of
 * that row.  The lines of a row are those of the histogram tables that hold a bin with a count, in
 * their order, and -- when there are others -- one more line with the column sums of the others
 * (CvfSlots, factored.h): the bins without counts enter the result through the mass only, and the
 * mass is linear in the profiles.  Without a tail the mass does not enter at all: the tables K1 runs
 * on are then the row tables of the lines with counts, and the line of the sums holds zeros.  K1
 * writes 512 contiguous bytes per (copy, line) with one warp-wide store; every thread of the prefix
 * kernel fetches its own slots of a row, one double per slot, into a private cp.async ring; K2
 * scatters 16 rows x one line into its fragment order while loading. */
#define CVF_STAGE_DOUBLES (CV_GB * CV_NA_MAX * CV_W)

/* The accumulators of a lane after the slices of ONE copy are its share of the profile of that
 * copy over block `blk`: rows mt of group r, columns 8 nt + 2 q + c.  They are transposed through
 * the warp's stage in shared memory ([row][column % 8][column / 8], the 16-byte chunks of odd
 * groups swapped pairwise against bank conflicts) and leave as full 512-byte lines. */
template <int NA>
__device__ __forceinline__ void cvf_store_profile(int lane, int blk, int o, int nsteps,
                                                  const double *__restrict__ slot_mult /* pairs */,
                                                  const int *__restrict__ line_map, int sum_line, bool sums,
                                                  double *__restrict__ Wg, double *stage, const double *acc)
{
    const int r = lane >> 2, q = lane & 3;
#pragma unroll
    for (int mt = 0; mt < NA; mt++)
#pragma unroll
        for (int c = 0; c < 2; c++) {
            const int chunk = (2 * q + c) ^ (r & 1);
            *reinterpret_cast<double2 *>(stage + (NA * r + mt) * CV_W + 2 * chunk) =
                make_double2(acc[4 * mt + c], acc[4 * mt + 2 + c]);
        }
    __syncwarp();
    /* row o - 1 of the group's profiles, pair `lane` of its lines */
    double *row0 = Wg + (long long)(o - 1) * nsteps * CVF_NS + lane * 2;
    double2 rest = make_double2(0.0, 0.0); /* the lane's columns of the lines without counts */
#pragma unroll
    for (int ns = 0; ns < 2 * NA; ns++) {
        const int row = 4 * ns + (lane >> 3);
        const int chunk = (lane & 7) ^ ((row / NA) & 1);
        double2 v = *reinterpret_cast<const double2 *>(stage + row * CV_W + 2 * chunk);
        /* the scale of the accumulators ends here: slot_mult of the pair's two slots (0 = the slot
         * is no bin of the histogram; its profile is an exact zero) */
        const double2 mm = __ldg(reinterpret_cast<const double2 *>(slot_mult) + (blk * (2 * NA) + ns) * 32 + lane);
        v.x = cv_mul(v.x, mm.x); /* the accumulators are finite (that is what the scale is for): times 0 is 0 */
        v.y = cv_mul(v.y, mm.y);
        const int line = __ldg(line_map + blk * (2 * NA) + ns); /* the same in every lane */
        if (line >= 0) {
            *reinterpret_cast<double2 *>(row0 + line * CVF_NS) = v;
        } else if (sums) {
            rest.x = cv_add(rest.x, v.x);
            rest.y = cv_add(rest.y, v.y);
        }
    }
    if (sum_line >= 0) {
        /* one sum per lane: the first half of the line; block after block adds to the lane's own
         * double, a fixed order.  The second half stays zero (K2 reads whole lines).  Without a tail
         * (sums = false) nothing reads the sums: the line is written as zeros. */
        double *dst = Wg + ((long long)(o - 1) * nsteps + sum_line) * CVF_NS + lane;
        double sum = 0.0;
        if (sums) {
            sum = cv_add(rest.x, rest.y);
            if (blk > 0)
                sum = cv_add(*dst, sum);
        }
        dst[0] = sum;
        dst[32] = 0.0;
    }
    __syncwarp();
}

template <int NA>
__device__ __forceinline__ void cvf_profile_item(int lane, const CvModelDesc &m, CvWarpMem &M,
                                                 int o0, int omax4, int nsteps, const int *__restrict__ line_map,
                                                 int sum_line, double *__restrict__ Wg, double *stage)
{
    const int sp = cvf_copy_slots(m.n_err);
    const int cpt = cvf_copies_per_tile(m.n_err);
    const int kpc = sp >> 2; /* MMA slices per copy */
    const bool sums = m.tail != 0.0; /* the mass enters the result: the line of the sums carries it */
    for (int oa = o0; oa < o0 + CVF_KC && oa <= omax4; oa += cpt) {
        cv_w_mass(lane, m, oa, cpt * sp, sp, M);
        __syncwarp();
        const CvTerm tm = cv_w_term(lane, m, oa, cpt * sp, sp, 0, 1.0, M);
        for (int blk = 0; blk < m.n_blocks; blk++) {
            const CvLaneGroup G = cv_lane_group(lane, m, blk, M);
            cv_w_prep<NA>(lane, m, blk, tm, M);
            __syncwarp();
            for (int cc = 0; cc < cpt; cc++) {
                double acc[4 * NA];
#pragma unroll
                for (int i = 0; i < 4 * NA; i++)
                    acc[i] = 0.0;
                cv_w_fused<NA>(lane, G, cc * kpc, (cc + 1) * kpc, *M.fx, acc);
                cvf_store_profile<NA>(lane, blk, oa + cc, nsteps, m.tab.slot_mult_pair, line_map, sum_line, sums, Wg, stage,
                                      acc);
            }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(32 * CV_WARPS_MAX, 1)
cvf_profile_kernel(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
                   const double *__restrict__ params, int clip, CvfPlan pl, int n_groups,
                   int first_item, int n_items, double *__restrict__ W, long long w_base, int nsteps,
                   const int *__restrict__ line_map, int sum_line, unsigned long long *counter, int groups_staged)
{
    extern __shared__ __align__(16) unsigned char cv_smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int S = m.n_err;
    CvWarpMem M;
    {
        double *tab = reinterpret_cast<double *>(cv_smem_raw);
        const int ntab = groups_staged * CV_GD;
        unsigned char *wbase = cv_smem_raw + (size_t)ntab * sizeof(double) + (size_t)warp * cv_warp_bytes(S);
        CvWarpFixed *fx = reinterpret_cast<CvWarpFixed *>(wbase);
        cv_warp_mem_carve(M, fx, reinterpret_cast<double *>(wbase + sizeof(CvWarpFixed)), S);
        for (int i = threadIdx.x; i < ntab; i += blockDim.x)
            tab[i] = m.tab.grp[i];
        M.grp = tab;
    }
    double *stage = reinterpret_cast<double *>(cv_smem_raw + (size_t)groups_staged * CV_GD * sizeof(double) +
                                               (size_t)(blockDim.x >> 5) * cv_warp_bytes(S)) +
                    (size_t)warp * CVF_STAGE_DOUBLES;
    __syncthreads();
    for (;;) {
        long long it = 0;
        if (lane == 0)
            it = (long long)atomicAdd(counter, 1ULL);
        it = __shfl_sync(CV_FULL_MASK, it, 0);
        if (it >= n_items)
            break;
        const int item = first_item + (int)it;
        const int g = cvf_find_warp(pl.item_start, n_groups, item, lane);
        const int kchunk = item - pl.item_start[g];
        const int a = pl.g_start[g];
        const int omax = pl.g_omax[g] - 1;
        const int omax4 = (omax + 3) & ~3;
        double row[CV_MAX_PARAMS];
        cvf_raw_row(m, lat, params, pl.idx_sorted[a], row);
        __syncwarp();
        cv_w_header(lane, m, row, clip, M);
        __syncwarp();
        double *Wg = W + (pl.w_off[g] - w_base);
        const int o0 = kchunk * CVF_KC + 1;
        switch (m.na) {
        case 1: cvf_profile_item<1>(lane, m, M, o0, omax4, nsteps, line_map, sum_line, Wg, stage); break;
        case 2: cvf_profile_item<2>(lane, m, M, o0, omax4, nsteps, line_map, sum_line, Wg, stage); break;
        case 4: cvf_profile_item<4>(lane, m, M, o0, omax4, nsteps, line_map, sum_line, Wg, stage); break;
        default: cvf_profile_item<8>(lane, m, M, o0, omax4, nsteps, line_map, sum_line, Wg, stage); break;
        }
    }
}

/* ------------------------------------------------------------------------------------------- */
/* K2: GEMM + epilogue                                                                          */
/* ------------------------------------------------------------------------------------------- */
#define CVF_STAGES 4
struct CvfSmem {
    double2 Bs[CVF_STAGES][CVF_TILE_DOUBLES / 2];     /* profile tiles in flight, fragment order */
    double2 As[CVF_STAGES][CVF_M * CVF_KC / 2];       /* copy-weight tiles in flight, fragment order */
    double red_sum[2][CVF_M];
    double red_mh[2][CVF_M], red_ml[2][CVF_M];
    double log_tab[2 * CV_LOG_N]; /* cv_log_tab: (invc, logc) */
    int othr[CVF_M];
    unsigned int pidx[CVF_M];
    int tile;
};

__device__ __forceinline__ void cvf_cp_async16(void *dst_smem, const void *src)
{
    unsigned int d = (unsigned int)__cvta_generic_to_shared(dst_smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void cvf_cp_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cvf_cp_wait_pipe()
{
    asm volatile("cp.async.wait_group %0;\n" ::"n"(CVF_STAGES - 2) : "memory");
}
__device__ __forceinline__ void cvf_cp_wait0() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

__device__ __forceinline__ void cvf_two_sum_acc(double &hi, double &lo, double x)
{
    cv_dd s = cv_two_sum(hi, x);
    hi = s.hi;
    lo = cv_add(lo, s.lo);
}

/* Four MMAs of one row tile (one A value, the four column tiles of the warp), skipped as a whole
 * when copy index kk is past the copies the 8 points of the row tile use.  The condition is the
 * same in every lane.  Written as a loop of zero or one trips: ptxas turns a plain branch into four
 * predicated MMAs, which still occupy the FP64 pipe when predicated off. */
__device__ __forceinline__ void cvf_dmma4_if(double *acc, double a, const double *b, int kk, int kend)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        ".reg .s32 n;\n"
        "sub.s32 n, %14, %13;\n"       /* > 0: the row tile still has copies */
        "min.s32 n, n, 1;\n"
        "CVF_LOOP:\n"
        "setp.le.s32 p, n, 0;\n"
        "@p bra CVF_DONE;\n"
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%8}, {%9}, {%0,%1};\n"
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%2,%3}, {%8}, {%10}, {%2,%3};\n"
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%4,%5}, {%8}, {%11}, {%4,%5};\n"
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%6,%7}, {%8}, {%12}, {%6,%7};\n"
        "sub.s32 n, n, 1;\n"
        "bra CVF_LOOP;\n"
        "CVF_DONE:\n"
        "}\n"
        : "+d"(acc[0]), "+d"(acc[1]), "+d"(acc[2]), "+d"(acc[3]), "+d"(acc[4]), "+d"(acc[5]), "+d"(acc[6]),
          "+d"(acc[7])
        : "d"(a), "d"(b[0]), "d"(b[1]), "d"(b[2]), "d"(b[3]), "r"(kk), "r"(kend));
}

/* The running copy weights of one point for the generator role of a thread: b(o) of
 * models.py:193-208 for the 8 copies of its half of a K-chunk, as a running product (relative
 * error below 1e-13 at o = 1000).  half 0 covers copies 16 kc + 1 .. + 8, half 1 the next eight. */
struct CvfWeights {
    double q1, two, many, base, b16, cur0, cur;
    int othr, half;
};

__device__ __forceinline__ void cvf_weights_chunk(CvfWeights &w, int kc, double *v)
{
    if (kc == 0)
        w.cur = w.cur0;
    if (kc == 0 && w.half == 0) {
        v[0] = w.q1;
        v[1] = w.two;
        v[2] = w.many;
#pragma unroll
        for (int i = 3; i < 8; i++)
            v[i] = cv_mul(v[i - 1], w.base);
    } else {
        v[0] = w.cur;
#pragma unroll
        for (int i = 1; i < 8; i++)
            v[i] = cv_mul(v[i - 1], w.base);
        w.cur = cv_mul(w.cur, w.b16);
    }
    const int o_first = kc * CVF_KC + 8 * w.half + 1;
#pragma unroll
    for (int i = 0; i < 8; i++)
        if (!(o_first + i < w.othr)) /* models.py:235: copies o < O_thr */
            v[i] = 0.0;
}

/* The MMAs of one K-chunk for the row tiles LO .. HI - 1 of a warp: 4 K slices x (HI - LO) row
 * tiles x 4 column tiles.  as2 / bs2 point at the lane's chunk of K slice 0. */
template <int LO, int HI>
__device__ __forceinline__ void cvf_chunk_mma(double *acc, const double2 *as2, const double2 *bs2)
{
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
        double a[4] = {0.0, 0.0, 0.0, 0.0};
        if (LO < 2) {
            const double2 a01 = as2[(ks * 2 + 0) * 32];
            a[0] = a01.x;
            a[1] = a01.y;
        }
        if (HI > 2) {
            const double2 a23 = as2[(ks * 2 + 1) * 32];
            a[2] = a23.x;
            a[3] = a23.y;
        }
        const double2 b01 = bs2[(ks * 2 + 0) * 32], b23 = bs2[(ks * 2 + 1) * 32];
        const double b[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int mt = LO; mt < HI; mt++)
#pragma unroll
            for (int nt = 0; nt < 4; nt++)
                cv_dmma(acc[(mt * 4 + nt) * 2], acc[(mt * 4 + nt) * 2 + 1], a[mt], b[nt]);
    }
}

/* Position (in doubles) inside a 128 x 16 tile of copy weights of (row p of the tile, copy index
 * k % 16): the order in which the warps of K2 read their A fragments,
 * [warp row wm][K slice][row-tile pair][lane = r * 4 + (k % 4 ^ swizzle)][row-tile parity].
 * Row tile J = p / 8 belongs to warp row wm = J % 4 as its tile mt = J / 4, so that every warp row
 * holds short and long rows of the sorted tile alike. */
__device__ __forceinline__ int cvf_a_index(int p, int kin)
{
    const int J = p >> 3, r = p & 7, wm = J & 3, mt = J >> 2;
    const int ks = kin >> 2, q = kin & 3;
    return ((((wm * 4 + ks) * 2 + (mt >> 1)) * 32 + r * 4 + (q ^ ((r >> 1) & 3))) * 2) + (mt & 1);
}

/* K1b: the copy weights b(o) of models.py:193-208 of every tile of K2, masked by o < O_thr
 * (models.py:235), written as ready-made A tiles.  One CTA per tile; thread (point, half) fills 8
 * copies of every K-chunk, the chunk leaves through shared memory as 16-byte stores. */
__global__ void __launch_bounds__(CVF_THREADS)
cvf_weights_kernel(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
                   const double *__restrict__ params, int clip, CvfPlan pl, int first_tile, int n_tiles,
                   double *__restrict__ A, long long a_base)
{
    __shared__ double2 stage[CVF_M * CVF_KC / 2];
    const int tid = threadIdx.x;
    const int tile = first_tile + blockIdx.x;
    if (blockIdx.x >= n_tiles)
        return;
    const int nkc = pl.t_nkc[tile];
    if (nkc == 0)
        return;
    const int pfirst = pl.t_first[tile], cnt = pl.t_cnt[tile];
    /* the 16 lanes of a half warp take the row tiles J and J + 4 (different halves of a 16-byte
     * chunk of the stage): conflict-free stores */
    const int warp = tid >> 5;
    const int gp = 8 * ((warp & 3) + 8 * (warp >> 2) + 4 * ((tid >> 3) & 1)) + (tid & 7), half = (tid >> 4) & 1;
    CvfWeights wg;
    wg.q1 = wg.two = wg.many = wg.base = 0.0;
    wg.othr = 0;
    wg.half = half;
    if (gp < cnt) {
        const unsigned int pi = pl.idx_sorted[pfirst + gp];
        double row[CV_MAX_PARAMS];
        cvf_raw_row(m, lat, params, pi, row);
        wg.q1 = cvf_clipped(m, row, clip, 2);
        const double q2 = cvf_clipped(m, row, clip, 3), qq = cvf_clipped(m, row, clip, 4);
        wg.two = cv_mul(cv_sub(1.0, wg.q1), q2);
        wg.many = cv_mul(cv_mul(cv_sub(1.0, wg.q1), cv_sub(1.0, q2)), qq);
        wg.base = cv_sub(1.0, qq);
        wg.othr = pl.othr[pi];
    }
    {
        const double b2 = cv_mul(wg.base, wg.base), b4 = cv_mul(b2, b2), b8 = cv_mul(b4, b4);
        wg.b16 = cv_mul(b8, b8);
        /* b(o) of the first copy of the thread's half in chunk 0 (half 1: o = 9, many base^6)
         * resp. chunk 1 (half 0: o = 17, many base^14) */
        wg.cur0 = half ? cv_mul(wg.many, cv_mul(b4, b2)) : cv_mul(wg.many, cv_mul(b8, cv_mul(b4, b2)));
        wg.cur = wg.cur0;
    }
    double2 *out = reinterpret_cast<double2 *>(A + ((long long)pl.t_aoff[tile] - a_base) * (CVF_M * CVF_KC));
    for (int kc = 0; kc < nkc; kc++) {
        double v[8];
        cvf_weights_chunk(wg, kc, v);
        double *st = reinterpret_cast<double *>(stage);
#pragma unroll
        for (int i = 0; i < 8; i++)
            st[cvf_a_index(gp, 8 * half + i)] = v[i];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; j++)
            out[(long long)kc * (CVF_M * CVF_KC / 2) + tid + j * CVF_THREADS] = stage[tid + j * CVF_THREADS];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(CVF_THREADS, 2)
cvf_gemm_kernel(const __grid_constant__ CvModelDesc m, CvfPlan pl, int first_tile, int n_tiles,
                const double *__restrict__ W, long long w_base, const double *__restrict__ A,
                long long a_base, const double2 *__restrict__ slot_mh, const int *__restrict__ step_mask,
                const double *__restrict__ log_tab, int nsteps, double *__restrict__ out_ll,
                unsigned long long *counter)
{
    extern __shared__ __align__(16) unsigned char cvf_smem_raw[];
    CvfSmem &S = *reinterpret_cast<CvfSmem *>(cvf_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp >> 1, wn = warp & 1;
    const int r = lane >> 2, q = lane & 3;
    const int apos = r * 4 + (q ^ ((r >> 1) & 3)); /* swizzled position of the lane's A chunk */
    for (int i = tid; i < 2 * CV_LOG_N; i += CVF_THREADS)
        S.log_tab[i] = log_tab[i];
    /* loader role: 16-byte chunks tid and tid + 256 of a profile tile ([copy][pair]) go to the
     * fragment order [N half][K slice][n-tile pair][lane = (column % 8) * 4 + copy % 4] */
    int b_dst[2];
    long long b_src[2]; /* double2 units from the first row of the K-chunk */
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const int i = tid + j * CVF_THREADS;
        const int oc = i >> 5, L = i & 31, row = L >> 3, rr = L & 7;
        b_dst[j] = (((row >> 1) * 4 + (oc >> 2)) * 2 + (row & 1)) * 32 + rr * 4 + (oc & 3);
        b_src[j] = (long long)oc * nsteps * (CVF_NS / 2) + L;
    }
    const bool want_mass = m.tail != 0.0;

    for (;;) {
        __syncthreads(); /* the previous tile's readers of shared memory are done */
        if (tid == 0)
            S.tile = (int)atomicAdd(counter, 1ULL);
        __syncthreads();
        if (S.tile >= n_tiles)
            break;
        const int tile = pl.t_sorted[S.tile]; /* longest tiles first */
        const int pfirst = pl.t_first[tile], cnt = pl.t_cnt[tile], nkc = pl.t_nkc[tile];
        const int g = pl.t_group[tile];
        if (tid < CVF_M) {
            unsigned int pi = 0;
            int othr = 0;
            if (tid < cnt) {
                pi = pl.idx_sorted[pfirst + tid];
                othr = pl.othr[pi];
            }
            S.othr[tid] = othr;
            S.pidx[tid] = pi;
        }
        __syncthreads();
        const double *Wg = W + (pl.w_off[g] - w_base);
        const double2 *Ag = reinterpret_cast<const double2 *>(A + ((long long)pl.t_aoff[tile] - a_base) * (CVF_M * CVF_KC));
        /* copies the 8 points of each of the warp's row tiles need (ascending: the last live one) */
        int kend[4];
#pragma unroll
        for (int mt = 0; mt < 4; mt++) {
            const int first = 8 * (4 * mt + wm);
            kend[mt] = first < cnt ? S.othr[min(first + 7, cnt - 1)] - 1 : 0;
        }
        const int kend_hi = max(max(kend[0], kend[1]), max(kend[2], kend[3]));
        int nlive = 0; /* row tiles of this warp row that hold points */
#pragma unroll
        for (int mt = 0; mt < 4; mt++)
            nlive += 8 * (4 * mt + wm) < cnt;

        int ld_kc = 0, ld_ns = 0, ld_buf = 0; /* the next (profile, weight) tile pair to request */
        auto issue = [&]() {
            if (ld_ns < nsteps) {
                /* 16 rows (copies) x one line of 64 slots: 16-byte chunk i = tid + 256 j is pair
                 * i % 32 of row i / 32 */
                const double2 *src = reinterpret_cast<const double2 *>(
                    Wg + ((long long)ld_kc * CVF_KC * nsteps + ld_ns) * CVF_NS);
                double2 *dst = S.Bs[ld_buf];
                cvf_cp_async16(dst + b_dst[0], src + b_src[0]);
                cvf_cp_async16(dst + b_dst[1], src + b_src[1]);
                const double2 *asrc = Ag + (long long)ld_kc * (CVF_M * CVF_KC / 2);
                double2 *adst = S.As[ld_buf];
#pragma unroll
                for (int j = 0; j < 4; j++)
                    cvf_cp_async16(adst + tid + j * CVF_THREADS, asrc + tid + j * CVF_THREADS);
                if (++ld_kc == nkc) {
                    ld_kc = 0;
                    ld_ns++;
                }
                ld_buf = ld_buf == CVF_STAGES - 1 ? 0 : ld_buf + 1;
            }
            cvf_cp_commit();
        };
        if (nkc == 0)
            ld_ns = nsteps; /* nothing to load */
#pragma unroll
        for (int i = 0; i < CVF_STAGES - 1; i++)
            issue();

        double sum[4] = {0.0, 0.0, 0.0, 0.0};
        double mass_h[4] = {0.0, 0.0, 0.0, 0.0}, mass_l[4] = {0.0, 0.0, 0.0, 0.0};
        int cons_buf = 0;
        for (int ns = 0; ns < nsteps; ns++) {
            double acc[32];
#pragma unroll
            for (int i = 0; i < 32; i++)
                acc[i] = 0.0;
            for (int kc = 0; kc < nkc; kc++, cons_buf = cons_buf == CVF_STAGES - 1 ? 0 : cons_buf + 1) {
                cvf_cp_wait_pipe();
                __syncthreads(); /* this chunk's tiles landed, the previous chunk is consumed */
                issue();
                const int k0 = kc * CVF_KC;
                if (k0 >= kend_hi)
                    continue;
                const double2 *as2 = S.As[cons_buf] + (wm * 4) * 2 * 32 + apos;
                const double2 *bs2 = S.Bs[cons_buf] + (wn * 4) * 2 * 32 + lane;
                /* row tiles lo .. nlive - 1 are still running (ascending copies along the sorted
                 * rows); when none of them ends inside this chunk the MMAs need no checks */
                int lo = 0;
                bool partial = false;
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
                    if (mt < nlive) {
                        const int rem = kend[mt] - k0;
                        lo += rem <= 0;
                        partial |= rem > 0 && rem < CVF_KC;
                    }
                if (!partial) {
                    switch (lo * 4 + nlive) {
                    case 0 * 4 + 4: cvf_chunk_mma<0, 4>(acc, as2, bs2); break;
                    case 1 * 4 + 4: cvf_chunk_mma<1, 4>(acc, as2, bs2); break;
                    case 2 * 4 + 4: cvf_chunk_mma<2, 4>(acc, as2, bs2); break;
                    case 3 * 4 + 4: cvf_chunk_mma<3, 4>(acc, as2, bs2); break;
                    case 0 * 4 + 3: cvf_chunk_mma<0, 3>(acc, as2, bs2); break;
                    case 1 * 4 + 3: cvf_chunk_mma<1, 3>(acc, as2, bs2); break;
                    case 2 * 4 + 3: cvf_chunk_mma<2, 3>(acc, as2, bs2); break;
                    case 0 * 4 + 2: cvf_chunk_mma<0, 2>(acc, as2, bs2); break;
                    case 1 * 4 + 2: cvf_chunk_mma<1, 2>(acc, as2, bs2); break;
                    case 0 * 4 + 1: cvf_chunk_mma<0, 1>(acc, as2, bs2); break;
                    default: break;
                    }
                } else {
                    const int nks = min(4, (kend_hi - k0 + 3) >> 2);
                    for (int ks = 0; ks < nks; ks++) {
                        const double2 a01 = as2[(ks * 2 + 0) * 32], a23 = as2[(ks * 2 + 1) * 32];
                        const double2 b01 = bs2[(ks * 2 + 0) * 32], b23 = bs2[(ks * 2 + 1) * 32];
                        const double a[4] = {a01.x, a01.y, a23.x, a23.y};
                        const double b[4] = {b01.x, b01.y, b23.x, b23.y};
                        const int kk = k0 + 4 * ks;
#pragma unroll
                        for (int mt = 0; mt < 4; mt++) /* row tiles whose points stop earlier hold zeros */
                            cvf_dmma4_if(acc + mt * 8, a[mt], b, kk, kend[mt]);
                    }
                }
            }
            /* epilogue of the N-step, models.py:100-107: the lane holds row r of its four row
             * tiles and slots 64 ns + 32 wn + 8 nt + 2 q + c; bit 2 nt + c of the step mask says
             * whether any of those four slots has a count */
            const int mask = want_mass ? 0xff : __ldg(step_mask + 2 * ns + wn);
            if (mask) {
#pragma unroll
                for (int nt = 0; nt < 4; nt++)
#pragma unroll
                    for (int c = 0; c < 2; c++) {
                        if (!((mask >> (2 * nt + c)) & 1))
                            continue;
                        const int slot = ns * CVF_NS + 32 * wn + 8 * nt + 2 * q + c;
                        const double2 mh = __ldg(slot_mh + slot);
                        const bool in_hist = mh.x != 0.0;
                        const bool counted = mh.y != 0.0; /* models.py:106 `if h` */
                        double p[4];
#pragma unroll
                        for (int mt = 0; mt < 4; mt++)
                            p[mt] = in_hist ? acc[(mt * 4 + nt) * 2 + c] : 0.0; /* K1 applied slot_mult */
                        if (want_mass) {
#pragma unroll
                            for (int mt = 0; mt < 4; mt++)
                                cvf_two_sum_acc(mass_h[mt], mass_l[mt], p[mt]);
                        }
                        if (__any_sync(CV_FULL_MASK, counted)) {
#pragma unroll
                            for (int mt = 0; mt < 4; mt++) {
                                /* utils.py:32-35 safe_log */
                                double lg = p[mt] >= CV_P_BAND ? cv_log_tab(p[mt], S.log_tab, CV_PSCALE_EXP)
                                                               : cv_log_scaled(p[mt]);
                                if (counted)
                                    sum[mt] = cv_add(sum[mt], cv_mul(mh.y, lg));
                            }
                        }
                    }
            }
        }
        cvf_cp_wait0();
        /* the four lanes of a quad hold different slots of the same points */
#pragma unroll
        for (int mt = 0; mt < 4; mt++) {
#pragma unroll
            for (int d = 1; d <= 2; d <<= 1) {
                sum[mt] = cv_add(sum[mt], __shfl_xor_sync(CV_FULL_MASK, sum[mt], d));
                if (want_mass) {
                    double oh = __shfl_xor_sync(CV_FULL_MASK, mass_h[mt], d);
                    double ol = __shfl_xor_sync(CV_FULL_MASK, mass_l[mt], d);
                    cvf_two_sum_acc(mass_h[mt], mass_l[mt], oh);
                    mass_l[mt] = cv_add(mass_l[mt], ol);
                }
            }
            if (q == 0) {
                const int pt = 8 * (4 * mt + wm) + r;
                S.red_sum[wn][pt] = sum[mt];
                S.red_mh[wn][pt] = mass_h[mt];
                S.red_ml[wn][pt] = mass_l[mt];
            }
        }
        __syncthreads();
        if (tid < cnt) {
            CvPartial part;
            part.sum = cv_add(S.red_sum[0][tid], S.red_sum[1][tid]);
            part.mass_h = S.red_mh[0][tid];
            part.mass_l = S.red_ml[0][tid];
            cvf_two_sum_acc(part.mass_h, part.mass_l, S.red_mh[1][tid]);
            part.mass_l = cv_add(part.mass_l, S.red_ml[1][tid]);
            out_ll[S.pidx[tid]] = cv_point_finish(m, part);
        }
    }
}

/* ------------------------------------------------------------------------------------------- */
/* K2p: prefix kernel                                                                           */
/* ------------------------------------------------------------------------------------------- */
/* The copy weights beyond o = 2 are geometric, b(o) = many * (1 - q)^(o - 3) (models.py:196-208), so
 * for points of a group that share q
 *
 *     p[j] = q1 P_1[j] + two P_2[j] + many * R_q(O_thr)[j],   R_q(O)[j] = sum_{3 <= o < O} (1 - q)^(o-3) P_o[j]
 *
 * and all cut-offs O_thr of such a *q-run* are served by ONE running sum over the copies: the
 * contraction over o is done once per q-run instead of once per point.  A CTA takes a tile (one
 * batch: up to CVF_NQ whole q-runs of a group with up to CVF_PB points; or a window of a longer
 * run).  Every thread owns SL slots per pass (template parameter, 3 or 4) and keeps the CVF_NQ running sums of its slots in
 * registers.  The points of the batch are put in the order of their cut-offs once (the *schedule*);
 * the threads then walk the copies upwards -- the profile of copy o travels through a private
 * cp.async ring, CVF_PD copies ahead -- and finish every point as soon as its copies are in: the
 * three-term combination for the thread's slots, models.py:100-107 per bin (log only for bins with
 * counts), the lane partials parked in a transpose buffer and summed over the lanes for CVF_PE points
 * at a time.  Values do not depend on what else is in the batch: a point's sums run over its own
 * copies and over the bins in a fixed order.
 *
 * Slots to threads: a CTA has NW warps (template parameter: 8 for rows of more than 768 slots, else
 * as many as it takes to cover the row in one pass -- histograms with few bins that have counts,
 * cvf_build_slots); a pass covers 32 * NW * SL slots = NW * SL half-lines (a line = the 64
 * doubles of one copy and one N-step in the layout of K1); warp w takes the half-lines
 * u = i * NW + w, i < SL, lane l the double l of each.  Bins with counts usually are the
 * first ones of the histogram, so this deals them evenly to the warps. */
#define CVF_WARPS_SM 16 /* warps per SM the register budget of the prefix kernel is cut for */
#define CVF_PD 4       /* copies in flight per thread (cp.async ring in shared memory) */
#define CVF_PL2 6      /* copies ahead of the ring that are requested into L2 */
#define CVF_PE 8       /* points whose lane partials wait in the transpose buffer of a warp (4: 1.45 ms on cfg3, 8: 1.35 ms) */
#define CVF_PEW 33    /* doubles per row of that buffer (odd: conflict-free both ways) */

struct __align__(16) CvfEvent {
    double q1, two, many;
    int info, need;
};

/* explicit shared-window accesses: the hot loop addresses its records, the logarithm table and the
 * transpose buffer with 32-bit addresses kept in registers */
/* a shared-window address the compiler must keep in a register: without this it re-derives the
 * window base (S2UR SR_CgaCtaId + ULEA) in front of every access of the hot loop */
__device__ __forceinline__ unsigned int cvf_pin(unsigned int a)
{
    unsigned int r;
    asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(a));
    return r;
}
__device__ __forceinline__ double2 cvf_lds128(unsigned int a)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void cvf_lds_event(unsigned int a, double &many, int &info, int &need)
{
    asm volatile("ld.shared.f64 %0, [%3+16];\n\tld.shared.v2.s32 {%1, %2}, [%3+24];"
                 : "=d"(many), "=r"(info), "=r"(need)
                 : "r"(a));
}
__device__ __forceinline__ void cvf_sts64(unsigned int a, double v)
{
    asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}

struct CvfPrefixSmem {
    double log_tab[2 * CV_LOG_N]; /* cv_log_table */
    /* the points of the batch by ascending cut-off (the schedule), 32 bytes each: weights of
     * copy 1, copy 2 and of the running sum; batch position | run << 16; copies = O_thr - 1 */
    CvfEvent ev[CVF_PB + 2];
    double base[CVF_NQ];
    int seg[CVF_NQ + 1]; /* batch positions where its q-runs start */
    int tile, bend;
    /* then, in this order:
     *   double ring[CVF_PD][SL][threads]   every thread's own slots of the copies in flight
     *   double tbuf[planes][warps][CVF_PE][CVF_PEW]   lane partials of the last points, per warp
     *                                           (while the schedule is built: int need[CVF_PB], the
     *                                           copies of the points by batch position)
     * planes = 1 (sum) or, with a tail, 3 (sum, mass high, mass low: compensated)
     * and in global memory, per CTA (L2-resident scratch):
     *   double red[planes][warps][CVF_PB]    per (warp, point) partial */
};
#define CVF_SMEM_HEAD ((sizeof(CvfPrefixSmem) + 127) & ~(size_t)127)

/* nw = warps of the CTA (the kernel's NW), sl = slots per thread and pass (its SL) */
static size_t cvf_prefix_smem_bytes(bool mass, int nw, int sl)
{
    const size_t planes = mass ? 3 : 1;
    return CVF_SMEM_HEAD + (size_t)CVF_PD * sl * 32 * nw * 8 +
           planes * (size_t)nw * CVF_PE * CVF_PEW * sizeof(double);
}

/* safe_log (utils.py:32-35) off the fast path: below the band limit (cvmodel.h CV_PSCALE), zero,
 * negative, infinite, NaN */
__device__ __noinline__ double cvf_log_rare(double x)
{
    return cv_log_scaled(x);
}

/* fast path of the logarithms: scaled probability in [2^-902, inf), i.e. p >= 2^-1030 (CV_P_BAND) */
#define CVF_FAST_LO ((1023 - 902) << 20)
#define CVF_FAST_SPAN (0x7ff00000u - (unsigned int)CVF_FAST_LO)

/* cv_log_tab's algorithm for positive normal x with the index arithmetic on the high word and the
 * table at the shared-window address `tab_s`; everything else takes cvf_log_rare.
 *
 * |r| <= 2^-8 on every table interval, so log1p(r) - r = r^2 (-1/2 + r/3 - r^2/4 + r^3/5) leaves
 * r^6/6 <= 5.9e-16: the logarithm is 9 FP64 instructions in four dependent steps -- k ln 2 + logc in
 * one FMA (|k| <= 1100: 0.3 ulp of the result from the rounded ln 2), hi + r, and the polynomial
 * joined by a last FMA.  Measured against logl over 4e7 arguments: relative error <= 9.3e-16 for
 * x < 0.6875 (every probability of a bin that is not ~1), absolute error <= 5.8e-16 on
 * [0.6875, 1.375); the count-weighted sum has a 1e-9 gate.  The coefficient 1/5 of r^5 is cut to 20
 * mantissa bits (it fits the immediate field of the FP64 instructions; error below 2^-58). */
/* the fast path of cvf_safe_log alone: x positive, normal, finite */
__device__ __forceinline__ double cvf_log_fast(double x, unsigned int tab_s)
{
    const int hi = __double2hiint(x);
    const int t = hi - (int)(CV_LOG_OFF >> 32);
    const double z = __hiloint2double(hi - (t & (int)0xfff00000), __double2loint(x));
    const double2 c = cvf_lds128(tab_s + ((t >> 9) & ((CV_LOG_N - 1) << 4))); /* (invc, logc) of interval (t >> 13) & 127 */
    const double r = cv_fma(z, c.x, -1.0);
    const double kd = (double)((t >> 20) - CV_PSCALE_EXP); /* log(x 2^-128) */
    const double r2 = cv_mul(r, r);
    const double a = cv_fma(r, 1.0 / 3.0, -0.5);
    const double b = cv_fma(r, 0x1.9999ap-3 /* 1/5 */, -0.25);
    const double hi_part = cv_fma(kd, 0x1.62e42fefa39efp-1, c.y);
    const double p = cv_fma(r2, b, a);
    return cv_fma(r2, p, cv_add(hi_part, r)); /* hi_part + r does not wait for the polynomial */
}

__device__ __forceinline__ double cvf_safe_log(double x, unsigned int tab_s)
{
    if ((unsigned int)(__double2hiint(x) - CVF_FAST_LO) >= CVF_FAST_SPAN)
        return cvf_log_rare(x);
    return cvf_log_fast(x, tab_s);
}

/* number of entries of the ascending a[0..n) that are < x (strict) resp. <= x */
__device__ __forceinline__ int cvf_count_below(const int *a, int n, int x, bool or_equal)
{
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const int v = a[mid];
        if (v < x || (or_equal && v == x))
            lo = mid + 1;
        else
            hi = mid;
    }
    return lo;
}

/* MASS: the histogram has a tail (models.py:103-104): the mass sum_j p_j enters the result through
 * 1 - mass and is summed compensated (the reference uses fsum).  Without a tail the tail term is
 * tail * log(1 - mass) = +-0 whenever it is formed: the mass is not formed at all, the result is the
 * count-weighted sum of logarithms, and the slots read are those of the lines with counts.
 * FULL: the slots are a multiple of a pass (32 NW SL), no thread ever idles in a pass.
 * ONE: the bins with counts all lie in the first of a thread's SL slots (histograms whose
 * counted bins are the first quarter of every pass): the code for the other slots' logarithms is
 * not even compiled in. */
template <bool MASS, bool FULL, bool ONE, int NW, int SL>
__global__ void __launch_bounds__(32 * NW, CVF_WARPS_SM / NW)
cvf_prefix_kernel(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
                  const double *__restrict__ params, int clip, CvfPlan pl, int first_tile, int n_tiles,
                  const double *__restrict__ W, long long w_base, const double2 *__restrict__ slot_mh,
                  const double *__restrict__ log_tab, int nsteps, int nslots, double *__restrict__ out_ll,
                  unsigned long long *counter, double *__restrict__ scratch)
{
    constexpr int PT_ = 32 * NW, PW_ = NW;          /* threads, warps */
    constexpr int PASS_ = PT_ * SL;             /* slots per pass */
    constexpr int RING_ = CVF_PD * SL * PT_ * 8; /* bytes */
    constexpr int TBUF_ = PW_ * CVF_PE * CVF_PEW;   /* doubles per plane */
    extern __shared__ __align__(16) unsigned char cvf_smem_raw[];
    CvfPrefixSmem &S = *reinterpret_cast<CvfPrefixSmem *>(cvf_smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double *ring = reinterpret_cast<double *>(cvf_smem_raw + CVF_SMEM_HEAD) + tid;
    double *tbuf = reinterpret_cast<double *>(cvf_smem_raw + CVF_SMEM_HEAD + RING_) +
                   warp * (CVF_PE * CVF_PEW); /* plane stride TBUF_ */
    /* by batch position: copies of the point; only while the schedule is built, in the place of the transpose buffers */
    int *need_s = reinterpret_cast<int *>(cvf_smem_raw + CVF_SMEM_HEAD + RING_);
    static_assert(TBUF_ * 8 >= CVF_PB * 4, "the transpose buffers hold the cut-offs of a batch");
    double *red_all = scratch + (size_t)blockIdx.x * (3 * PW_ * CVF_PB);
    double *red = red_all + warp * CVF_PB; /* plane stride PW_ * CVF_PB */
    const unsigned int ring_s = cvf_pin((unsigned int)__cvta_generic_to_shared(ring));
    const unsigned int log_s = cvf_pin((unsigned int)__cvta_generic_to_shared(S.log_tab));
    const unsigned int ev_s = cvf_pin((unsigned int)__cvta_generic_to_shared(S.ev));
    const unsigned int tbuf_s = cvf_pin((unsigned int)__cvta_generic_to_shared(tbuf + lane)); /* the lane's column */
    for (int i = tid; i < 2 * CV_LOG_N; i += PT_)
        S.log_tab[i] = log_tab[i];
    /* nslots: the slots of a row that can be other than zero (a multiple of 32; the line of the sums ends after its first half) */
    const long long row_stride = (long long)nsteps * CVF_NS; /* doubles between the rows of consecutive copies */

    for (;;) {
        __syncthreads();
        if (tid == 0)
            S.tile = (int)atomicAdd(counter, 1ULL);
        __syncthreads();
        if (S.tile >= n_tiles)
            break;
        const int tile = pl.t_sorted[S.tile];
        const int tfirst = pl.t_first[tile], tend = tfirst + pl.t_cnt[tile];
        const double *Wg = W + (pl.w_off[pl.t_group[tile]] - w_base);

        for (int b0 = tfirst; b0 < tend;) {
            /* ---- the batch: up to CVF_PB points in up to CVF_NQ q-runs ---- */
            const int nload = min(CVF_PB, tend - b0);
            const int rid0 = pl.rid[b0];
            if (tid == 0)
                S.bend = nload;
            if (tid <= CVF_NQ)
                S.seg[tid] = nload;
            __syncthreads();
            for (int t = tid; t < nload; t += PT_) {
                const int rel = pl.rid[b0 + t] - rid0;
                if (rel >= CVF_NQ)
                    atomicMin(&S.bend, t);
                else if (t == 0 || pl.head2[b0 + t])
                    S.seg[rel] = t;
            }
            __syncthreads();
            const int npts = S.bend;
            /* per point: its copies */
            for (int t = tid; t < npts; t += PT_) {
                const unsigned int pi = pl.idx_sorted[b0 + t];
                need_s[t] = pl.othr[pi] - 1;
                if (t == 0 || pl.head2[b0 + t]) {
                    double row[CV_MAX_PARAMS];
                    cvf_raw_row(m, lat, params, pi, row);
                    S.base[pl.rid[b0 + t] - rid0] = cv_sub(1.0, cvf_clipped(m, row, clip, 4));
                }
            }
            __syncthreads();
            int seg0[CVF_NQ], seg_end[CVF_NQ], last_need[CVF_NQ];
            double base[CVF_NQ];
            int omax_b = 0; /* copies the batch needs: cut-offs ascend inside a q-run */
#pragma unroll
            for (int s = 0; s < CVF_NQ; s++) {
                seg0[s] = min(S.seg[s], npts);
                seg_end[s] = s + 1 < CVF_NQ ? min(S.seg[s + 1], npts) : npts;
                if (seg_end[s] < seg0[s])
                    seg_end[s] = seg0[s];
                base[s] = seg_end[s] > seg0[s] ? S.base[s] : 0.0;
                last_need[s] = seg_end[s] > seg0[s] ? need_s[seg_end[s] - 1] : -1;
                omax_b = max(omax_b, last_need[s]);
            }
            /* the schedule: rank of a point = points before it by (copies, run, position) */
            for (int t = tid; t < npts; t += PT_) {
                const int need = need_s[t];
                int rank = 0, mine = 0;
#pragma unroll
                for (int s = 0; s < CVF_NQ; s++)
                    if (t >= seg0[s] && t < seg_end[s]) {
                        mine = s;
                        rank += t - seg0[s];
                    }
#pragma unroll
                for (int s = 0; s < CVF_NQ; s++)
                    if (s != mine && seg_end[s] > seg0[s])
                        rank += cvf_count_below(need_s + seg0[s], seg_end[s] - seg0[s], need, s < mine);
                double row[CV_MAX_PARAMS];
                cvf_raw_row(m, lat, params, pl.idx_sorted[b0 + t], row);
                const double q1 = cvf_clipped(m, row, clip, 2), q2 = cvf_clipped(m, row, clip, 3),
                             qq = cvf_clipped(m, row, clip, 4);
                CvfEvent e;
                /* copies beyond the cut-off do not enter (models.py:235): exact zero weights (the
                 * profiles are probabilities, finite) */
                e.q1 = need >= 1 ? q1 : 0.0;
                e.two = need >= 2 ? cv_mul(cv_sub(1.0, q1), q2) : 0.0;
                e.many = need >= 3 ? cv_mul(cv_mul(cv_sub(1.0, q1), cv_sub(1.0, q2)), qq) : 0.0;
                e.info = t | (mine << 16);
                e.need = need;
                S.ev[rank] = e;
            }
            if (tid < 2) { /* read ahead by the loop below, never used */
                CvfEvent e;
                e.q1 = e.two = e.many = 0.0;
                e.info = e.need = 0;
                S.ev[npts + tid] = e;
            }
            __syncthreads();

            /* ---- passes over the slots ---- */
            for (int pass0 = 0; pass0 < nslots; pass0 += PASS_) {
                /* the thread's slots: double `lane` of the half-lines u = pass0 / 32 + i * PW_ + warp */
                const int u0 = (pass0 >> 5) + warp;
                const double *src0 = Wg + u0 * 32 + lane; /* row 0 (copy 1) */
                constexpr long long SRC_STEP = (long long)PW_ * 32; /* doubles between i and i + 1 */
                double hcnt[SL];
                int log_mask = 0;
                bool live[SL];
#pragma unroll
                for (int i = 0; i < SL; i++) {
                    const int u = u0 + i * PW_;
                    live[i] = FULL || u * 32 < nslots;
                    const int e = (u & 1) * 32 + lane, L = e >> 1; /* pair L, member e & 1 of N-step u / 2 */
                    const int slot = (u >> 1) * CVF_NS + 16 * (L >> 3) + (L & 7) + 8 * (e & 1);
                    hcnt[i] = live[i] ? __ldg(&slot_mh[slot].y) : 0.0;
                    log_mask |= (__any_sync(CV_FULL_MASK, hcnt[i] != 0.0) ? 1 : 0) << i;
                }
                /* The profile of copy o for the thread's slots: copy o lives at (o - 1) / 16 chunks +
                 * (o - 1) % 16 lines of 64 doubles.  Copies travel through the thread's own places
                 * of a ring in shared memory (cp.async, CVF_PD copies in flight, nothing to
                 * synchronise between threads); further ahead they are requested into L2. */
                const bool wide = !ONE && log_mask == (1 << SL) - 1; /* measured: also taking masks with one slot less gains nothing */
                /* are the values of two points in all of the thread's slots with counts on the fast path of the logarithm? */
                auto pair_fast = [&](const double *pa, const double *pb) {
                    unsigned int worst = 0;
#pragma unroll
                    for (int i = 0; i < SL; i++) {
                        const unsigned int ca = (unsigned int)(__double2hiint(pa[i]) - CVF_FAST_LO),
                                           cb = (unsigned int)(__double2hiint(pb[i]) - CVF_FAST_LO);
                        if (hcnt[i] != 0.0)
                            worst = max(worst, max(ca, cb));
                    }
                    return worst < CVF_FAST_SPAN;
                };
                int o_req = 1;                 /* the next copy to request */
                unsigned int dst_req = ring_s; /* its place in the ring */
                const double *src_req = src0;  /* its first slot */
                const double *src_far = src0 + (long long)CVF_PL2 * row_stride;
                const bool far_lane = (lane & 15) == 0; /* one request per 128-byte line */
                auto request = [&]() { /* one commit group per call, also when there is nothing left to load */
                    if (o_req <= omax_b) {
#pragma unroll
                        for (int i = 0; i < SL; i++)
                            if (live[i])
                                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst_req + i * PT_ * 8),
                                             "l"(src_req + i * SRC_STEP)
                                             : "memory");
                        if (o_req + CVF_PL2 <= omax_b && far_lane) {
#pragma unroll
                            for (int i = 0; i < SL; i++)
                                if (live[i])
                                    asm volatile("prefetch.global.L2 [%0];" ::"l"(src_far + i * SRC_STEP));
                        }
                    }
                    cvf_cp_commit();
                    src_req += row_stride;
                    src_far += row_stride;
                    dst_req = (o_req % CVF_PD == 0) ? ring_s : dst_req + SL * PT_ * 8;
                    o_req++;
                };
                int slot_take = 0;
                auto take = [&](double *x) { /* the oldest copy in flight has landed */
                    asm volatile("cp.async.wait_group %0;\n" ::"n"(CVF_PD - 1) : "memory");
#pragma unroll
                    for (int i = 0; i < SL; i++) {
                        double v;
                        asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(ring_s + (unsigned int)((slot_take * SL + i) * PT_ * 8)));
                        x[i] = live[i] ? v : 0.0;
                    }
                    slot_take = slot_take == CVF_PD - 1 ? 0 : slot_take + 1;
                };
#pragma unroll
                for (int o = 1; o <= CVF_PD; o++)
                    request();
                double P1[SL], P2[SL];
#pragma unroll
                for (int i = 0; i < SL; i++)
                    P1[i] = P2[i] = 0.0;
                if (omax_b >= 1) {
                    take(P1);
                    request();
                }
                if (omax_b >= 2) {
                    take(P2);
                    request();
                }
                double R[CVF_NQ][SL], w[CVF_NQ];
#pragma unroll
                for (int s = 0; s < CVF_NQ; s++) {
#pragma unroll
                    for (int i = 0; i < SL; i++)
                        R[s][i] = 0.0;
                    w[s] = 1.0;
                }
                const bool first_pass = pass0 == 0;
                int pending = 0; /* points in the transpose buffer */
                int mypt = 0;    /* lane e: the point in row e of the buffer */
                /* row e of the buffer summed over the 32 lane partials (32 / CVF_PE columns per lane,
                 * then across the lane groups): fixed order, the warp's partial of that point */
                auto flush = [&]() {
                    __syncwarp();
                    /* lane group g = lane / CVF_PE takes the columns g * CVF_PE .. + CVF_PE - 1 of row e */
                    const int e = lane & (CVF_PE - 1), c0 = (lane / CVF_PE) * CVF_PE;
                    const double *rowp = tbuf + e * CVF_PEW + c0;
                    double acc0 = rowp[0], acc1 = 0.0, acc2 = 0.0;
                    if (MASS) {
                        acc1 = rowp[TBUF_];
                        acc2 = rowp[2 * TBUF_];
                    }
#pragma unroll
                    for (int c = 1; c < CVF_PE; c++) {
                        acc0 = cv_add(acc0, rowp[c]);
                        if (MASS) { /* high parts exactly (two-sum), low parts plainly */
                            cvf_two_sum_acc(acc1, acc2, rowp[TBUF_ + c]);
                            acc2 = cv_add(acc2, rowp[2 * TBUF_ + c]);
                        }
                    }
#pragma unroll
                    for (int d = CVF_PE; d <= 16; d <<= 1) {
                        acc0 = cv_add(acc0, __shfl_xor_sync(CV_FULL_MASK, acc0, d));
                        if (MASS) {
                            const double oh = __shfl_xor_sync(CV_FULL_MASK, acc1, d);
                            const double ol = __shfl_xor_sync(CV_FULL_MASK, acc2, d);
                            cvf_two_sum_acc(acc1, acc2, oh);
                            acc2 = cv_add(acc2, ol);
                        }
                    }
                    const int pt = __shfl_sync(CV_FULL_MASK, mypt, e);
                    if (lane < pending) {
                        double *r0 = red + pt, *r1 = r0 + PW_ * CVF_PB, *r2 = r1 + PW_ * CVF_PB;
                        if (first_pass) {
                            *r0 = acc0;
                            if (MASS) {
                                *r1 = acc1;
                                *r2 = acc2;
                            }
                        } else {
                            *r0 = cv_add(*r0, acc0);
                            if (MASS) {
                                double h = *r1, l = *r2;
                                cvf_two_sum_acc(h, l, acc1);
                                *r1 = h;
                                *r2 = cv_add(l, acc2);
                            }
                        }
                    }
                    pending = 0;
                    __syncwarp();
                };
                int o_done = 2;
                unsigned int ev_a = ev_s; /* the record of the point after the current one */
                double q1, two, many;
                int info, need;
                {
                    const double2 qt = cvf_lds128(ev_a);
                    q1 = qt.x;
                    two = qt.y;
                    cvf_lds_event(ev_a, many, info, need);
                }
                unsigned int tb_a = tbuf_s; /* row `pending` of the transpose buffer */
                auto step = [&]() { /* one more copy into the running sums (o_done >= 3 afterwards) */
                    o_done++;
                    double x[SL];
                    take(x);
                    request();
#pragma unroll
                    for (int s = 0; s < CVF_NQ; s++)
                        if (o_done <= last_need[s]) { /* runs whose points are all out need no more copies */
#pragma unroll
                            for (int i = 0; i < SL; i++)
                                R[s][i] = cv_fma(w[s], x[i], R[s][i]);
                            w[s] = cv_mul(w[s], base[s]);
                        }
                };
                for (int k = 0; k < npts; k++) {
                    /* the next point's record travels while this one is worked on */
                    ev_a += (unsigned int)sizeof(CvfEvent);
                    const double2 qt_next = cvf_lds128(ev_a);
                    double many_next;
                    int info_next, need_next;
                    cvf_lds_event(ev_a, many_next, info_next, need_next);
                    while (o_done < need)
                        step();
                    if (k + 1 < npts) {
                        /* two points at once: this one is combined now, the next one after the copies
                         * it still needs; then their logarithms run side by side (two dependent
                         * chains instead of one) and the bookkeeping is shared */
                        double pa[SL], pb[SL];
#pragma unroll
                        for (int i = 0; i < SL; i++)
                            pa[i] = cv_fma(two, P2[i], cv_mul(q1, P1[i]));
                        switch ((info >> 16) & 3) {
#define CVF_CASE(s_)                                                                                   \
    case s_:                                                                                           \
        _Pragma("unroll") for (int i = 0; i < SL; i++) pa[i] = cv_fma(many, R[s_][i], pa[i]);      \
        break;
                            CVF_CASE(0)
                            CVF_CASE(1)
                            CVF_CASE(2)
                            CVF_CASE(3)
#undef CVF_CASE
                        }
                        while (o_done < need_next)
                            step();
#pragma unroll
                        for (int i = 0; i < SL; i++)
                            pb[i] = cv_fma(qt_next.y, P2[i], cv_mul(qt_next.x, P1[i]));
                        switch ((info_next >> 16) & 3) {
#define CVF_CASE(s_)                                                                                   \
    case s_:                                                                                           \
        _Pragma("unroll") for (int i = 0; i < SL; i++) pb[i] = cv_fma(many_next, R[s_][i], pb[i]); \
        break;
                            CVF_CASE(0)
                            CVF_CASE(1)
                            CVF_CASE(2)
                            CVF_CASE(3)
#undef CVF_CASE
                        }
                        const int pt_a = info & 0xffff, pt_b = info_next & 0xffff;
                        /* the record after the pair becomes the current one */
                        ev_a += (unsigned int)sizeof(CvfEvent);
                        {
                            const double2 qt = cvf_lds128(ev_a);
                            q1 = qt.x;
                            two = qt.y;
                            cvf_lds_event(ev_a, many, info, need);
                        }
                        k++;
                        double ma = 0.0, mb = 0.0, mla = 0.0, mlb = 0.0; /* models.py:103: the mass */
                        if (MASS) {
#pragma unroll
                            for (int i = 0; i < SL; i++) {
                                cvf_two_sum_acc(ma, mla, pa[i]);
                                cvf_two_sum_acc(mb, mlb, pb[i]);
                            }
                        }
                        double sa = 0.0, sb = 0.0;
                        if (ONE ? log_mask != 0 : log_mask == 1) { /* the usual case: only the warp's first half-line has counts */
                            const unsigned int ca = (unsigned int)(__double2hiint(pa[0]) - CVF_FAST_LO),
                                               cb = (unsigned int)(__double2hiint(pb[0]) - CVF_FAST_LO);
                            double la, lb;
                            if (ca < CVF_FAST_SPAN && cb < CVF_FAST_SPAN) { /* both on the fast path */
                                la = cvf_log_fast(pa[0], log_s);
                                lb = cvf_log_fast(pb[0], log_s);
                            } else {
                                la = cvf_safe_log(pa[0], log_s);
                                lb = cvf_safe_log(pb[0], log_s);
                            }
                            sa = cv_mul(hcnt[0], la);
                            sb = cv_mul(hcnt[0], lb);
                            if (hcnt[0] == 0.0) /* models.py:106 `if h` */
                                sa = sb = 0.0;
                        } else if (wide && pair_fast(pa, pb)) {
                            /* counts in all of the warp's half-lines (rows that keep only the
                             * lines with counts) and this thread's values all on the fast path: the 2 SL
                             * logarithms side by side, nothing between them to branch on; what they make
                             * of a slot without a count is not used */
#pragma unroll
                            for (int i = 0; i < SL; i++) {
                                const double la = cvf_log_fast(pa[i], log_s),
                                             lb = cvf_log_fast(pb[i], log_s);
                                double ta = cv_mul(hcnt[i], la), tb = cv_mul(hcnt[i], lb);
                                if (hcnt[i] == 0.0)
                                    ta = tb = 0.0;
                                sa = cv_add(sa, ta);
                                sb = cv_add(sb, tb);
                            }
                        } else if (!ONE && log_mask) {
#pragma unroll
                            for (int i = 0; i < SL; i++)
                                if ((log_mask >> i) & 1) { /* some lane of the warp has a count in its slot i */
                                    const unsigned int ca = (unsigned int)(__double2hiint(pa[i]) - CVF_FAST_LO),
                                                       cb = (unsigned int)(__double2hiint(pb[i]) - CVF_FAST_LO);
                                    double la, lb;
                                    if (ca < CVF_FAST_SPAN && cb < CVF_FAST_SPAN) {
                                        la = cvf_log_fast(pa[i], log_s);
                                        lb = cvf_log_fast(pb[i], log_s);
                                    } else {
                                        la = cvf_safe_log(pa[i], log_s);
                                        lb = cvf_safe_log(pb[i], log_s);
                                    }
                                    double ta = cv_mul(hcnt[i], la), tb = cv_mul(hcnt[i], lb);
                                    if (hcnt[i] == 0.0)
                                        ta = tb = 0.0;
                                    sa = cv_add(sa, ta);
                                    sb = cv_add(sb, tb);
                                }
                        }
                        if (pending == CVF_PE - 1) { /* no room for two rows */
                            flush();
                            tb_a = tbuf_s;
                        }
                        cvf_sts64(tb_a, sa);
                        cvf_sts64(tb_a + CVF_PEW * 8, sb);
                        if (MASS) {
                            cvf_sts64(tb_a + TBUF_ * 8, ma);
                            cvf_sts64(tb_a + CVF_PEW * 8 + TBUF_ * 8, mb);
                            cvf_sts64(tb_a + 2 * TBUF_ * 8, mla);
                            cvf_sts64(tb_a + CVF_PEW * 8 + 2 * TBUF_ * 8, mlb);
                        }
                        tb_a += 2 * CVF_PEW * 8;
                        if (lane == pending)
                            mypt = pt_a;
                        if (lane == pending + 1)
                            mypt = pt_b;
                        pending += 2;
                        if (pending == CVF_PE) {
                            flush();
                            tb_a = tbuf_s;
                        }
                        continue;
                    }
                    /* the three-term combination for the thread's slots, models.py:235-241 */
                    const int pt = info & 0xffff;
                    double p[SL];
#pragma unroll
                    for (int i = 0; i < SL; i++)
                        p[i] = cv_fma(two, P2[i], cv_mul(q1, P1[i]));
                    switch ((info >> 16) & 3) {
#define CVF_CASE(s_)                                                                                   \
    case s_:                                                                                           \
        _Pragma("unroll") for (int i = 0; i < SL; i++) p[i] = cv_fma(many, R[s_][i], p[i]);        \
        break;
                        CVF_CASE(0)
                        CVF_CASE(1)
                        CVF_CASE(2)
                        CVF_CASE(3)
#undef CVF_CASE
                    }
                    q1 = qt_next.x;
                    two = qt_next.y;
                    many = many_next;
                    info = info_next;
                    need = need_next;
                    /* models.py:100-107 for the thread's slots */
                    double sum = 0.0, mh = 0.0, ml = 0.0;
                    if (MASS) {
#pragma unroll
                        for (int i = 0; i < SL; i++)
                            cvf_two_sum_acc(mh, ml, p[i]);
                    }
                    if (ONE ? log_mask != 0 : log_mask == 1) { /* the usual case: the warp's first half-line holds the bins with counts */
                        double term = cv_mul(hcnt[0], cvf_safe_log(p[0], log_s)); /* utils.py:32-35 */
                        if (hcnt[0] == 0.0) /* models.py:106 `if h` */
                            term = 0.0;
                        sum = term;
                    } else if (!ONE && log_mask) {
#pragma unroll
                        for (int i = 0; i < SL; i++)
                            if ((log_mask >> i) & 1) { /* some lane of the warp has a count in its slot i */
                                double term = cv_mul(hcnt[i], cvf_safe_log(p[i], log_s));
                                if (hcnt[i] == 0.0)
                                    term = 0.0;
                                sum = cv_add(sum, term);
                            }
                    }
                    cvf_sts64(tb_a, sum);
                    if (MASS) {
                        cvf_sts64(tb_a + TBUF_ * 8, mh);
                        cvf_sts64(tb_a + 2 * TBUF_ * 8, ml);
                    }
                    tb_a += CVF_PEW * 8;
                    if (lane == pending)
                        mypt = pt;
                    if (++pending == CVF_PE) {
                        flush();
                        tb_a = tbuf_s;
                    }
                }
                if (pending)
                    flush();
                cvf_cp_wait0();
            }
            __syncthreads();
            for (int t = tid; t < npts; t += PT_) {
                CvPartial part;
                part.sum = red_all[t];
                part.mass_h = MASS ? red_all[PW_ * CVF_PB + t] : 0.0;
                part.mass_l = MASS ? red_all[2 * PW_ * CVF_PB + t] : 0.0;
                for (int wv = 1; wv < PW_; wv++) {
                    part.sum = cv_add(part.sum, red_all[wv * CVF_PB + t]);
                    if (MASS) {
                        cvf_two_sum_acc(part.mass_h, part.mass_l, red_all[(PW_ + wv) * CVF_PB + t]);
                        part.mass_l = cv_add(part.mass_l, red_all[(2 * PW_ + wv) * CVF_PB + t]);
                    }
                }
                out_ll[pl.idx_sorted[b0 + t]] = MASS ? cv_point_finish(m, part) : part.sum;
            }
            b0 += npts;
            __syncthreads();
        }
    }
}

/* ------------------------------------------------------------------------------------------- */
/* host side                                                                                    */
/* ------------------------------------------------------------------------------------------- */
void cvf_release(CvFactorWork &wk)
{
    if (wk.plan)
        cudaFree(wk.plan);
    if (wk.W)
        cudaFree(wk.W);
    if (wk.h_header)
        cudaFreeHost(wk.h_header);
    if (wk.d_counters)
        cudaFree(wk.d_counters);
    if (wk.d_scratch)
        cudaFree(wk.d_scratch);
    wk.d_scratch = nullptr;
    if (wk.lattice.dev)
        cudaFree(wk.lattice.dev);
    if (wk.lattice.pinned)
        cudaFreeHost(wk.lattice.pinned);
    if (wk.lattice.uploaded)
        cudaEventDestroy(wk.lattice.uploaded);
    wk.lattice = CvfLatticeCache();
    for (cudaEvent_t &e : wk.ev)
        if (e) {
            cudaEventDestroy(e);
            e = nullptr;
        }
    wk.plan = nullptr;
    wk.W = nullptr;
    wk.h_header = nullptr;
    wk.d_counters = nullptr;
    wk.plan_cap = wk.w_cap = 0;
}

static size_t cvf_align(size_t x) { return (x + 255) & ~(size_t)255; }

#define CVF_CK(call)              \
    do {                          \
        cudaError_t e_ = (call);  \
        if (e_ != cudaSuccess)    \
            return e_;            \
    } while (0)

/* ---- the template of a lattice's groups, on the host ---- */
static double cvf_host_clip(const CvModelDesc &m, double v, int clip, int a)
{
    return clip ? cv_clip(v, m.lo[a], m.hi[a]) : v;
}

static void cvf_lattice_template(const CvModelDesc &m, int clip, const double *q1v, int n1, const double *q2v,
                                 int n2, const double *qv, int nq, CvfLatticeCache &T)
{
    const int R = n1 * n2, M = R * nq;
    T.M = M;
    T.R = R;
    T.nq = nq;
    /* runs in ascending order of the clipped q (NaN first), as the sort key of the general plan
     * orders them: neighbours then need about the same number of copies */
    std::vector<int> qorder(nq);
    std::vector<double> qc(nq);
    for (int i = 0; i < nq; i++) {
        qorder[i] = i;
        const double v = cvf_host_clip(m, qv[i], clip, 4);
        qc[i] = v > 0.0 ? (v < 1.0 ? v : 1.0) : 0.0;
    }
    std::stable_sort(qorder.begin(), qorder.end(), [&](int a, int b) { return qc[a] < qc[b]; });
    std::vector<int> perm(M), othr(M);
    std::vector<std::pair<int, int>> run(R); /* (cut-off, lattice offset) */
    int omax = 0;
    for (int r = 0; r < nq; r++) {
        const int iq = qorder[r];
        const double q = cvf_host_clip(m, qv[iq], clip, 4);
        const double base = cv_sub(1.0, q);
        for (int i1 = 0; i1 < n1; i1++) {
            const double q1 = cvf_host_clip(m, q1v[i1], clip, 2);
            for (int i2 = 0; i2 < n2; i2++) {
                const double q2 = cvf_host_clip(m, q2v[i2], clip, 3);
                const double two = cv_mul(cv_sub(1.0, q1), q2);                          /* models.py:195 */
                const double many = cv_mul(cv_mul(cv_sub(1.0, q1), cv_sub(1.0, q2)), q); /* models.py:196 */
                run[i1 * n2 + i2] = std::make_pair(cvf_cutoff(m, q1, two, many, base), (i1 * n2 + i2) * nq + iq);
            }
        }
        std::stable_sort(run.begin(), run.end(),
                         [](const std::pair<int, int> &a, const std::pair<int, int> &b) { return a.first < b.first; });
        for (int t = 0; t < R; t++) {
            othr[r * R + t] = run[t].first;
            perm[r * R + t] = run[t].second;
            omax = std::max(omax, run[t].first - 1);
        }
    }
    T.omax = omax;
    /* tiles: cvf_prefix_tiles over runs of R points each */
    std::vector<int> tf, tc, tk;
    for (int r = 0; r < nq;) {
        const int first = r * R, rfirst = r;
        int end = first, runs = 0;
        while (r < nq && runs < CVF_NQ) {
            const int re = (r + 1) * R;
            if (runs > 0 && re - first > CVF_PB)
                break;
            end = re;
            r++;
            runs++;
        }
        for (int p = first; p < end; p += CVF_PSPLIT) {
            const int cnt = std::min(CVF_PSPLIT, end - p);
            int kmax = 0;
            for (int rr = rfirst; rr < rfirst + runs; rr++) {
                const int last = std::min((rr + 1) * R, p + cnt) - 1;
                if (last >= p && last >= rr * R)
                    kmax = std::max(kmax, othr[last] - 1);
            }
            tf.push_back(p);
            tc.push_back(cnt);
            tk.push_back(kmax);
        }
    }
    const int nT = (int)tf.size();
    T.nT = nT;
    std::vector<int> order(nT);
    for (int i = 0; i < nT; i++)
        order[i] = i;
    std::stable_sort(order.begin(), order.end(),
                     [&](int a, int b) { return 4 * tc[a] + 3 * tk[a] > 4 * tc[b] + 3 * tk[b]; });
    T.host.clear();
    T.host.insert(T.host.end(), perm.begin(), perm.end());
    T.host.insert(T.host.end(), othr.begin(), othr.end());
    T.host.insert(T.host.end(), tf.begin(), tf.end());
    T.host.insert(T.host.end(), tc.begin(), tc.end());
    T.host.insert(T.host.end(), tk.begin(), tk.end());
    T.host.insert(T.host.end(), order.begin(), order.end());
}

/* Can the batch be planned from its axes?  Points i of a group must be consecutive lattice indices
 * starting at a multiple of M = |q1| |q2| |q|. */
static bool cvf_lattice_aligned(const CvModelDesc &m, const CvLattice &lat, long long n, long long *M_out)
{
    if (!lat.enabled || lat.n_axes != 5 || m.n_param != 5)
        return false;
    const long long M = (long long)lat.len[2] * lat.len[3] * lat.len[4];
    *M_out = M;
    if (M <= 0 || M > 0x7fffffffLL || n % M)
        return false;
    if (lat.block % M == 0)
        return true;
    return lat.block == 1 && lat.stride == 1 && lat.first % M == 0;
}

cudaError_t cvf_eval(const CvModelDesc &m, const CvLattice &lat, const double *const *lat_axes_host,
                     const double *params, long long n,
                     int clip, double *out_ll, const CvfSlots &sl,
                     const double *log_tab, CvFactorWork &wk, int n_sm, int smem_max, size_t w_limit,
                     double min_group, double min_run, int kernel_mode, cudaStream_t stream,
                     int *used)
{
    *used = 0;
    wk.launches = 0;
    if (n <= 0 || n > 0x7fffffffLL || !cvf_supported(m))
        return cudaSuccess;
    /* the slots of a profile row as the batch kernels see them (cvf_build_slots) */
    const int nsteps = sl.nsteps;
    const int slots_padded = nsteps * CVF_NS;
    const double2 *slot_mh = sl.slot_mh;
    const int *step_mask = sl.step_mask;

    /* ---- carve the plan ---- */
    size_t sort_tmp = 0, sort_tmp_t = 0, scan_tmp_i = 0, scan_tmp_l = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (unsigned long long *)nullptr,
                                    (unsigned long long *)nullptr, (unsigned int *)nullptr,
                                    (unsigned int *)nullptr, (int)n, 0, 64, stream);
    cub::DeviceRadixSort::SortPairsDescending(nullptr, sort_tmp_t, (int *)nullptr, (int *)nullptr,
                                              (int *)nullptr, (int *)nullptr, (int)n, 0, 32, stream);
    cub::DeviceScan::InclusiveSum(nullptr, scan_tmp_i, (unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                  (int)n + 1, stream);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp_l, (long long *)nullptr, (long long *)nullptr,
                                  (int)n + 1, stream);
    const size_t tmp_bytes = std::max(std::max(sort_tmp, sort_tmp_t), std::max(scan_tmp_i, scan_tmp_l)) + 256;
    const size_t n1 = (size_t)n + 1;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t at = off;
        off += cvf_align(bytes);
        return at;
    };
    const size_t o_keys = take(n * 8), o_keys_alt = take(n * 8), o_idx = take(n * 4), o_idx_alt = take(n * 4);
    const size_t o_othr = take(n * 4), o_head = take(n * 4), o_gid = take(n * 4);
    const size_t o_head2 = take(n * 4), o_rid = take(n * 4), o_gomax = take(n1 * 4);
    const size_t o_rstart = take(n1 * 4), o_grfirst = take(n1 * 4), o_flags2 = take(n * 8);
    const size_t o_gstart = take(n1 * 4), o_tile = take(n1 * 4), o_item = take(n1 * 4), o_woff = take(n1 * 8);
    const size_t o_astart = take(n1 * 4);
    size_t o_t[9];
    for (size_t &o : o_t)
        o = take(n1 * 4);
    const size_t o_header = take(64), o_tmp = take(tmp_bytes);
    if (off > wk.plan_cap) {
        if (wk.plan)
            cudaFree(wk.plan);
        wk.plan = nullptr;
        wk.plan_cap = 0;
        CVF_CK(cudaMalloc(&wk.plan, off));
        wk.plan_cap = off;
    }
    if (!wk.h_header)
        CVF_CK(cudaMallocHost((void **)&wk.h_header, 64));
    if (!wk.d_counters)
        CVF_CK(cudaMalloc((void **)&wk.d_counters, 2 * sizeof(unsigned long long)));
    /* the CTAs of the prefix kernel own a scratch of partials each: at most 32 warps per SM */
    if (!wk.d_scratch)
        CVF_CK(cudaMalloc((void **)&wk.d_scratch, (size_t)n_sm * 32 * 3 * CVF_PB * sizeof(double)));
    if (wk.timed && !wk.ev[0])
        for (cudaEvent_t &e : wk.ev)
            CVF_CK(cudaEventCreate(&e));
    unsigned char *base = (unsigned char *)wk.plan;
    CvfPlan pl;
    pl.keys = (unsigned long long *)(base + o_keys);
    pl.keys_alt = (unsigned long long *)(base + o_keys_alt);
    pl.idx = (unsigned int *)(base + o_idx);
    pl.idx_alt = (unsigned int *)(base + o_idx_alt);
    pl.idx_sorted = nullptr;
    pl.othr = (int *)(base + o_othr);
    pl.head = (int *)(base + o_head);
    pl.gid = (int *)(base + o_gid);
    pl.head2 = (int *)(base + o_head2);
    pl.rid = (int *)(base + o_rid);
    pl.g_omax = (int *)(base + o_gomax);
    pl.flags2 = (unsigned long long *)(base + o_flags2);
    pl.r_start = (int *)(base + o_rstart);
    pl.g_rfirst = (int *)(base + o_grfirst);
    pl.g_start = (int *)(base + o_gstart);
    pl.tile_start = (int *)(base + o_tile);
    pl.item_start = (int *)(base + o_item);
    pl.w_off = (long long *)(base + o_woff);
    pl.a_start = (int *)(base + o_astart);
    pl.t_first = (int *)(base + o_t[0]);
    pl.t_cnt = (int *)(base + o_t[1]);
    pl.t_nkc = (int *)(base + o_t[2]);
    pl.t_aoff = (int *)(base + o_t[3]);
    pl.t_group = (int *)(base + o_t[4]);
    pl.t_key = (int *)(base + o_t[5]);
    pl.t_key_alt = (int *)(base + o_t[6]);
    pl.t_order = (int *)(base + o_t[7]);
    pl.t_order_alt = (int *)(base + o_t[8]);
    pl.t_sorted = nullptr;
    pl.header = (long long *)(base + o_header);
    pl.obits = 1;
    while ((1 << pl.obits) <= m.max_bin + CV_COPY_PAD)
        pl.obits++;
    void *tmp = base + o_tmp;

    const int tb = 256;
    const unsigned int nb = (unsigned int)((n + tb - 1) / tb), nb1 = (unsigned int)((n + 1 + tb - 1) / tb);
    if (wk.timed)
        CVF_CK(cudaEventRecord(wk.ev[0], stream));

    /* K0 .. totals for one ordering of the points; ends with the header on the host */
    auto build_plan = [&](int prefix) -> cudaError_t {
        pl.prefix = prefix;
        pl.tile_points = CVF_M;
        pl.keys = (unsigned long long *)(base + o_keys);
        pl.keys_alt = (unsigned long long *)(base + o_keys_alt);
        pl.idx = (unsigned int *)(base + o_idx);
        pl.idx_alt = (unsigned int *)(base + o_idx_alt);
        cvf_point_keys<<<nb, tb, 0, stream>>>(m, lat, params, n, clip, pl);
        CVF_CK(cudaGetLastError());
        {
            cub::DoubleBuffer<unsigned long long> dk(pl.keys, pl.keys_alt);
            cub::DoubleBuffer<unsigned int> dv(pl.idx, pl.idx_alt);
            size_t tb_ = tmp_bytes;
            CVF_CK(cub::DeviceRadixSort::SortPairs(tmp, tb_, dk, dv, (int)n, 0, 64, stream));
            pl.idx_sorted = dv.Current();
        }
        cvf_heads<<<nb, tb, 0, stream>>>(m, lat, params, n, clip, pl);
        CVF_CK(cudaGetLastError());
        {
            size_t tb_ = tmp_bytes;
            CVF_CK(cub::DeviceScan::InclusiveSum(tmp, tb_, pl.flags2, pl.flags2, (int)n, stream));
        }
        CVF_CK(cudaMemsetAsync(pl.g_omax, 0, n1 * sizeof(int), stream));
        cvf_group_starts<<<nb, tb, 0, stream>>>(n, pl);
        CVF_CK(cudaGetLastError());
        cvf_group_counts<<<nb1, tb, 0, stream>>>(n, slots_padded, pl);
        CVF_CK(cudaGetLastError());
        cvf_group_scan<<<1, 1024, 0, stream>>>(pl);
        CVF_CK(cudaGetLastError());
        CVF_CK(cudaMemcpyAsync(wk.h_header, pl.header, 6 * sizeof(long long), cudaMemcpyDeviceToHost, stream));
        CVF_CK(cudaStreamSynchronize(stream));
        wk.launches += 17; /* K0, radix sort (10), heads, one scan (2), starts, counts, group scan */
        return cudaSuccess;
    };
    /* ---- a lattice handed over as axes: the plan follows from the axes (no sort, no sync) ---- */
    int prefix = kernel_mode != 1;
    long long latM = 0;
    bool analytic = false;
    CvfLatticeDev TD;
    memset(&TD, 0, sizeof(TD));
    long long n_groups = 0, n_tiles = 0, n_items = 0, w_total = 0, a_total = 0;
    if (prefix && lat_axes_host && cvf_lattice_aligned(m, lat, n, &latM) && (double)latM >= min_group &&
        (double)(lat.len[2] * (long long)lat.len[3]) >= (kernel_mode == 0 ? min_run : 1.0)) {
        CvfLatticeCache &T = wk.lattice;
        const int n1 = lat.len[2], n2 = lat.len[3], nq = lat.len[4];
        std::vector<double> key;
        key.reserve(4 + n1 + n2 + nq);
        key.push_back((double)clip);
        key.push_back((double)n1);
        key.push_back((double)n2);
        key.push_back((double)nq);
        key.insert(key.end(), lat_axes_host[2], lat_axes_host[2] + n1);
        key.insert(key.end(), lat_axes_host[3], lat_axes_host[3] + n2);
        key.insert(key.end(), lat_axes_host[4], lat_axes_host[4] + nq);
        const bool same = key.size() == T.key.size() && T.dev &&
                          memcmp(key.data(), T.key.data(), key.size() * sizeof(double)) == 0;
        if (!same) {
            cvf_lattice_template(m, clip, lat_axes_host[2], n1, lat_axes_host[3], n2, lat_axes_host[4], nq, T);
            const size_t ints = T.host.size();
            if (ints > T.dev_cap) {
                if (T.dev)
                    cudaFree(T.dev);
                T.dev = nullptr;
                T.dev_cap = 0;
                CVF_CK(cudaMalloc((void **)&T.dev, ints * sizeof(int)));
                T.dev_cap = ints;
            }
            if (!T.uploaded)
                CVF_CK(cudaEventCreateWithFlags(&T.uploaded, cudaEventDisableTiming));
            else
                CVF_CK(cudaEventSynchronize(T.uploaded)); /* the staging buffer is free again */
            if (ints > T.pinned_cap) {
                if (T.pinned)
                    cudaFreeHost(T.pinned);
                T.pinned = nullptr;
                T.pinned_cap = 0;
                CVF_CK(cudaMallocHost((void **)&T.pinned, ints * sizeof(int)));
                T.pinned_cap = ints;
            }
            memcpy(T.pinned, T.host.data(), ints * sizeof(int));
            T.key.clear(); /* not valid until the copy is enqueued */
            CVF_CK(cudaMemcpyAsync(T.dev, T.pinned, ints * sizeof(int), cudaMemcpyHostToDevice, stream));
            CVF_CK(cudaEventRecord(T.uploaded, stream));
            T.key = key;
        }
        const int M = T.M, nT = T.nT;
        const int G = (int)(n / M);
        const int items = (T.omax + CVF_KC - 1) / CVF_KC;
        const long long wpg = (long long)items * CVF_KC * slots_padded;
        TD.perm = T.dev;
        TD.othr = T.dev + M;
        TD.tt_first = T.dev + 2 * (size_t)M;
        TD.tt_cnt = TD.tt_first + nT;
        TD.tt_kmax = TD.tt_cnt + nT;
        TD.tt_order = TD.tt_kmax + nT;
        pl.prefix = 1;
        pl.tile_points = CVF_M;
        pl.idx_sorted = pl.idx;
        const long long work = std::max<long long>(n, (long long)G * T.nq + 1);
        cvf_lattice_fill<<<(unsigned int)((work + tb - 1) / tb), tb, 0, stream>>>(pl, TD, G, M, T.R, T.nq, nT, T.omax,
                                                                                items, wpg);
        CVF_CK(cudaGetLastError());
        wk.launches += 1;
        analytic = true;
        n_groups = G;
        n_tiles = (long long)G * nT;
        n_items = (long long)G * items;
        w_total = (long long)G * wpg;
        a_total = 0;
        wk.n_groups = G;
        wk.n_runs = (long long)G * T.nq;
    }
    wk.analytic = analytic ? 1 : 0;
    if (!analytic) {
        /* ordering for the prefix kernel first: it also tells how many q-runs the batch has */
        CVF_CK(build_plan(prefix));
        wk.n_groups = wk.h_header[0];
        wk.n_runs = wk.h_header[5];
        if (wk.n_groups <= 0 || (double)n < min_group * (double)wk.n_groups)
            return cudaSuccess; /* too little sharing: the per-point kernel is the better tool */
        if (prefix && kernel_mode == 0 && (double)n < min_run * (double)wk.n_runs) {
            prefix = 0; /* few points per q-run: the GEMM shares the profiles between all points of a group */
            CVF_CK(build_plan(0));
        }
        n_groups = wk.h_header[0];
        n_tiles = wk.h_header[1];
        n_items = wk.h_header[2];
        w_total = wk.h_header[3];
        a_total = wk.h_header[4];
        cvf_tile_table<<<(unsigned int)((n_groups + 127) / 128), 128, 0, stream>>>((int)n_groups, pl);
        CVF_CK(cudaGetLastError());
        wk.launches++;
    }
    wk.n_tiles = n_tiles;
    wk.n_items = n_items;
    wk.w_doubles = w_total;
    wk.prefix = prefix;

    /* ---- group ranges whose profiles fit the workspace ---- */
    std::vector<int> cut; /* group boundaries */
    cut.push_back(0);
    std::vector<int> h_tile, h_item, h_achunk;
    std::vector<long long> h_woff;
    if ((size_t)w_total > w_limit) {
        h_tile.resize(n_groups + 1);
        h_item.resize(n_groups + 1);
        h_achunk.resize(n_groups + 1);
        h_woff.resize(n_groups + 1);
        if (analytic) { /* every group has the same tiles, items and profile size */
            for (long long g = 0; g <= n_groups; g++) {
                h_tile[g] = (int)(g * (n_tiles / n_groups));
                h_item[g] = (int)(g * (n_items / n_groups));
                h_achunk[g] = 0;
                h_woff[g] = g * (w_total / n_groups);
            }
        } else {
        CVF_CK(cudaMemcpyAsync(h_tile.data(), pl.tile_start, (n_groups + 1) * 4, cudaMemcpyDeviceToHost, stream));
        CVF_CK(cudaMemcpyAsync(h_item.data(), pl.item_start, (n_groups + 1) * 4, cudaMemcpyDeviceToHost, stream));
        CVF_CK(cudaMemcpyAsync(h_achunk.data(), pl.a_start, (n_groups + 1) * 4, cudaMemcpyDeviceToHost, stream));
        CVF_CK(cudaMemcpyAsync(h_woff.data(), pl.w_off, (n_groups + 1) * 8, cudaMemcpyDeviceToHost, stream));
        CVF_CK(cudaStreamSynchronize(stream));
        }
        int g0 = 0;
        while (g0 < n_groups) {
            int g1 = g0 + 1;
            while (g1 < n_groups && (size_t)(h_woff[g1 + 1] - h_woff[g0]) <= w_limit)
                g1++;
            cut.push_back(g1);
            g0 = g1;
        }
    } else {
        cut.push_back((int)n_groups);
    }
    const bool ranged = !h_woff.empty();
    size_t w_need = 0, a_need = 0;
    for (size_t i = 0; i + 1 < cut.size(); i++) {
        const long long wa = ranged ? h_woff[cut[i]] : 0, wb_ = ranged ? h_woff[cut[i + 1]] : w_total;
        const long long aa = ranged ? h_achunk[cut[i]] : 0, ab = ranged ? h_achunk[cut[i + 1]] : a_total;
        w_need = std::max(w_need, (size_t)(wb_ - wa));
        a_need = std::max(a_need, (size_t)(ab - aa) * (CVF_M * CVF_KC));
    }
    if (w_need + a_need > wk.w_cap) { /* profiles, then the copy-weight tiles */
        if (wk.W)
            cudaFree(wk.W);
        wk.W = nullptr;
        wk.w_cap = 0;
        CVF_CK(cudaMalloc((void **)&wk.W, std::max(w_need + a_need, (size_t)2) * sizeof(double)));
        wk.w_cap = w_need + a_need;
    }
    double *A = wk.W + w_need;
    if (wk.poison) { /* tests: what this evaluation reads of W and the partials, it must have written first */
        CVF_CK(cudaMemsetAsync(wk.W, wk.poison, (w_need + a_need) * sizeof(double), stream));
        CVF_CK(cudaMemsetAsync(wk.d_scratch, wk.poison, (size_t)n_sm * 32 * 3 * CVF_PB * sizeof(double), stream));
    }

    /* ---- K1, then K1b + K2 or the prefix kernel, per range ---- */
    const size_t wb = cv_warp_bytes(m.n_err);
    const int groups_staged = m.n_blocks * CV_GB;
    const size_t tab = (size_t)groups_staged * CV_GD * sizeof(double);
    const size_t wb1 = wb + CVF_STAGE_DOUBLES * sizeof(double); /* working set + profile stage */
    int k1_warps = (int)std::min<long long>(CV_WARPS_MAX, ((long long)smem_max - (long long)tab) / (long long)wb1);
    if (k1_warps < 1)
        return cudaErrorInvalidConfiguration;
    const size_t k1_smem = tab + (size_t)k1_warps * wb1;
    const bool want_mass = m.tail != 0.0;
    /* warps of the prefix kernel's CTAs: one pass over the row when 768 slots or fewer do it */
    /* The line of the sums is half a line with a tail and not read without one -- except when no line
     * has a count: then its first half (zeros, written by K1) is read, so that every point's sum is
     * formed by a pass (0, models.py:106) and the epilogue reads partials this launch wrote. */
    const int kp_slots = slots_padded - (sl.sum_line >= 0 ? (want_mass || nsteps == 1 ? 32 : CVF_NS) : 0);
    /* Geometry of the prefix kernel: warps per CTA and slots per thread so that one pass covers the
     * row when 32 half-lines or fewer do it -- the fewest warps, then the fewest slots (measured on
     * the 9 half-lines of cfg3 with a mass: 3 warps x 3 slots 0.82 ms, 3 x 4 0.91 ms; on its 8 half-lines
     * without one: 2 x 4 0.685 ms, 3 x 3 0.745 ms) */
    const int kp_half = kp_slots / 32;
    int kp_nw = 8, kp_sl = 4;
    if (kp_half <= 24) {
        static const int nws[] = {1, 2, 3, 4, 6, 8};
        int n3 = 8, n4 = 8;
        for (int i = 5; i >= 0; i--) {
            if (nws[i] * 3 >= kp_half && nws[i] != 4 && nws[i] != 8)
                n3 = nws[i];
            if (nws[i] * 4 >= kp_half)
                n4 = nws[i];
        }
        if (n3 <= n4) {
            kp_nw = n3;
            kp_sl = 3;
        } else {
            kp_nw = n4;
        }
    }
    const size_t kp_smem = cvf_prefix_smem_bytes(want_mass, kp_nw, kp_sl);
    const bool full_passes = kp_slots % (8 * 32 * 4) == 0;
    const bool counts_first = sl.counts_first;
    typedef decltype(&cvf_prefix_kernel<true, true, true, 8, 4>) CvfPrefixFn;
    CvfPrefixFn kp = nullptr;
    const bool full_one = kp_slots == kp_nw * 32 * kp_sl; /* the one pass of a small geometry has no idle thread */
#define CVF_PICK(nw_, sl_)                                                                                          \
    (full_one ? (want_mass ? cvf_prefix_kernel<true, true, false, nw_, sl_> : cvf_prefix_kernel<false, true, false, nw_, sl_>) \
              : (want_mass ? cvf_prefix_kernel<true, false, false, nw_, sl_> : cvf_prefix_kernel<false, false, false, nw_, sl_>))
    switch (kp_nw * 10 + kp_sl) {
    case 13: kp = CVF_PICK(1, 3); break;
    case 14: kp = CVF_PICK(1, 4); break;
    case 23: kp = CVF_PICK(2, 3); break;
    case 24: kp = CVF_PICK(2, 4); break;
    case 33: kp = CVF_PICK(3, 3); break;
    case 34: kp = CVF_PICK(3, 4); break;
    case 44: kp = CVF_PICK(4, 4); break;
    case 63: kp = CVF_PICK(6, 3); break;
    case 64: kp = CVF_PICK(6, 4); break;
    default:
        kp = want_mass ? (full_passes ? (counts_first ? cvf_prefix_kernel<true, true, true, 8, 4> : cvf_prefix_kernel<true, true, false, 8, 4>)
                                      : (counts_first ? cvf_prefix_kernel<true, false, true, 8, 4> : cvf_prefix_kernel<true, false, false, 8, 4>))
                       : (full_passes ? (counts_first ? cvf_prefix_kernel<false, true, true, 8, 4> : cvf_prefix_kernel<false, true, false, 8, 4>)
                                      : (counts_first ? cvf_prefix_kernel<false, false, true, 8, 4> : cvf_prefix_kernel<false, false, false, 8, 4>));
    }
#undef CVF_PICK
    CVF_CK(cudaFuncSetAttribute(cvf_profile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1_smem));
    CVF_CK(cudaFuncSetAttribute(cvf_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)sizeof(CvfSmem)));
    CVF_CK(cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kp_smem));
    if (wk.timed)
        CVF_CK(cudaEventRecord(wk.ev[1], stream));
    for (size_t i = 0; i + 1 < cut.size(); i++) {
        const int g0 = cut[i], g1 = cut[i + 1];
        const int item0 = ranged ? h_item[g0] : 0, item1 = ranged ? h_item[g1] : (int)n_items;
        const int tile0 = ranged ? h_tile[g0] : 0, tile1 = ranged ? h_tile[g1] : (int)n_tiles;
        const long long w0 = ranged ? h_woff[g0] : 0;
        const long long a0 = ranged ? h_achunk[g0] : 0;
        CVF_CK(cudaMemsetAsync(wk.d_counters, 0, 2 * sizeof(unsigned long long), stream));
        if (item1 > item0) {
            const int items = item1 - item0;
            int grid = (items + k1_warps - 1) / k1_warps;
            if (grid > n_sm)
                grid = n_sm;
            cvf_profile_kernel<<<grid, 32 * k1_warps, k1_smem, stream>>>(
                m, lat, params, clip, pl, (int)n_groups, item0, items, wk.W, w0, nsteps, sl.line_map, sl.sum_line,
                wk.d_counters, groups_staged);
            CVF_CK(cudaGetLastError());
            wk.launches++;
        }
        if (tile1 > tile0) {
            const int tiles = tile1 - tile0;
            if (!prefix) {
                cvf_weights_kernel<<<tiles, CVF_THREADS, 0, stream>>>(m, lat, params, clip, pl, tile0, tiles, A, a0);
                CVF_CK(cudaGetLastError());
                wk.launches++;
            }
            /* tiles of the range by descending cost: the long ones start first */
            if (analytic) {
                cvf_lattice_order<<<(unsigned int)((tiles + tb - 1) / tb), tb, 0, stream>>>(
                    TD, g0, g1, (int)(n_tiles / n_groups), pl.t_order_alt + tile0);
                CVF_CK(cudaGetLastError());
                pl.t_sorted = pl.t_order_alt + tile0;
            } else {
                cub::DoubleBuffer<int> dk(pl.t_key + tile0, pl.t_key_alt + tile0);
                cub::DoubleBuffer<int> dv(pl.t_order + tile0, pl.t_order_alt + tile0);
                size_t tb_ = tmp_bytes;
                CVF_CK(cub::DeviceRadixSort::SortPairsDescending(tmp, tb_, dk, dv, tiles, 0, 32, stream));
                pl.t_sorted = dv.Current();
            }
            if (wk.timed && i + 2 == cut.size())
                CVF_CK(cudaEventRecord(wk.ev[2], stream));
            int grid = tiles < 2 * n_sm ? tiles : 2 * n_sm;
            if (prefix) {
                const int per_sm = std::max(1, std::min(CVF_WARPS_SM / kp_nw, (int)((size_t)smem_max / (kp_smem + 1024))));
                grid = tiles < per_sm * n_sm ? tiles : per_sm * n_sm;
                kp<<<grid, 32 * kp_nw, kp_smem, stream>>>(m, lat, params, clip, pl, tile0, tiles, wk.W, w0, slot_mh,
                                                           log_tab, nsteps, kp_slots, out_ll, wk.d_counters + 1,
                                                           wk.d_scratch);
            } else {
                cvf_gemm_kernel<<<grid, CVF_THREADS, sizeof(CvfSmem), stream>>>(
                    m, pl, tile0, tiles, wk.W, w0, A, a0, slot_mh, step_mask, log_tab, nsteps, out_ll,
                    wk.d_counters + 1);
            }
            CVF_CK(cudaGetLastError());
            wk.launches += 2;
        }
    }
    if (wk.timed)
        CVF_CK(cudaEventRecord(wk.ev[3], stream));
    *used = prefix ? 2 : 1;
    return cudaSuccess;
}
