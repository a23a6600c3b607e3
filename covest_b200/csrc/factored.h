/*
 * factored.h -- the batched ("factored") evaluation of the repeats model: launch interface between
 * the C ABI (capi.cu) and factored.cu.
 *
 * The reference evaluates p_j = sum_o b(o) * [sum_s a_os * tp(o*l_s, j)] (models.py:235-241).  The
 * bracket -- the *profile* of copy number o -- depends on (coverage, error rate) only, the weight
 * b(o) on (q1, q2, q) only (models.py:193-208).  A batch of parameter points (an initial grid, a
 * grid-search round, the stencils of a multi-start refinement) holds few distinct (c, e) pairs and
 * many (q1, q2, q) per pair, so the batch is evaluated as
 *
 *   K0  per point: clip (models.py:60-69), cut-off O_thr (models.py:185-191), a sort key
 *       (hash of (c, e), O_thr); radix sort; groups = runs of equal (c, e), ascending O_thr inside
 *   K1  per group and copy number o <= max O_thr of the group: the profile over all bins, with the
 *       machinery of the per-point kernel (cvpoint.h), written to HBM in the fragment order K2 reads
 *   K2  per tile of 128 points of one group: P[point][bin] = sum_o b_point(o) * profile[o][bin] as a
 *       dense FP64 GEMM on the tensor cores (m8n8k4), copy weights from K1b,
 *       then the epilogue of models.py:100-107 straight from the accumulators
 *   K2p (instead of K1b + K2 when points of a group also share q, as lattices do): b(o) is geometric
 *       beyond o = 2, so one running sum over the copies per q-run serves all its cut-offs; per
 *       point only the three-term combination and the epilogue remain
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "kernels.h"

/* The template of a lattice's groups (factored.cu, "The plan of a lattice"): computed on the host
 * from the (q1, q2, q) axes, kept until the axes change, mirrored on the device. */
struct CvfLatticeCache {
    std::vector<double> key; /* clip flag, axis lengths and values the template was made from */
    std::vector<int> host;   /* perm[M], othr[M], then tt_first, tt_cnt, tt_kmax, tt_order [nT each] */
    int M = 0, R = 0, nq = 0, nT = 0, omax = 0;
    int *dev = nullptr;
    size_t dev_cap = 0;      /* ints */
    int *pinned = nullptr;   /* staging of the upload */
    size_t pinned_cap = 0;
    cudaEvent_t uploaded = nullptr; /* the last upload has left the staging buffer */
};

/* The sizes of a batch's plan in the order of its header on the device: groups, tiles, profile items,
 * profile doubles, K-chunks of copy weights, q-runs */
struct CvfSizes { long long groups, tiles, items, w_doubles, a_chunks, runs; };

struct CvFactorWork {
    unsigned char *plan = nullptr; /* sort keys, indices, group tables, cub scratch */
    size_t plan_cap = 0;
    double *W = nullptr;  /* profiles */
    size_t w_cap = 0;     /* doubles */
    CvfSizes *h_sizes = nullptr; /* pinned host: the sizes the general plan counted */
    unsigned long long *d_counters = nullptr; /* two device words */
    double *d_scratch = nullptr; /* prefix kernel: per CTA the per-(warp, point) partials of a batch */
    /* timing of the most recent evaluation (events recorded when `timed`) */
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool timed = false;
    /* facts about the most recent evaluation */
    long long n_groups = 0, n_tiles = 0, n_items = 0, w_doubles = 0, n_runs = 0;
    int launches = 0;
    int analytic = 0; /* 1: the plan came from the lattice axes (no sort, no host synchronisation) */
    int poison = 0;   /* tests (COVEST_B200_POISON): byte W and d_scratch are filled with at each evaluation, 0 = off */
    CvfLatticeCache lattice;
};

/* The slots of a profile row as the batch kernels (K1's stores, K2, K2p) see them.
 *
 * The histogram tables (cvtables.h) lay the bins out in lines of 64 slots.  A bin without a count
 * enters the log-likelihood only through the mass sum_j p_j (models.py:103-107), and p_j is linear
 * in the profiles: sum over such bins of p_j = sum_o b(o) * (sum over such bins of P_o[j]).  So a
 * profile row keeps the lines that hold at least one bin with a count as they are, and ONE more line
 * whose first half holds the sums of all other lines (32 partial sums per copy, one per lane of the
 * warp that stores the row; its second half is zero).  With a tail every profile value is evaluated
 * by K1 and is part of the mass.  Without a tail the mass does not enter the result: K1 evaluates the
 * row tables (cv_build_row_tables: the lines with counts only), writes the line of the sums as zeros
 * and K2p does not read it.  Histograms simulated or counted to a fixed max_hist are mostly zero
 * beyond a few multiples of the coverage: cfg3 keeps 4 + 1 of its 16 lines. */
struct CvfSlots {
    int nsteps = 0;                /* lines of a row */
    int sum_line = -1;             /* the line of the sums, -1: every line has counts */
    const int *line_map = nullptr; /* device: line of the histogram tables -> line of the row, -1: summed */
    const double2 *slot_mh = nullptr; /* device: (slot_mult or 1 on the sum line, count) per slot of the row */
    const int *step_mask = nullptr;   /* device: cvf_step_masks of those counts */
    bool counts_first = false;        /* cvf_counts_first of those counts */
};

/* host: the row layout for the tables (slot_mult, slot_h), both of the same length, a multiple of
 * 64.  compact = false keeps every line (the layout before this existed; COVEST_B200_ROWS=full).
 * sums = true adds the line of the sums even when every line of these tables has a count (row tables,
 * whose histogram tables have lines without counts). */
static inline void cvf_build_slots(const std::vector<double> &slot_mult, const std::vector<double> &slot_h,
                                   bool compact, bool sums, std::vector<int> &line_map, std::vector<double2> &mh,
                                   std::vector<double> &row_h, int *sum_line)
{
    const size_t lines = slot_h.size() / 64;
    line_map.assign(lines, -1);
    mh.clear();
    row_h.clear();
    int kept = 0;
    for (size_t l = 0; l < lines; l++) {
        bool counts = !compact;
        for (int i = 0; i < 64 && !counts; i++)
            counts = slot_h[l * 64 + i] != 0.0;
        if (!counts)
            continue;
        line_map[l] = kept++;
        for (int i = 0; i < 64; i++) {
            double2 v;
            v.x = slot_mult[l * 64 + i];
            v.y = slot_h[l * 64 + i];
            mh.push_back(v);
            row_h.push_back(v.y);
        }
    }
    *sum_line = -1;
    if ((size_t)kept < lines || sums) {
        *sum_line = kept;
        for (int i = 0; i < 64; i++) {
            double2 v;
            v.x = 1.0; /* a slot of the histogram as far as K2 is concerned */
            v.y = 0.0;
            mh.push_back(v);
            row_h.push_back(0.0);
        }
    }
}

/* Can this context use the factored path at all (repeats model, few enough error classes)? */
bool cvf_supported(const CvModelDesc &m);

/* What cvf_eval is asked to run: path mode 0, 2, 3 or 4 of cvb_set_path (Forced: the batched path
 * however few points share a group, the kernel as in Auto) */
enum class CvfRequest { Auto, Forced, Gemm, Prefix };
/* What it ran.  None: the batch does not group well enough (nothing written to out_ll) */
enum class CvfRan { None, Gemm, Prefix };

/* Evaluates n points.  sl: the row layout (CvfSlots).  `log_tab` = cv_log_table.  w_limit = largest
 * profile workspace in doubles; larger batches run in several group ranges.  lat_axes_host: the
 * lattice axes in host memory (n_param pointers) when lat.enabled, else NULL. */
cudaError_t cvf_eval(const CvModelDesc &m, const CvLattice &lat, const double *const *lat_axes_host,
                     const double *params, long long n, int clip, double *out_ll, const CvfSlots &sl,
                     const double *log_tab, CvFactorWork &wk, int n_sm, int smem_max, size_t w_limit,
                     CvfRequest req, cudaStream_t stream, CvfRan *ran);

/* host: the geometry of the prefix kernel (warps per CTA, slots per thread and pass) for rows of
 * `half_lines` half-lines of 32 slots: one pass covers the row when 32 half-lines or fewer do it --
 * the fewest warps, then the fewest slots (measured on the 9 half-lines of cfg3 with a mass: 3 warps
 * x 3 slots 0.82 ms, 3 x 4 0.91 ms; on its 8 half-lines without one: 2 x 4 0.685 ms, 3 x 3
 * 0.745 ms).  Longer rows take 8 x 4, in several passes beyond 32 half-lines.  Only these
 * geometries are instantiated: 3 slots with 1, 2, 3 or 6 warps, 4 slots with 1, 2, 3, 4, 6 or 8. */
struct CvfPrefixGeometry { int nw, sl; };
static inline CvfPrefixGeometry cvf_prefix_geometry(int half_lines)
{
    if (half_lines > 24)
        return {8, 4};
    static const int nws[] = {1, 2, 3, 4, 6, 8};
    int n3 = 8, n4 = 8;
    for (int i = 5; i >= 0; i--) {
        if (nws[i] * 3 >= half_lines && nws[i] != 4 && nws[i] != 8)
            n3 = nws[i];
        if (nws[i] * 4 >= half_lines)
            n4 = nws[i];
    }
    if (n3 <= n4)
        return {n3, 3};
    return {n4, 4};
}

/* A range of consecutive groups whose profiles fit the workspace, with its bounds in the plan's
 * prefix tables: tiles, profile items, profile doubles, K-chunks of copy weights */
struct CvfRange {
    int g0, g1, tile0, tile1, item0, item1; /* groups g0 .. g1 - 1 */
    long long w0, w1, a0, a1;
};

/* host: groups 0 .. n - 1 cut into ranges whose profiles take at most w_limit doubles each, or one
 * group alone when it takes more.  The tables are the exclusive prefix sums over the groups, n + 1
 * entries each, as the plan holds them. */
static inline std::vector<CvfRange> cvf_group_ranges(const std::vector<int> &tile, const std::vector<int> &item,
                                                     const std::vector<int> &achunk, const std::vector<long long> &woff,
                                                     size_t w_limit)
{
    std::vector<CvfRange> out;
    const int n = (int)woff.size() - 1;
    for (int g0 = 0; g0 < n;) {
        int g1 = g0 + 1;
        while (g1 < n && (size_t)(woff[g1 + 1] - woff[g0]) <= w_limit)
            g1++;
        out.push_back({g0, g1, tile[g0], tile[g1], item[g0], item[g1], woff[g0], woff[g1], achunk[g0], achunk[g1]});
        g0 = g1;
    }
    return out;
}

/* host: the step masks of a slot_h table (length a multiple of 32): per 32 slots, bit 2 nt + c set
 * when one of the slots 8 nt + 2 q + c, q < 4, has a count */
static inline std::vector<int> cvf_step_masks(const std::vector<double> &slot_h)
{
    std::vector<int> out(slot_h.size() / 32, 0);
    for (size_t s = 0; s < slot_h.size(); s++)
        if (slot_h[s] != 0.0) {
            const int in32 = (int)(s & 31), nt = in32 >> 3, c = in32 & 1;
            out[s / 32] |= 1 << (2 * nt + c);
        }
    return out;
}

/* host: do all slots with counts lie in the first of the four slots a thread of the prefix kernel
 * owns per pass?  (slot -> half-line u = 2 * (slot / 64) + (slot % 64) / 32; a pass has 32
 * half-lines, a thread's slot i is half-line (u % 32) / 8.) */
static inline bool cvf_counts_first(const std::vector<double> &slot_h)
{
    for (size_t s = 0; s < slot_h.size(); s++)
        if (slot_h[s] != 0.0 && (((2 * (s / 64) + (s % 64) / 32) % 32) >> 3) != 0)
            return false;
    return true;
}

void cvf_release(CvFactorWork &wk);
