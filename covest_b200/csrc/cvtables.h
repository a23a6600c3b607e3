/*
 * cvtables.h -- host-side construction of the histogram tables a context keeps in HBM
 * (CvTables, cvpoint.h).  Host only; used by the C-ABI library at ctx_create and by the
 * test-only emulation.
 *
 * The bins of `hist` (models.py:27; any set of non-negative keys, in the caller's dict order) are
 * covered by *groups* of NA rows of 16 consecutive bins each: the smallest uncovered key opens a
 * group.  NA is the smallest of 1, 2, 4 that covers the histogram with at most 8 groups, else 8
 * (any number of groups, in blocks of 8).  Slots of a group whose bin is not a key of hist are
 * padding (slot_mult = 0).  Inside a block, groups that follow each other without a gap form runs
 * of at most CV_RUNMAX groups -- the unit that is anchored by one exp() per mixture term.
 */
#pragma once
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "cvpoint.h"

struct CvHostTables {
    std::vector<double> grp, slot_mult, slot_h;
    std::vector<double> copy_log_h, copy_log_l;
    std::vector<int> slot_bin, run_first, run_len, blk_run_begin;
    int n_groups = 0, n_blocks = 0, na = 0, max_bin = 0;
};

/* log(j!) as a double-double for every j of the ascending list `at` */
static inline void cv_log_factorials(const std::vector<long> &at, std::vector<cv_dd> &out)
{
    out.resize(at.size());
    cv_dd acc = {0.0, 0.0};
    long j = 1; /* acc = log(j!) */
    for (size_t i = 0; i < at.size(); i++) {
        long want = at[i] < 1 ? 1 : at[i];
        while (j < want) {
            j++;
            acc = cv_dd_add(acc, cv_log_dd((double)j));
        }
        out[i] = acc;
    }
}

/* prod_{i=1..n} (j + i) */
static inline long double cv_rising(long j, int n)
{
    long double run = 1.0L;
    for (int i = 1; i <= n; i++)
        run *= (long double)(j + i);
    return run;
}

/* returns "" or an error message */
static inline std::string cv_build_tables(int n_bins, const int *bin_j, const double *bin_h,
                                          CvHostTables &T)
{
    if (n_bins <= 0)
        return "empty histogram";
    std::vector<std::pair<long, int>> keys(n_bins);
    for (int b = 0; b < n_bins; b++) {
        if (bin_j[b] < 0)
            return "negative histogram key";
        if (bin_j[b] > (1 << 24))
            return "histogram key above 2^24";
        keys[b] = std::make_pair((long)bin_j[b], b);
    }
    std::sort(keys.begin(), keys.end());
    for (int b = 1; b < n_bins; b++)
        if (keys[b].first == keys[b - 1].first)
            return "duplicate histogram key";
    T.max_bin = (int)keys.back().first;

    std::vector<long> heads;
    int na = 1;
    for (;; na *= 2) {
        heads.clear();
        const long span = (long)CV_W * na;
        for (int b = 0; b < n_bins;) {
            long j0 = keys[b].first;
            heads.push_back(j0);
            while (b < n_bins && keys[b].first < j0 + span)
                b++;
        }
        if (na == CV_NA_MAX || (int)heads.size() <= CV_GB)
            break;
    }
    const long span = (long)CV_W * na;
    const int sub_bins = na == 1 ? CV_W : 2 * CV_W;
    const int nsub = (int)(span / sub_bins);
    T.na = na;
    T.n_groups = (int)heads.size();
    T.n_blocks = (T.n_groups + CV_GB - 1) / CV_GB;
    const int padded = T.n_blocks * CV_GB;
    const size_t nslots = (size_t)padded * na * CV_W;
    T.grp.assign((size_t)padded * CV_GD, 0.0);
    T.slot_mult.assign(nslots, 0.0);
    T.slot_h.assign(nslots, 0.0);
    T.slot_bin.assign(nslots, -1);

    /* log-factorials at the first bin of every group and at the bin after it */
    std::vector<long> at;
    for (long j0 : heads) {
        at.push_back(j0);
        at.push_back(j0 + span);
    }
    std::sort(at.begin(), at.end());
    at.erase(std::unique(at.begin(), at.end()), at.end());
    std::vector<cv_dd> logfact;
    cv_log_factorials(at, logfact);
    auto head_at = [&](long j) {
        size_t i = std::lower_bound(at.begin(), at.end(), j) - at.begin();
        cv_dd neg = {-logfact[i].hi, -logfact[i].lo};
        return cv_dd_add_d(neg, CV_SCALE_LOG);
    };

    const long double unscale = expl(-(long double)CV_SCALE_LOG);
    std::vector<long double> row_scale((size_t)T.n_groups * na, 1.0L); /* R'_m of DESIGN.md */
    for (int g = 0; g < T.n_groups; g++) {
        const long j0 = heads[g];
        double *rec = T.grp.data() + (size_t)g * CV_GD;
        rec[CV_G_J0] = (double)j0;
        cv_dd h0 = head_at(j0), h1 = head_at(j0 + span);
        rec[CV_G_HEAD] = h0.hi;
        rec[CV_G_HEAD + 1] = h0.lo;
        rec[CV_G_EHEAD] = h1.hi;
        rec[CV_G_EHEAD + 1] = h1.lo;
        /* c^16 with c the geometric mean of the bins j0+1 .. j0+span; the chain multiplies by the
         * DOUBLE c^-16, so the row scales below are built from that double */
        long double c16 = powl(cv_rising(j0, (int)span), 1.0L / (long double)na);
        const double cinv = (double)(1.0L / c16);
        rec[CV_G_CINV] = cinv;
        rec[CV_G_C16] = (double)(1.0L / (long double)cinv);
        long double scale = 1.0L;
        for (int mrow = 1; mrow <= na; mrow++) {
            scale = scale / (long double)cinv / cv_rising(j0 + (long)CV_W * (mrow - 1), CV_W);
            if (mrow < na)
                row_scale[(size_t)g * na + mrow] = scale;
        }
        rec[CV_G_ENORM] = (double)(1.0L / scale);
        for (int u = 0; u < 4; u++) {
            rec[CV_G_UP + u] = 1.0;
            rec[CV_G_DN + u] = 1.0;
            if (u < nsub) {
                long double run = cv_rising(j0 + (long)sub_bins * u, sub_bins);
                rec[CV_G_UP + u] = (double)(1.0L / run);
                rec[CV_G_DN + u] = (double)run;
            }
        }
    }
    /* slots */
    {
        int g = 0;
        for (int b = 0; b < n_bins; b++) {
            long j = keys[b].first;
            while (j >= heads[g] + span)
                g++;
            int d = (int)(j - heads[g]);
            int mrow = d / CV_W, i = d % CV_W;
            long double run = cv_rising(heads[g] + (long)CV_W * mrow, i);
            size_t slot = ((size_t)g * na + mrow) * CV_W + i;
            /* times 2^128: see CV_PSCALE (cvmodel.h) */
            T.slot_mult[slot] = (double)(unscale * row_scale[(size_t)g * na + mrow] / run * (long double)CV_PSCALE);
            T.slot_h[slot] = bin_h ? bin_h[keys[b].second] : 0.0;
            T.slot_bin[slot] = keys[b].second;
        }
    }
    /* log(o) for every copy number the cut-off can reach (models.py:186: o < max(hist)), plus the
     * few the profile kernel evaluates to fill its last slice of copies */
    T.copy_log_h.assign((size_t)T.max_bin + 2 + CV_COPY_PAD, 0.0);
    T.copy_log_l.assign((size_t)T.max_bin + 2 + CV_COPY_PAD, 0.0);
    for (int o = 2; o <= T.max_bin + 1 + CV_COPY_PAD; o++) {
        cv_dd lg = cv_log_dd((double)o);
        T.copy_log_h[o] = lg.hi;
        T.copy_log_l[o] = lg.lo;
    }
    /* runs */
    T.blk_run_begin.assign(T.n_blocks + 1, 0);
    T.run_first.clear();
    T.run_len.clear();
    for (int blk = 0; blk < T.n_blocks; blk++) {
        T.blk_run_begin[blk] = (int)T.run_first.size();
        int lo = blk * CV_GB, hi = std::min(T.n_groups, lo + CV_GB);
        int g = lo;
        while (g < hi) {
            int start = g;
            g++;
            while (g < hi && g - start < CV_RUNMAX && heads[g] == heads[g - 1] + span)
                g++;
            T.run_first.push_back(start - lo);
            T.run_len.push_back(g - start);
        }
    }
    T.blk_run_begin[T.n_blocks] = (int)T.run_first.size();
    return "";
}

/* The row tables of T: the tables of the keys of T's 64-slot lines that hold a count.  Keys without
 * a count inside those lines stay, so that the groups start where they did.  Without a tail only
 * these bins enter the log-likelihood (models.py:103-107), and the batched path evaluates them alone.
 * Returns false when they would not leave out a line of T or need more than one block of groups.
 * R's max_bin and copy_log are those of the subset: O_thr and the copy logarithms must come from T. */
static inline bool cv_build_row_tables(const CvHostTables &T, const int *bin_j, const double *bin_h,
                                       CvHostTables &R)
{
    const size_t lines = T.slot_h.size() / 64;
    std::vector<int> sub_j;
    std::vector<double> sub_h;
    for (size_t l = 0; l < lines; l++) {
        bool counts = false;
        for (int i = 0; i < 64; i++)
            counts = counts || T.slot_h[l * 64 + i] != 0.0;
        for (int i = 0; i < 64 && counts; i++) {
            const int b = T.slot_bin[l * 64 + i];
            if (b >= 0) {
                sub_j.push_back(bin_j[b]);
                sub_h.push_back(bin_h[b]);
            }
        }
    }
    if (!cv_build_tables((int)sub_j.size(), sub_j.data(), sub_h.data(), R).empty())
        return false; /* no count at all */
    /* A subset of the keys never needs more lines (greedy groups cover a subset with no more groups).
     * Row tables of one block only, a measured rule whose cause is not known: on one B200, cfg3
     * (16 lines -> 4, one block) and cfg5 (32 -> 4, two blocks -> one) gain, while cfg4's row tables
     * (80 lines -> 48, five blocks -> three, 7 runs of groups instead of 10) made the profile kernel
     * slower, 0.54 ms instead of 0.40.  Multi-block row tables are left to a measurement that
     * explains that. */
    return R.n_blocks == 1 && R.slot_h.size() < T.slot_h.size();
}

static inline CvTables cv_tables_view(const CvHostTables &T)
{
    CvTables v;
    v.grp = T.grp.data();
    v.slot_mult = T.slot_mult.data();
    v.slot_mult_pair = nullptr; /* device only (capi.cu) */
    v.slot_h = T.slot_h.data();
    v.slot_bin = T.slot_bin.data();
    v.copy_log_h = T.copy_log_h.data();
    v.copy_log_l = T.copy_log_l.data();
    v.run_first = T.run_first.data();
    v.run_len = T.run_len.data();
    v.blk_run_begin = T.blk_run_begin.data();
    return v;
}
