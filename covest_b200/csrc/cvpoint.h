/*
 * cvpoint.h -- the per-point evaluation of the CovEst mixture likelihood, written as a sequence
 * of warp-wide *phases*.  Inside the sm_100a kernel (kernels.cu) ONE WARP evaluates one parameter
 * point at a time: its 32 lanes call each phase with their own `lane`, the phases are separated by
 * __syncwarp(), and nothing is shared between the warps of a CTA except read-only group tables.
 * The test-only host emulation (tests/host_math/emulate.cpp) calls the same functions in a serial
 * loop over `lane`, phase by phase, which is the same computation.
 *
 *   header      clip the parameters (models.py:60-69), error-class rates l_s (models.py:71-79),
 *               the constants of the copy-number weights (models.py:193-208)
 *   per pass of 32 copy numbers o: the weights b(o), one per lane, and the cut-off O_thr
 *               (models.py:185-191) -- the weights stay in registers and reach the terms by shuffle
 *   per tile of up to 32 mixture terms (o, s), ONE TERM PER LANE:
 *     mass      n_os = comb[s] * (1.0 - exp(-o*l_s))                      (models.py:87, :221)
 *     prep      a_os = n_os / sum_s n_os, w = b(o) * a_os, the log-domain constants of the term;
 *               its powers PW[i] = lam^i, i < 16; its *anchors*: the scaled value of the term at the
 *               first bin of every group of NA rows (16 NA bins) of the current block -- one exp()
 *               per run of up to four groups, at the anchor next to the mode of the term, then the
 *               reference's own product recurrence (covest_poissonmodule.c:22-24) walked outwards
 *               one group at a time
 *     fused     lane (r, q) = (lane / 4, lane % 4) owns group r of the block: for each of the 4-term
 *               slices of the tile it extends the anchor of term q of the slice over the NA rows of
 *               its group with one multiplication per row -- which is exactly its A fragment of
 *               an m8n8k4 FP64 tensor-core MMA -- and issues
 *                   ACC[row][i] += A[row][t] * PW[i][t]      one FP64 FMA per (term, bin)
 *               for the 8 NA x 16 block (NA x 2 MMA tiles, 4 NA accumulators per lane)
 *   epilogue    p_j = ACC * slot_mult, mass += p_j, sum += h_j * log p_j  (models.py:100-107)
 *
 * Reference lines are relative to /root/reference.
 */
#pragma once
#include "cvmodel.h"

#define CV_W 16        /* bins per row */
#define CV_GB 8        /* groups per block (one per MMA row index) */
#define CV_NA_MAX 8    /* rows per group: 1, 2, 4 (histograms of up to 8, 16, 32 rows) or 8 */
#define CV_CT 32       /* mixture terms per tile: one per lane */
#define CV_RUNMAX 4    /* longest run of groups anchored from one exp() */
#define CV_MAX_PARAMS 5
#define CV_WARPS_MAX 12 /* warps (= points in flight) per CTA of the per-point kernel; one CTA per SM */
#define CV_COPY_PAD 40  /* copies past max(hist) that copy_log still covers */

/* record of a group in CvTables::grp */
#define CV_GD 16       /* doubles per record */
#define CV_G_J0 0      /* first bin of the group */
#define CV_G_HEAD 1    /* CV_SCALE_LOG - lgamma(j0 + 1), double-double (2) */
#define CV_G_EHEAD 3   /* the same at the bin after the group, j0 + 16 NA (2) */
#define CV_G_CINV 5    /* c^-16, c = geometric mean of the bins of the group: the chain normaliser */
#define CV_G_C16 6     /* its inverse */
#define CV_G_ENORM 7   /* takes the value at the bin after the group to the chain's scale */
#define CV_G_UP 8      /* (4) factorial ratios of the sub-steps of an anchor step, walking up */
#define CV_G_DN 12     /* (4) and walking down */

/* Histogram-side tables of a context.  Device memory in the product, host memory in the
 * emulation.  Built by cv_build_tables (cvtables.h).  slot = (group * NA + row) * 16 + column. */
struct CvTables {
    const double *grp;         /* CV_GD doubles per group */
    const double *slot_mult;   /* exp(-CV_SCALE_LOG) * (chain scale of the row) * j0! / (j0+i)!;
                                  0 marks a slot that is not in hist */
    const double *slot_mult_pair; /* slot_mult as the profile kernel stores it: per 64-slot line the
                                     32 pairs (slot 16 (L / 8) + L % 8, the same + 8), L = 0..31 */
    const double *slot_h;      /* count h_j */
    const int *slot_bin;       /* position of the bin in the caller's hist order, -1 = padding */
    const double *copy_log_h;  /* log(o), o = 0..max_bin, as a double-double (entry 0 unused) */
    const double *copy_log_l;
    const int *run_first;      /* runs: consecutive groups inside one block, at most CV_RUNMAX */
    const int *run_len;
    const int *blk_run_begin;  /* [n_blocks + 1] */
};

struct CvModelDesc {
    int model_kind; /* 0 basic (models.py:17), 1 repeats (models.py:173) */
    int k, r;
    int n_err;      /* max_error (models.py:28-31) */
    int n_param;
    int n_bins, n_groups, n_blocks;
    int na;         /* rows per group */
    int max_bin;    /* max(hist), models.py:186 */
    double tail;
    double threshold; /* NaN = None */
    double lo[CV_MAX_PARAMS], hi[CV_MAX_PARAMS]; /* NaN = open */
    double comb[CV_MAX_ERR];  /* models.py:25, as the host computed it */
    double pow3[CV_MAX_ERR];  /* 3 ** -s as the host computed it */
    CvTables tab;
};

/* Fixed-size part of the working set of one warp (= one point in flight); shared memory on the
 * device.  PW and ANC hold one 16-byte chunk per (term, group index / column pair); the chunk of
 * (t, g) sits at position (g + 2 t) & 7 of the 128 bytes of term t, so that the 8 lanes that read
 * together (2 groups x 4 terms) touch 8 different bank groups. */
struct CvWarpFixed {
    union {
        struct {
            double PW[CV_CT * 16];  /* chunk (t, i), i < 8: {lam^i, lam^(8+i)} */
            double ANC[CV_CT * 16]; /* chunk (t, g), g < 8: value of the term at the first bin of
                                       group g, and at the bin after the group */
        } t;
        double spill[CV_GB * CV_NA_MAX * CV_W]; /* the accumulators on their way to the epilogue */
    } u;
    double PWR[CV_CT * 2]; /* {lam^16, lam^-16} */
    double par[CV_MAX_PARAMS];
    double two, many, base; /* (1-q1)*q2, (1-q1)*(1-q2)*q, 1-q */
};

/* The working set of a warp: the fixed part, the arrays whose length depends on the number of
 * error classes, and the group tables every warp of the CTA reads. */
struct CvWarpMem {
    CvWarpFixed *fx;
    double *ls;            /* [S] l_s */
    double *lls_h, *lls_l; /* [S] log(l_s), double-double */
    double *nmass;         /* [group terms] n_os */
    double *glam;          /* [group terms] o * l_s */
    const double *grp;     /* CvTables::grp, staged in shared memory */
};

/* terms of the largest group: whole copies, at most 32 terms unless one copy alone has more */
CV_HD int cv_copies_per_group(int n_err) { return n_err >= CV_CT ? 1 : CV_CT / n_err; }
CV_HD int cv_group_terms_max(int n_err) { return n_err > CV_CT ? 2 * CV_CT : CV_CT; }
/* doubles of the variable part of a warp's working set */
CV_HD int cv_warp_var_doubles(int n_err) { return 3 * n_err + 2 * cv_group_terms_max(n_err); }

CV_HD void cv_warp_mem_carve(CvWarpMem &M, CvWarpFixed *fx, double *var, int n_err)
{
    int gm = cv_group_terms_max(n_err);
    M.fx = fx;
    M.ls = var;
    M.lls_h = var + n_err;
    M.lls_l = var + 2 * n_err;
    M.nmass = var + 3 * n_err;
    M.glam = M.nmass + gm;
}

struct CvPartial {
    double sum;            /* sum_j h_j log p_j */
    double mass_h, mass_l; /* sum_j p_j, compensated */
};

/* ---- header ------------------------------------------------------------------------------- */
/* `row` holds the raw parameters of the point (every lane has them). */
CV_HD void cv_w_header(int lane, const CvModelDesc &m, const double *row, int clip, CvWarpMem &M)
{
    CvWarpFixed &F = *M.fx;
    double c = row[0], e = row[1];
    if (clip) {
        c = cv_clip(c, m.lo[0], m.hi[0]);
        e = cv_clip(e, m.lo[1], m.hi[1]);
    }
    double ck = cv_kmer_coverage(c, m.k, m.r);
    for (int s = lane; s < m.n_err; s += 32) {
        double l = cv_error_class_rate(ck, m.pow3[s], e, m.k, s);
        M.ls[s] = l;
        cv_dd lg = {0.0, 0.0};
        if (l > 0.0 && l - l == 0.0) /* positive and finite */
            lg = cv_log_dd(l);
        M.lls_h[s] = lg.hi;
        M.lls_l[s] = lg.lo;
    }
    if (lane == 31) {
        double par[CV_MAX_PARAMS];
#pragma unroll
        for (int i = 0; i < CV_MAX_PARAMS; i++) {
            par[i] = 0.0;
            if (i < m.n_param)
                par[i] = clip ? cv_clip(row[i], m.lo[i], m.hi[i]) : row[i];
            F.par[i] = par[i];
        }
        if (m.model_kind) {
            double q1 = par[2], q2 = par[3], q = par[4];
            F.two = cv_mul(cv_sub(1.0, q1), q2);                          /* models.py:195 */
            F.many = cv_mul(cv_mul(cv_sub(1.0, q1), cv_sub(1.0, q2)), q); /* models.py:196 */
            F.base = cv_sub(1.0, q);
        } else {
            F.two = F.many = F.base = 0.0;
        }
    }
}

/* One lane's share of a pass of the cut-off search models.py:187-190 over copies
 * first_o .. first_o + 31: lane i looks at o = first_o + i.  Returns true when the evaluated
 * copies end BEFORE o (the caller takes the lowest such lane); *b is b(o), models.py:198-206.
 * The basic model is the single copy o = 1 with weight 1. */
CV_HD bool cv_w_copy_pass(int lane, const CvModelDesc &m, const CvWarpMem &M, int first_o, double *b)
{
    int o = first_o + lane;
    if (!m.model_kind) {
        *b = 1.0;
        return o >= 2;
    }
    if (o >= m.max_bin) { /* models.py:191: no cut found, O_thr = max(hist) */
        *b = 0.0;
        return true;
    }
    const CvWarpFixed &F = *M.fx;
    double w = cv_copy_weight(o, F.par[2], F.two, F.many, F.base);
    *b = w;
    return w <= m.threshold;
}

/* ---- per group of copies ------------------------------------------------------------------ */
/* models.py:87 / :221.  Slot t of the group is copy o = group_o + t / sp, error class s = t % sp;
 * sp >= S is the number of slots a copy takes (S in the per-point kernel, S rounded up to a
 * multiple of 4 in the profile kernel, whose MMA slices must not mix copies); slots with s >= S
 * are dead. */
CV_HD void cv_w_mass(int lane, const CvModelDesc &m, int group_o, int nslots, int sp, CvWarpMem &M)
{
    int S = m.n_err;
    for (int t = lane; t < nslots; t += 32) {
        int g = t / sp, s = t - g * sp;
        if (s >= S)
            continue;
        double lam = cv_mul((double)(group_o + g), M.ls[s]); /* o * l_s, models.py:238 */
        M.glam[t] = lam;
        M.nmass[t] = cv_class_mass(m.comb[s], lam);
    }
}

/* Constants of the term in slot t = sub + lane of the group (a dead term when the slot is past
 * the group or past the error classes of its copy); `b` is the weight b(o) of the copy this lane's
 * term belongs to. */
CV_HD CvTerm cv_w_term(int lane, const CvModelDesc &m, int group_o, int nslots, int sp, int sub,
                       double b, const CvWarpMem &M)
{
    const CvTerm dead = {1.0, 0.0, 0.0, 0.0, 0.0}; /* contributes exactly 0 */
    int t = sub + lane;
    if (t >= nslots)
        return dead;
    int S = m.n_err;
    int g = t / sp, s = t - g * sp;
    if (s >= S)
        return dead;
    int o = group_o + g;
    /* models.py:88 / :224: Python sum(), left to right starting from int 0 */
    double total = 0.0;
    for (int i = 0; i < S; i++)
        total = cv_add(total, M.nmass[g * sp + i]);
    if (total == 0.0)
        total = 1.0; /* utils.py:25-29 fix_zero */
    double lam = M.glam[t];
    /* log(lam) = log(o) + log(l_s) + log(lam / (o*l_s)); the last part undoes the rounding of the
     * product lam = RN(o*l_s) and is -(o*l_s - lam)/lam to first order (|.| <= 2^-53) */
    double ls = M.ls[s];
    double resid = cv_fma((double)o, ls, -lam);
    cv_dd lo_ = {m.tab.copy_log_h[o], m.tab.copy_log_l[o]};
    cv_dd ll_ = {M.lls_h[s], M.lls_l[s]};
    cv_dd lg = cv_dd_add(lo_, ll_);
    if (resid != 0.0)
        lg = cv_dd_add_d(lg, -cv_div(resid, lam));
    return cv_term_make(lam, cv_mul(b, M.nmass[t]), total, lg.hi, lg.lo);
}

/* two adjacent doubles, one 16-byte access on the device */
struct cv_pair {
    double x, y;
};
CV_HD cv_pair cv_ld2(const double *p)
{
#if defined(__CUDA_ARCH__)
    double2 v = *reinterpret_cast<const double2 *>(p);
    cv_pair r = {v.x, v.y};
    return r;
#else
    cv_pair r = {p[0], p[1]};
    return r;
#endif
}
CV_HD void cv_st2(double *p, double x, double y)
{
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<double2 *>(p) = make_double2(x, y);
#else
    p[0] = x;
    p[1] = y;
#endif
}

/* position (in doubles) of chunk (t, g) inside PW / ANC */
CV_HD int cv_chunk(int t, int g) { return (t * 8 + ((g + 2 * t) & 7)) * 2; }

/* ---- prep: powers and anchors of the lane's term ------------------------------------------- */
/* An anchor step (16 NA bins) is taken as NSUB sub-steps of 32 bins (16 when NA = 1), each the
 * product lam^32 * (factorial ratio): every factor stays far inside the double range for any rate
 * the model can produce.
 *
 * Where the walk over the n + 1 anchors of a run starts:
 *   - mode of the term (j ~ lam) at or above the last anchor: there, walking down;
 *   - otherwise at the first anchor, walking up through the mode, when the value there is well
 *     inside the double range (it always is unless the weight of the term is minute);
 *   - otherwise at the anchor below the mode, walking up and then down, so that a value that
 *     underflowed never has to grow back.
 * The first two cases share one loop with a per-lane direction, so lanes do not diverge. */
template <int NA>
CV_HD void cv_w_prep(int lane, const CvModelDesc &m, int blk, const CvTerm &tm, CvWarpMem &M)
{
    constexpr int NSUB = NA >= 2 ? NA / 2 : 1;
    constexpr double INV_SPAN = 1.0 / (CV_W * NA);
    CvWarpFixed &F = *M.fx;
    const CvTables &T = m.tab;
    const double lam = tm.lam, lh = tm.lh, lin = tm.lin, f = tm.f;
    const double l2 = cv_mul(lam, lam);
    const double l3 = cv_mul(l2, lam);
    const double l4 = cv_mul(l2, l2);
    const double l5 = cv_mul(l4, lam);
    const double l6 = cv_mul(l4, l2);
    const double l7 = cv_mul(l4, l3);
    const double l8 = cv_mul(l4, l4);
    const double l16 = cv_mul(l8, l8);
    const double inv16 = cv_div(1.0, l16);
    {
        double *pw = F.u.t.PW;
        cv_st2(pw + cv_chunk(lane, 0), 1.0, l8);
        cv_st2(pw + cv_chunk(lane, 1), lam, cv_mul(l8, lam));
        cv_st2(pw + cv_chunk(lane, 2), l2, cv_mul(l8, l2));
        cv_st2(pw + cv_chunk(lane, 3), l3, cv_mul(l8, l3));
        cv_st2(pw + cv_chunk(lane, 4), l4, cv_mul(l8, l4));
        cv_st2(pw + cv_chunk(lane, 5), l5, cv_mul(l8, l5));
        cv_st2(pw + cv_chunk(lane, 6), l6, cv_mul(l8, l6));
        cv_st2(pw + cv_chunk(lane, 7), l7, cv_mul(l8, l7));
        cv_st2(F.PWR + 2 * lane, l16, inv16);
    }
    const double step_up = NA >= 2 ? cv_mul(l16, l16) : l16;
    const double step_dn = NA >= 2 ? cv_mul(inv16, inv16) : inv16;
    double *anc = F.u.t.ANC;
    const int rb = T.blk_run_begin[blk], re = T.blk_run_begin[blk + 1];
    for (int run = rb; run < re; run++) {
        const int first = T.run_first[run], n = T.run_len[run];
        const double *g0 = M.grp + (size_t)(blk * CV_GB + first) * CV_GD;
        const double j0 = g0[CV_G_J0];
        const double off = cv_mul(cv_sub(lam, j0), INV_SPAN);
        /* exponent of the scaled term at the first anchor, to a few ulps */
        const double e0 = cv_sub(cv_fma(j0, lh, g0[CV_G_HEAD]), lin);
        int rs;
        if (off >= (double)n)
            rs = n;
        else if (e0 > -460.0 && !(f < 0x1p-200))
            rs = 0;
        else
            rs = off > 0.0 ? (int)off : 0;
        const bool down = rs == n;
        {
            const double *ga = g0 + (down ? n - 1 : rs) * CV_GD;
            const double ja = down ? cv_add(ga[CV_G_J0], (double)(CV_W * NA)) : ga[CV_G_J0];
            const double hh = ga[down ? CV_G_EHEAD : CV_G_HEAD];
            const double hl = ga[down ? CV_G_EHEAD + 1 : CV_G_HEAD + 1];
            const double seed = cv_seed(ja, hh, hl, lh, tm.ll, lin, f);
            if (rs < n)
                anc[cv_chunk(lane, first + rs)] = seed;
            if (rs > 0)
                anc[cv_chunk(lane, first + rs - 1) + 1] = seed;
            double v = seed;
            const int n1 = down ? n : n - rs;
            const double step = down ? step_dn : step_up;
            for (int k = 0; k < n1; k++) {
                const int gi = down ? n - 1 - k : rs + k; /* the group the step crosses */
                const double *fp = g0 + gi * CV_GD + (down ? CV_G_DN : CV_G_UP);
                double c[NSUB];
#pragma unroll
                for (int u = 0; u < NSUB; u++)
                    c[u] = cv_mul(step, fp[u]);
#pragma unroll
                for (int u = 0; u < NSUB; u++)
                    v = cv_mul(v, c[u]);
                const int a = down ? gi : gi + 1; /* the anchor reached */
                if (a < n)
                    anc[cv_chunk(lane, first + a)] = v;
                if (a > 0)
                    anc[cv_chunk(lane, first + a - 1) + 1] = v;
            }
            if (!down) { /* the anchors below an interior starting anchor */
                v = seed;
                for (int a = rs - 1; a >= 0; a--) {
                    const double *fp = g0 + a * CV_GD + CV_G_DN;
#pragma unroll
                    for (int u = 0; u < NSUB; u++)
                        v = cv_mul(v, cv_mul(step_dn, fp[u]));
                    anc[cv_chunk(lane, first + a)] = v;
                    if (a > 0)
                        anc[cv_chunk(lane, first + a - 1) + 1] = v;
                }
            }
        }
    }
}

/* One m8n8k4 FP64 MMA: D = A (8 x 4, row) * B (4 x 8, col) + D.  Lane l holds A[l >> 2][l & 3],
 * B[l & 3][l >> 2] and D[l >> 2][2 (l & 3) + {0, 1}]. */
#if defined(__CUDACC__)
__device__ __forceinline__ void cv_dmma(double &d0, double &d1, double a, double b)
{
#if defined(__CUDA_ARCH__)
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
#endif
}
#endif
#if defined(__CUDA_ARCH__)
#define CV_WARP_ANY(x) __any_sync(0xffffffffu, (x))
#else
#define CV_WARP_ANY(x) (x)
#endif

/* The constants of the lane's group (r = lane >> 2) for the fused phase; zeros past the last
 * group of the block, which turns the lane's rows into exact zeros. */
struct CvLaneGroup {
    double cinv, c16, enorm;
    int live;
};
CV_HD CvLaneGroup cv_lane_group(int lane, const CvModelDesc &m, int blk, const CvWarpMem &M)
{
    CvLaneGroup G = {0.0, 0.0, 0.0, 0};
    int g = blk * CV_GB + (lane >> 2);
    if (g < m.n_groups) {
        const double *rec = M.grp + (size_t)g * CV_GD;
        G.cinv = rec[CV_G_CINV];
        G.c16 = rec[CV_G_C16];
        G.enorm = rec[CV_G_ENORM];
        G.live = 1;
    }
    return G;
}

/* The values of term t over the NA rows of the lane's group, on the chain's scale (row m is the
 * true scaled value divided by a row constant that slot_mult carries): a[0] is the anchor, every
 * further row one multiplication by E = (lam / c)^16.  A chain whose anchor underflowed although
 * the values grow along the group is walked down from the far anchor instead. */
template <int NA>
CV_HD void cv_row_chain(const CvWarpFixed &F, const CvLaneGroup &G, int r, int t, double *a)
{
    cv_pair av = cv_ld2(F.u.t.ANC + cv_chunk(t, r));
    cv_pair pr = cv_ld2(F.PWR + 2 * t);
    const double start = G.live ? av.x : 0.0;
    const double end = G.live ? av.y : 0.0;
    a[0] = start;
    if (NA == 1)
        return;
    const double E = cv_mul(pr.x, G.cinv);
#pragma unroll
    for (int i = 1; i < NA; i++)
        a[i] = cv_mul(a[i - 1], E);
    const bool need_down = start < 0x1p-1000 && end > start;
    if (CV_WARP_ANY(need_down)) {
        const double Einv = cv_mul(pr.y, G.c16);
        double d = cv_mul(end, G.enorm);
#pragma unroll
        for (int i = NA - 1; i >= 1; i--) {
            d = cv_mul(d, Einv);
            if (need_down)
                a[i] = d;
        }
    }
}

/* The accumulators of a lane: MMA tile (mt, nt), mt < NA row tiles, nt < 2 column tiles, holds row
 * mt of group r and columns 8 nt + 2 q + {0, 1} with r = lane >> 2, q = lane & 3;
 * acc[4 mt + 2 nt + {0, 1}].  The terms of the tile are contracted 4 at a time (nkg slices); lane q
 * supplies term q of each slice; slices kg0 .. nkg - 1 are contracted.  On the host (test emulation) the same sums are formed with scalar
 * FMAs in the same term order. */
template <int NA>
CV_HD void cv_w_fused(int lane, const CvLaneGroup &G, int kg0, int nkg, const CvWarpFixed &F, double *acc)
{
    const int r = lane >> 2, q = lane & 3;
#if defined(__CUDA_ARCH__)
#pragma unroll 2
    for (int kg = kg0; kg < nkg; kg++) {
        const int t = 4 * kg + q;
        double a[NA];
        cv_row_chain<NA>(F, G, r, t, a);
        cv_pair b = cv_ld2(F.u.t.PW + cv_chunk(t, r));
#pragma unroll
        for (int mt = 0; mt < NA; mt++) {
            cv_dmma(acc[4 * mt + 0], acc[4 * mt + 1], a[mt], b.x);
            cv_dmma(acc[4 * mt + 2], acc[4 * mt + 3], a[mt], b.y);
        }
    }
#else
    for (int kg = kg0; kg < nkg; kg++) {
        double a[4][NA];
        for (int k = 0; k < 4; k++)
            cv_row_chain<NA>(F, G, r, 4 * kg + k, a[k]);
        for (int mt = 0; mt < NA; mt++)
            for (int nt = 0; nt < 2; nt++)
                for (int c = 0; c < 2; c++) {
                    double v = acc[4 * mt + 2 * nt + c];
                    for (int k = 0; k < 4; k++) {
                        const double *ch = F.u.t.PW + cv_chunk(4 * kg + k, 2 * q + c);
                        v = cv_fma(a[k][mt], ch[nt], v);
                    }
                    acc[4 * mt + 2 * nt + c] = v;
                }
    }
#endif
}

/* The accumulators of a lane go to the spill area in slot order, slot = row * 16 + column (row
 * counted inside the block); the 16-byte chunks of odd groups are swapped between the halves of
 * the row so that a quarter warp (2 groups x 4 chunks) does not collide. */
template <int NA>
CV_HD int cv_spill_index(int slot)
{
    return slot ^ ((((slot >> 4) / NA) & 1) << 3); /* column ^= 8 in odd groups */
}
template <int NA>
CV_HD void cv_w_spill(int lane, CvWarpFixed &F, const double *acc)
{
    const int r = lane >> 2, q = lane & 3;
#pragma unroll
    for (int mt = 0; mt < NA; mt++)
#pragma unroll
        for (int nt = 0; nt < 2; nt++) {
            int slot = (NA * r + mt) * CV_W + 8 * nt + 2 * q;
            cv_st2(F.u.spill + cv_spill_index<NA>(slot), acc[4 * mt + 2 * nt], acc[4 * mt + 2 * nt + 1]);
        }
}

CV_HD void cv_partial_add_mass(CvPartial &p, double x)
{
    cv_dd s = cv_two_sum(p.mass_h, x);
    p.mass_h = s.hi;
    p.mass_l = cv_add(p.mass_l, s.lo);
}

CV_HD void cv_partial_merge(CvPartial &p, const CvPartial &q)
{
    cv_partial_add_mass(p, q.mass_h);
    p.mass_l = cv_add(p.mass_l, q.mass_l);
    p.sum = cv_add(p.sum, q.sum);
}

/* models.py:100-107 per bin: lane l finishes the slots l, l + 32, ... of the block, four at a time
 * so that the logarithms overlap.  The weighted logarithms all have one sign (p_j <= 1 outside the
 * reference's lam > 200 sawtooth), so their plain sum is good to ~1e-13; the mass needs the
 * compensated sum only for the tail term and is skipped when there is no tail. */
template <int NA>
CV_HD void cv_w_epilogue(int lane, const CvModelDesc &m, int blk, int ngroups_blk, const CvWarpFixed &F,
                         CvPartial &part, double *out_probs)
{
    constexpr int U = 4;
    const CvTables &T = m.tab;
    const size_t base = (size_t)blk * (CV_GB * NA * CV_W);
    const double *mult = T.slot_mult + base;
    const double *cnt = T.slot_h + base;
    const int *bin = T.slot_bin + base;
    const int nslots = ngroups_blk * NA * CV_W;
    const bool want_mass = m.tail != 0.0;
    double sum[U];
#pragma unroll
    for (int u = 0; u < U; u++)
        sum[u] = 0.0;
    for (int base = 0; base < nslots; base += 32 * U) { /* warp-uniform trip count */
        double p[U], h[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int e = base + lane + 32 * u;
            double mu = 0.0;
            h[u] = 0.0;
            p[u] = 0.0;
            if (e < nslots) {
                mu = mult[e];
                h[u] = cnt[e];
                p[u] = cv_mul(F.u.spill[cv_spill_index<NA>(e)], mu);
                if (out_probs && mu != 0.0)
                    out_probs[bin[e]] = cv_mul(p[u], CV_PUNSCALE); /* p[] stays scaled by 2^128 */
            }
            if (mu == 0.0) { /* a bin that is not in hist (p may be NaN * 0) */
                p[u] = 0.0;
                h[u] = 0.0;
            }
        }
        if (want_mass) {
#pragma unroll
            for (int u = 0; u < U; u++)
                cv_partial_add_mass(part, p[u]);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const bool counted = h[u] != 0.0; /* models.py:106 `if h` */
            if (CV_WARP_ANY(counted)) {
                double lg = cv_log_scaled(p[u]); /* utils.py:32-35 safe_log */
                if (counted)
                    sum[u] = cv_add(sum[u], cv_mul(h[u], lg));
            }
        }
    }
    part.sum = cv_add(part.sum, cv_add(cv_add(sum[0], sum[1]), cv_add(sum[2], sum[3])));
}

/* models.py:103-107 */
CV_HD double cv_point_finish(const CvModelDesc &m, const CvPartial &part)
{
    /* the partial sums are sums of probabilities scaled by 2^128 */
    double mass = cv_add(cv_mul(part.mass_h, CV_PUNSCALE), cv_mul(part.mass_l, CV_PUNSCALE));
    if (!(mass < 1.0))
        mass = 1.0; /* min(1, fsum(...)): keeps the 1 unless the sum is smaller (also for NaN) */
    return cv_finish_loglik(part.sum, mass, m.tail);
}
