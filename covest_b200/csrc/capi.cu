/*
 * capi.cu -- the C ABI of libcovest_b200.so (include/covest_b200.h): contexts, staging of host
 * buffers, kernel launches.  No arithmetic of the likelihood lives here -- and no CPU fallback:
 * every entry point needs a CUDA device.
 */
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/covest_b200.h"
#include "cvtables.h"
#include "factored.h"
#include "faithful.h"
#include "kernels.h"
#include "kmers.h"

#define CVB_CHUNK_POINTS (1LL << 22) /* staging granularity for host-resident batches */
#define CVB_MAX_TIMED_CHUNKS 64
#define CVB_TOPK_RADIX_MIN 32768 /* batches from this size on select their top-K by a radix selection or sort */

struct cvb_ctx {
    int device = 0;
    int n_sm = 0;
    int smem_max = 0; /* opt-in dynamic shared memory per CTA */
    CvModelDesc desc;
    std::vector<void *> owned; /* device allocations that live as long as the context */
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr; /* device -> host copy of the values while the top-K runs */
    cudaEvent_t copy_ev = nullptr;
    cudaEvent_t copy_done = nullptr; /* the side copy has finished: the main stream waits for it */
    /* calls of one context share its scratch (work counters, plan, profiles, staging): a call on a
     * different stream than the previous one first waits for the previous call's work */
    cudaEvent_t order_ev = nullptr;
    cudaStream_t last_stream = nullptr;
    bool order_valid = false;
    /* growable staging */
    double *d_params = nullptr;
    size_t cap_params = 0; /* doubles */
    double *d_ll = nullptr;
    size_t cap_ll = 0;
    double *d_probs = nullptr;
    size_t cap_probs = 0;
    double *d_cand_ll = nullptr, *d_sel_ll = nullptr, *d_rows = nullptr;
    long long *d_cand_idx = nullptr, *d_sel_idx = nullptr;
    int cap_k = 0;
    int topk_ctas = 0;
    unsigned char *d_topk_scratch = nullptr;
    size_t cap_topk_scratch = 0;
    double *d_axes = nullptr;
    size_t cap_axes = 0;
    unsigned long long *d_counter = nullptr;
    double *d_sink = nullptr;
    /* per-segment keys and lattice indices of cvb_lattice_profile, its rows when they go to host memory */
    unsigned long long *d_seg_key = nullptr, *d_seg_best = nullptr;
    size_t cap_seg_key = 0, cap_seg_best = 0;
    double *d_seg_rows = nullptr;
    size_t cap_seg_rows = 0;
    /* timing */
    bool timing = false;
    std::vector<cudaEvent_t> ev;
    int timed_chunks = 0;
    int last_launches = 0;
    cudaStream_t timed_stream = nullptr;
    /* the factored path of the repeats model (factored.h) */
    CvFactorWork fw;
    CvModelDesc fdesc;         /* desc with the row tables of the batched path (cv_build_row_tables), or desc itself */
    CvfSlots slots;            /* the row layout of the profiles (factored.h) */
    const double *d_log_tab = nullptr;
    int path_mode = 0;         /* 0 auto, 1 per-point kernel only, 2 factored whenever supported */
    size_t w_limit = (size_t)2 << 30; /* doubles: 16 GiB of profiles per group range */
    double min_group = 12.0;   /* auto: points per (c, e) group below which the per-point kernel runs */
    long long min_points = 2048; /* auto: batches below this go straight to the per-point kernel */
    int last_path = 0;         /* 1 per-point, 2 factored (GEMM), 3 factored (prefix kernel) */
    double min_run = 4.0;      /* auto: points per q-run below which the GEMM runs instead of the prefix kernel */
    /* re-evaluation of marked points (faithful.h) */
    CvFaithTables faith = {nullptr, nullptr, 0, 0, nullptr, 0};
    unsigned long long *d_fixed = nullptr; /* two words: marked points of the most recent evaluation, work cursor */
    unsigned int *d_marked = nullptr;      /* their indices */
    size_t cap_marked = 0;
    /* tests (COVEST_B200_POISON): byte every call first fills the double scratch it uses with, 0 = off */
    int poison = 0;
    std::string err;
};

static thread_local std::string g_create_error;

static int fail(cvb_ctx *ctx, int code, const std::string &msg)
{
    if (ctx)
        ctx->err = msg;
    else
        g_create_error = msg;
    return code;
}

static int fail_cuda(cvb_ctx *ctx, cudaError_t e, const char *what)
{
    return fail(ctx, CVB_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CU(call, what)                        \
    do {                                      \
        cudaError_t e_ = (call);              \
        if (e_ != cudaSuccess)                \
            return fail_cuda(ctx, e_, what);  \
    } while (0)

static bool is_device_ptr(const void *p)
{
    if (!p)
        return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

template <typename T>
static cudaError_t grow(T **buf, size_t *cap, size_t want)
{
    if (want <= *cap)
        return cudaSuccess;
    if (*buf)
        cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    cudaError_t e = cudaMalloc((void **)buf, want * sizeof(T));
    if (e == cudaSuccess)
        *cap = want;
    return e;
}

template <typename T>
static cudaError_t upload(cvb_ctx *ctx, const std::vector<T> &v, const T **out)
{
    void *d = nullptr;
    size_t bytes = (v.empty() ? 1 : v.size()) * sizeof(T);
    cudaError_t e = cudaMalloc(&d, bytes);
    if (e != cudaSuccess)
        return e;
    ctx->owned.push_back(d);
    if (!v.empty())
        e = cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    *out = (const T *)d;
    return e;
}

/* the tables the profile kernel reads: group records, runs, slot_mult in the order of its stores */
static cudaError_t upload_profile_tables(cvb_ctx *ctx, const CvHostTables &T, CvTables &t)
{
    cudaError_t e;
    if ((e = upload(ctx, T.grp, &t.grp)) != cudaSuccess)
        return e;
    std::vector<double> pr(T.slot_mult.size(), 0.0); /* per 64-slot line: pair L = slots 16 (L / 8) + L % 8 and + 8 */
    for (size_t line = 0; line + 64 <= T.slot_mult.size(); line += 64)
        for (int L = 0; L < 32; L++) {
            const size_t s0 = line + 16 * (L >> 3) + (L & 7);
            pr[line + 2 * L] = T.slot_mult[s0];
            pr[line + 2 * L + 1] = T.slot_mult[s0 + 8];
        }
    if ((e = upload(ctx, pr, &t.slot_mult_pair)) != cudaSuccess)
        return e;
    if ((e = upload(ctx, T.run_first, &t.run_first)) != cudaSuccess)
        return e;
    if ((e = upload(ctx, T.run_len, &t.run_len)) != cudaSuccess)
        return e;
    return upload(ctx, T.blk_run_begin, &t.blk_run_begin);
}

extern "C" const char *cvb_version(void) { return "covest_b200 0.2 (sm_100a)"; }

extern "C" int cvb_abi_version(void) { return CVB_ABI_VERSION; }

extern "C" const char *cvb_last_error(const cvb_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int cvb_n_param(const cvb_ctx *ctx) { return ctx ? ctx->desc.n_param : CVB_EINVAL; }

extern "C" int cvb_device_sm_count(const cvb_ctx *ctx) { return ctx ? ctx->n_sm : CVB_EINVAL; }

extern "C" void cvb_ctx_destroy(cvb_ctx *ctx)
{
    if (!ctx)
        return;
    cudaSetDevice(ctx->device);
    for (void *p : ctx->owned)
        cudaFree(p);
    void *bufs[] = {ctx->d_params, ctx->d_ll,      ctx->d_probs, ctx->d_cand_ll, ctx->d_sel_ll,
                    ctx->d_rows,   ctx->d_cand_idx, ctx->d_sel_idx, ctx->d_axes,   ctx->d_counter,
                    ctx->d_sink,   ctx->d_topk_scratch, ctx->d_marked, ctx->d_seg_key, ctx->d_seg_best,
                    ctx->d_seg_rows};
    for (void *p : bufs)
        if (p)
            cudaFree(p);
    for (cudaEvent_t e : ctx->ev)
        cudaEventDestroy(e);
    cvf_release(ctx->fw);
    if (ctx->copy_ev)
        cudaEventDestroy(ctx->copy_ev);
    if (ctx->copy_done)
        cudaEventDestroy(ctx->copy_done);
    if (ctx->order_ev)
        cudaEventDestroy(ctx->order_ev);
    if (ctx->copy_stream)
        cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream)
        cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int cvb_ctx_create(int model_kind, int k, int r, int max_error, int n_bins,
                              const int32_t *bin_j, const double *bin_h, double tail,
                              double threshold, const double *bounds, const double *comb,
                              const double *pow3, int device, cvb_ctx **out_ctx)
{
    cvb_ctx *ctx = nullptr; /* errors before the context exists go to the thread-local slot */
    if (!out_ctx)
        return fail(ctx, CVB_EINVAL, "out_ctx is NULL");
    *out_ctx = nullptr;
    if (model_kind != CVB_MODEL_BASIC && model_kind != CVB_MODEL_REPEATS)
        return fail(ctx, CVB_EINVAL, "model_kind must be 0 (basic) or 1 (repeats)");
    if (k < 1 || r < k)
        return fail(ctx, CVB_EINVAL, "need 1 <= k <= r");
    if (max_error < 1 || max_error > k + 1 || max_error > CV_MAX_ERR)
        return fail(ctx, CVB_EINVAL, "max_error must be in [1, min(k+1, 64)]");
    if (!bin_j || !bin_h || !bounds)
        return fail(ctx, CVB_EINVAL, "bin_j, bin_h and bounds are required");
    CvHostTables T;
    std::string why = cv_build_tables(n_bins, bin_j, bin_h, T);
    if (!why.empty())
        return fail(ctx, CVB_EINVAL, why);

    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(ctx, CVB_ECUDA,
                    std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0") +
                        " (libcovest_b200 has no CPU path)");
    }
    if (device < 0 || device >= n_dev)
        return fail(ctx, CVB_EINVAL, "device ordinal out of range");
    e = cudaSetDevice(device);
    if (e != cudaSuccess)
        return fail_cuda(ctx, e, "cudaSetDevice");

    cvb_ctx *c = new cvb_ctx();
    c->device = device;
    CvModelDesc &m = c->desc;
    memset(&m, 0, sizeof(m));
    m.model_kind = model_kind;
    m.k = k;
    m.r = r;
    m.n_err = max_error;
    m.n_param = model_kind ? 5 : 2;
    m.n_bins = n_bins;
    m.n_groups = T.n_groups;
    m.na = T.na;
    m.n_blocks = T.n_blocks;
    m.max_bin = T.max_bin;
    m.tail = tail;
    m.threshold = threshold;
    for (int i = 0; i < CV_MAX_PARAMS; i++) {
        m.lo[i] = i < m.n_param ? bounds[2 * i] : NAN;
        m.hi[i] = i < m.n_param ? bounds[2 * i + 1] : NAN;
    }
    for (int s = 0; s < max_error; s++) {
        if (comb) {
            m.comb[s] = comb[s];
        } else { /* C(k,s) * 3^s, exact in long double for every k <= 63 */
            long double v = 1.0L;
            for (int i = 1; i <= s; i++)
                v = v * (long double)(k - s + i) / (long double)i;
            m.comb[s] = (double)(v * powl(3.0L, (long double)s));
        }
        m.pow3[s] = pow3 ? pow3[s] : (s == 0 ? 1.0 : pow(3.0, (double)-s));
    }

    int rc = CVB_OK;
    do {
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
            break;
        c->n_sm = prop.multiProcessorCount;
        c->smem_max = (int)prop.sharedMemPerBlockOptin;
        if (prop.major < 10) {
            rc = fail(nullptr, CVB_ECUDA,
                      std::string("device is ") + prop.name + " (sm_" + std::to_string(prop.major) +
                          std::to_string(prop.minor) + "); this library holds sm_100a code only");
            break;
        }
        if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess)
            break;
        CvTables &t = m.tab;
        if (cv_loglik_smem_bytes(m, c->smem_max) < 0) {
            rc = fail(nullptr, CVB_EINVAL, "histogram too long: its group tables do not fit the shared memory of an SM");
            break;
        }
        if ((e = upload_profile_tables(c, T, t)) != cudaSuccess) break;
        if ((e = upload(c, T.slot_mult, &t.slot_mult)) != cudaSuccess) break;
        if ((e = upload(c, T.slot_h, &t.slot_h)) != cudaSuccess) break;
        if ((e = upload(c, T.slot_bin, &t.slot_bin)) != cudaSuccess) break;
        if ((e = upload(c, T.copy_log_h, &t.copy_log_h)) != cudaSuccess) break;
        if ((e = upload(c, T.copy_log_l, &t.copy_log_l)) != cudaSuccess) break;
        {
            /* rows of the profiles: the lines with counts, the others summed (COVEST_B200_ROWS=full: every line) */
            const char *rows = getenv("COVEST_B200_ROWS");
            const bool compact = !(rows && !strcmp(rows, "full"));
            /* without a tail the batched path evaluates the lines with counts alone (cv_build_row_tables);
             * O_thr (max_bin) and the copy logarithms stay those of the whole histogram */
            CvHostTables RT;
            const bool row_tables = compact && tail == 0.0 && cv_build_row_tables(T, bin_j, bin_h, RT);
            c->fdesc = m;
            if (row_tables) {
                CvModelDesc &f = c->fdesc;
                f.n_groups = RT.n_groups;
                f.na = RT.na;
                f.n_blocks = RT.n_blocks;
                /* the batched path reads the slots through its row layout (CvfSlots), not these */
                f.tab.slot_mult = f.tab.slot_h = nullptr;
                f.tab.slot_bin = nullptr;
                if ((e = upload_profile_tables(c, RT, f.tab)) != cudaSuccess) break;
            }
            const CvHostTables &FT = row_tables ? RT : T;
            std::vector<int> line_map;
            std::vector<double2> mh;
            std::vector<double> row_h;
            cvf_build_slots(FT.slot_mult, FT.slot_h, compact, row_tables, line_map, mh, row_h, &c->slots.sum_line);
            c->slots.nsteps = (int)(row_h.size() / 64);
            if ((e = upload(c, line_map, &c->slots.line_map)) != cudaSuccess) break;
            if ((e = upload(c, mh, &c->slots.slot_mh)) != cudaSuccess) break;
            if ((e = upload(c, cvf_step_masks(row_h), &c->slots.step_mask)) != cudaSuccess) break;
            c->slots.counts_first = cvf_counts_first(row_h);
            std::vector<double> lt(2 * CV_LOG_N);
            cv_log_table(lt.data());
            if ((e = upload(c, lt, &c->d_log_tab)) != cudaSuccess) break;
        }
        if (const char *pm = getenv("COVEST_B200_PATH"))
            c->path_mode = !strcmp(pm, "direct") ? 1 : !strcmp(pm, "factored") ? 2 : !strcmp(pm, "gemm") ? 3
                           : !strcmp(pm, "prefix") ? 4 : !strcmp(pm, "faithful") ? 5 : 0;
        if (const char *wl = getenv("COVEST_B200_PROFILE_MIB"))
            if (atoll(wl) > 0)
                c->w_limit = (size_t)atoll(wl) * (1 << 20) / sizeof(double);
        if (const char *po = getenv("COVEST_B200_POISON")) { /* tests: nan = bytes 0xFF, finite = 0x7F (~1.4e306) */
            c->poison = !strcmp(po, "nan") ? 0xFF : !strcmp(po, "finite") ? 0x7F : 0;
            if (!c->poison && *po) {
                rc = fail(nullptr, CVB_EINVAL, "COVEST_B200_POISON must be nan or finite");
                break;
            }
            c->fw.poison = c->poison;
        }
        { /* tables of the term-by-term re-evaluation (faithful.h): by bin index j - 1 */
            const int j_all = T.max_bin > 0 ? T.max_bin : 1;
            std::vector<double> cnt(j_all, -1.0), rcp(j_all);
            int j_counted = 0;
            for (int b = 0; b < n_bins; b++) {
                const int j = (int)bin_j[b];
                if (j >= 1 && j <= j_all) {
                    cnt[j - 1] = bin_h[b];
                    if (bin_h[b] != 0.0 && j > j_counted)
                        j_counted = j;
                }
            }
            for (int j = 1; j <= j_all; j++)
                rcp[j - 1] = 1.0 / (double)j;
            if ((e = upload(c, cnt, &c->faith.cnt_of_j)) != cudaSuccess) break;
            if ((e = upload(c, rcp, &c->faith.rcp)) != cudaSuccess) break;
            c->faith.j_all = j_all;
            c->faith.j_counted = j_counted;
            c->faith.acc_doubles = ((long long)j_all + 31) & ~31LL;
            void *scr = nullptr;
            if ((e = cudaMalloc(&scr, (size_t)cv_faithful_warps(c->n_sm) * (size_t)c->faith.acc_doubles * sizeof(double))) != cudaSuccess) break;
            c->owned.push_back(scr);
            c->faith.scratch = (double *)scr;
            if ((e = cudaMalloc((void **)&c->d_fixed, 4 * sizeof(unsigned long long))) != cudaSuccess) break;
            c->owned.push_back(c->d_fixed);
        }
        if ((e = cudaMalloc((void **)&c->d_counter, sizeof(unsigned long long))) != cudaSuccess) break;
        if ((e = cudaMalloc((void **)&c->d_sink, 64)) != cudaSuccess) break;
    } while (0);
    if (rc == CVB_OK && e != cudaSuccess)
        rc = fail_cuda(nullptr, e, "context setup");
    if (rc != CVB_OK) {
        cvb_ctx_destroy(c);
        return rc;
    }
    *out_ctx = c;
    return CVB_OK;
}

/* ---- timing ------------------------------------------------------------------------------- */
extern "C" int cvb_set_timing(cvb_ctx *ctx, int enabled)
{
    if (!ctx)
        return CVB_EINVAL;
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    if (enabled && ctx->ev.empty()) {
        ctx->ev.resize(2 * CVB_MAX_TIMED_CHUNKS);
        for (auto &e : ctx->ev)
            CU(cudaEventCreate(&e), "cudaEventCreate");
    }
    ctx->timing = enabled != 0;
    ctx->timed_chunks = 0;
    return CVB_OK;
}

extern "C" int cvb_last_kernel_ms(cvb_ctx *ctx, double *out_ms, int *out_launches)
{
    if (!ctx)
        return CVB_EINVAL;
    if (out_launches)
        *out_launches = ctx->last_launches;
    if (out_ms) {
        *out_ms = 0.0;
        if (!ctx->timing)
            return fail(ctx, CVB_EINVAL, "timing is off (cvb_set_timing)");
        CU(cudaSetDevice(ctx->device), "cudaSetDevice");
        for (int i = 0; i < ctx->timed_chunks; i++) {
            float ms = 0.f;
            CU(cudaEventSynchronize(ctx->ev[2 * i + 1]), "cudaEventSynchronize");
            CU(cudaEventElapsedTime(&ms, ctx->ev[2 * i], ctx->ev[2 * i + 1]), "cudaEventElapsedTime");
            *out_ms += ms;
        }
    }
    return CVB_OK;
}

/* one evaluation of n points on the device, optionally bracketed by events: the factored path
 * when the batch is large and groups well (never when per-bin probabilities are wanted), else the
 * per-point kernel */
static int launch_loglik(cvb_ctx *ctx, const CvLattice &lat, const double *const *lat_axes_host,
                         const double *d_params, long long n, int clip, double *d_ll, double *d_probs,
                         cudaStream_t s)
{
    bool timed = ctx->timing && ctx->timed_chunks < CVB_MAX_TIMED_CHUNKS;
    if (timed)
        CU(cudaEventRecord(ctx->ev[2 * ctx->timed_chunks], s), "cudaEventRecord");
    int used = 0;
    const bool forced = ctx->path_mode >= 2;
    const bool faithful_only = ctx->path_mode == 5 && !d_probs;
    const bool try_factored = !d_probs && ctx->path_mode != 1 && !faithful_only && cvf_supported(ctx->desc) &&
                              (forced || n >= ctx->min_points);
    if (faithful_only) {
        CU(cv_launch_mark_all(d_ll, n, s), "cv_mark_all_kernel launch");
        ctx->last_launches++;
        used = 3;
    }
    if (try_factored) {
        ctx->fw.timed = ctx->timing;
        CU(cvf_eval(ctx->fdesc, lat, lat_axes_host, d_params, n, clip, d_ll, ctx->slots,
                    ctx->d_log_tab, ctx->fw, ctx->n_sm,
                    ctx->smem_max, ctx->w_limit, forced ? 0.0 : ctx->min_group, ctx->min_run,
                    ctx->path_mode == 3 ? 1 : ctx->path_mode == 4 ? 2 : 0, s, &used),
           "factored evaluation");
        ctx->last_launches += ctx->fw.launches;
    }
    if (!used) {
        CU(cv_launch_loglik(ctx->desc, lat, d_params, n, clip, d_ll, d_probs, ctx->d_counter, ctx->n_sm,
                            ctx->smem_max, s),
           "cv_loglik_kernel launch");
        ctx->last_launches++;
    }
    ctx->last_path = used ? 1 + used : 1;
    /* points whose value hinges on the reference's subnormal roundings: again, term by term */
    CU(grow(&ctx->d_marked, &ctx->cap_marked, 2 * (size_t)n), "cudaMalloc(marked points)");
    CU(cv_launch_faithful(ctx->desc, lat, d_params, n, clip, d_ll, ctx->faith, ctx->n_sm, ctx->d_marked,
                          ctx->d_fixed, s),
       "cv_faithful_kernel launch");
    ctx->last_launches += 3; /* the scan for marked points, their re-evaluation (warp / CTA per point) */
    if (timed) {
        CU(cudaEventRecord(ctx->ev[2 * ctx->timed_chunks + 1], s), "cudaEventRecord");
        ctx->timed_chunks++;
    }
    return CVB_OK;
}

static int topk_device(cvb_ctx *ctx, const CvLattice &lat, const double *d_ll, const double *d_params,
                       long long n, int K, double *out_rows, cudaStream_t s);

/* COVEST_B200_POISON (tests): fill `doubles` of a scratch buffer with the context's byte pattern on the
 * call's stream, so that a kernel reading an element it did not write sees a NaN or a huge value instead
 * of a harmless leftover.  Only buffers of doubles: an index or a count read from poison could fault. */
static int poison_fill(cvb_ctx *ctx, void *buf, size_t doubles, cudaStream_t s)
{
    if (buf && doubles)
        CU(cudaMemsetAsync(buf, ctx->poison, doubles * sizeof(double), s), "cudaMemsetAsync(poison)");
    return CVB_OK;
}

static size_t faith_scratch_doubles(const cvb_ctx *ctx)
{
    return (size_t)cv_faithful_warps(ctx->n_sm) * (size_t)ctx->faith.acc_doubles;
}

/* stream ordering between the calls of one context (see cvb_ctx::order_ev) */
static int order_enter(cvb_ctx *ctx, cudaStream_t s)
{
    if (ctx->order_valid && ctx->last_stream != s)
        CU(cudaStreamWaitEvent(s, ctx->order_ev, 0), "cudaStreamWaitEvent");
    return CVB_OK;
}

static int order_leave(cvb_ctx *ctx, cudaStream_t s)
{
    if (!ctx->order_ev)
        CU(cudaEventCreateWithFlags(&ctx->order_ev, cudaEventDisableTiming), "cudaEventCreate");
    CU(cudaEventRecord(ctx->order_ev, s), "cudaEventRecord");
    ctx->last_stream = s;
    ctx->order_valid = true;
    return CVB_OK;
}

static int eval_batch(cvb_ctx *ctx, int64_t n_points, const double *params, int clip, double *out_p,
                      double *out_ll, int k_best, double *out_rows, void *stream)
{
    if (!ctx)
        return CVB_EINVAL;
    if (n_points < 0 || (n_points > 0 && !params))
        return fail(ctx, CVB_EINVAL, "n_points < 0 or params is NULL");
    if (!out_ll && !out_p && k_best <= 0)
        return fail(ctx, CVB_EINVAL, "no output buffer");
    if (k_best < 0 || (k_best > 0 && !out_rows))
        return fail(ctx, CVB_EINVAL, "k_best > 0 needs out_rows");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    ctx->timed_chunks = 0;
    ctx->last_launches = 0;
    if (n_points == 0 && k_best <= 0)
        return CVB_OK;
    if (int rc = order_enter(ctx, s))
        return rc;
    const int np = ctx->desc.n_param;
    const long long nb = ctx->desc.n_bins;
    const bool p_dev = is_device_ptr(params);
    const bool l_dev = out_ll ? is_device_ptr(out_ll) : true;
    const bool q_dev = out_p ? is_device_ptr(out_p) : true;
    const bool all_dev = p_dev && l_dev && q_dev;
    CvLattice lat;
    memset(&lat, 0, sizeof(lat));

    /* the row gather of a top-K needs the whole batch resident: no chunking then */
    long long chunk = (all_dev || k_best > 0) ? n_points : CVB_CHUNK_POINTS;
    if (chunk < 1)
        chunk = 1;
    if (out_p && !q_dev) { /* keep the probability staging buffer below ~1 GiB */
        long long lim = (1LL << 27) / (nb > 0 ? nb : 1);
        if (lim < 1)
            lim = 1;
        if (chunk > lim)
            chunk = lim;
    }
    if (chunk > n_points)
        chunk = n_points;
    if (!p_dev)
        CU(grow(&ctx->d_params, &ctx->cap_params, (size_t)chunk * np), "cudaMalloc(params staging)");
    if (!l_dev || !out_ll)
        CU(grow(&ctx->d_ll, &ctx->cap_ll, (size_t)chunk), "cudaMalloc(loglik staging)");
    const double *dp_all = p_dev ? params : ctx->d_params;
    const double *dl_all = (out_ll && l_dev) ? out_ll : ctx->d_ll;
    if (out_p && !q_dev)
        CU(grow(&ctx->d_probs, &ctx->cap_probs, (size_t)chunk * nb), "cudaMalloc(probs staging)");
    if (ctx->poison) {
        if (int rc = poison_fill(ctx, dl_all == ctx->d_ll ? ctx->d_ll : nullptr, (size_t)chunk, s))
            return rc;
        if (int rc = poison_fill(ctx, out_p && !q_dev ? ctx->d_probs : nullptr, (size_t)chunk * nb, s))
            return rc;
        if (int rc = poison_fill(ctx, ctx->faith.scratch, faith_scratch_doubles(ctx), s))
            return rc;
    }

    bool side_copy = false;
    for (long long off = 0; off < n_points; off += chunk) {
        long long n = n_points - off < chunk ? n_points - off : chunk;
        const double *dp = params + off * np;
        if (!p_dev) {
            CU(cudaMemcpyAsync(ctx->d_params, dp, (size_t)n * np * sizeof(double),
                               cudaMemcpyHostToDevice, s),
               "cudaMemcpyAsync(params)");
            dp = ctx->d_params;
        }
        double *dl = (out_ll && l_dev) ? out_ll + off : ctx->d_ll;
        double *dq = out_p ? (q_dev ? out_p + off * nb : ctx->d_probs) : nullptr;
        int rc = launch_loglik(ctx, lat, nullptr, dp, n, clip, dl, dq, s);
        if (rc != CVB_OK)
            return rc;
        if (out_ll && !l_dev) {
            /* with a top-K to follow the values leave on a stream of their own, next to it */
            cudaStream_t cs = s;
            if (k_best > 0 && n >= (1 << 16)) {
                if (!ctx->copy_stream)
                    CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
                if (!ctx->copy_ev)
                    CU(cudaEventCreateWithFlags(&ctx->copy_ev, cudaEventDisableTiming), "cudaEventCreate");
                if (!ctx->copy_done)
                    CU(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming), "cudaEventCreate");
                CU(cudaEventRecord(ctx->copy_ev, s), "cudaEventRecord");
                CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev, 0), "cudaStreamWaitEvent");
                cs = ctx->copy_stream;
                side_copy = true;
            }
            CU(cudaMemcpyAsync(out_ll + off, dl, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, cs),
               "cudaMemcpyAsync(loglik)");
            if (cs != s)
                CU(cudaEventRecord(ctx->copy_done, cs), "cudaEventRecord");
        }
        if (out_p && !q_dev)
            CU(cudaMemcpyAsync(out_p + off * nb, dq, (size_t)n * nb * sizeof(double),
                               cudaMemcpyDeviceToHost, s),
               "cudaMemcpyAsync(probs)");
        if (!all_dev && off + chunk < n_points)
            CU(cudaStreamSynchronize(s), "cudaStreamSynchronize"); /* staging is reused */
    }
    bool rows_to_host = false;
    if (k_best > 0) {
        int rc = topk_device(ctx, lat, dl_all, dp_all, n_points, k_best, out_rows, s);
        if (rc != CVB_OK)
            return rc;
        rows_to_host = !is_device_ptr(out_rows);
    }
    if (side_copy) /* the values left on the side stream: the main stream ends after them */
        CU(cudaStreamWaitEvent(s, ctx->copy_done, 0), "cudaStreamWaitEvent");
    if (int rc = order_leave(ctx, s))
        return rc;
    if (!all_dev || rows_to_host) /* one synchronisation per call, and only when something went to host memory */
        CU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}

extern "C" int cvb_loglik_batch(cvb_ctx *ctx, int64_t n_points, const double *params, double *out_ll,
                                void *stream)
{
    if (ctx && !out_ll)
        return fail(ctx, CVB_EINVAL, "out_ll is NULL");
    return eval_batch(ctx, n_points, params, 1, nullptr, out_ll, 0, nullptr, stream);
}

extern "C" int cvb_probs_batch(cvb_ctx *ctx, int64_t n_points, const double *params, int clip,
                               double *out_p, double *out_ll, void *stream)
{
    if (ctx && !out_p)
        return fail(ctx, CVB_EINVAL, "out_p is NULL");
    return eval_batch(ctx, n_points, params, clip ? 1 : 0, out_p, out_ll, 0, nullptr, stream);
}

extern "C" int cvb_loglik_topk(cvb_ctx *ctx, int64_t n_points, const double *params, double *out_ll,
                               int k_best, double *out_rows, void *stream)
{
    if (ctx && (k_best < 1 || !out_rows))
        return fail(ctx, CVB_EINVAL, "cvb_loglik_topk needs k_best >= 1 and out_rows");
    return eval_batch(ctx, n_points, params, 1, nullptr, out_ll, k_best, out_rows, stream);
}

/* ---- top-K -------------------------------------------------------------------------------- */
static int ensure_topk(cvb_ctx *ctx, int K)
{
    if (K <= ctx->cap_k)
        return CVB_OK;
    void *old[] = {ctx->d_cand_ll, ctx->d_cand_idx, ctx->d_sel_ll, ctx->d_sel_idx, ctx->d_rows};
    for (void *p : old)
        if (p)
            cudaFree(p);
    ctx->d_cand_ll = ctx->d_sel_ll = ctx->d_rows = nullptr;
    ctx->d_cand_idx = ctx->d_sel_idx = nullptr;
    ctx->cap_k = 0;
    ctx->topk_ctas = 2 * ctx->n_sm;
    size_t nc = (size_t)ctx->topk_ctas * K;
    CU(cudaMalloc((void **)&ctx->d_cand_ll, nc * sizeof(double)), "cudaMalloc(topk)");
    CU(cudaMalloc((void **)&ctx->d_cand_idx, nc * sizeof(long long)), "cudaMalloc(topk)");
    CU(cudaMalloc((void **)&ctx->d_sel_ll, (size_t)K * sizeof(double)), "cudaMalloc(topk)");
    CU(cudaMalloc((void **)&ctx->d_sel_idx, (size_t)K * sizeof(long long)), "cudaMalloc(topk)");
    CU(cudaMalloc((void **)&ctx->d_rows, (size_t)K * (1 + CV_MAX_PARAMS) * sizeof(double)),
       "cudaMalloc(topk)");
    ctx->cap_k = K;
    return CVB_OK;
}

/* d_ll: device, n entries.  params: device or null (lattice). */
static int topk_device(cvb_ctx *ctx, const CvLattice &lat, const double *d_ll, const double *d_params,
                       long long n, int K, double *out_rows, cudaStream_t s)
{
    int rc = ensure_topk(ctx, K);
    if (rc != CVB_OK)
        return rc;
    if (ctx->poison) { /* nothing of the call has used these buffers before the selection */
        if ((rc = poison_fill(ctx, ctx->d_cand_ll, (size_t)ctx->topk_ctas * K, s)))
            return rc;
        if ((rc = poison_fill(ctx, ctx->d_sel_ll, (size_t)K, s)))
            return rc;
        if ((rc = poison_fill(ctx, ctx->d_rows, (size_t)K * (1 + CV_MAX_PARAMS), s)))
            return rc;
    }
    if (n >= CVB_TOPK_RADIX_MIN && cv_topk_select_fits(n, K)) {
        /* large batch, few rows wanted: radix selection (topk.cu) */
        CU(grow(&ctx->d_topk_scratch, &ctx->cap_topk_scratch, cv_topk_select_bytes()), "cudaMalloc(topk scratch)");
        CU(cv_launch_topk_radix_select(d_ll, n, K, ctx->d_topk_scratch, ctx->n_sm, ctx->d_sel_ll, ctx->d_sel_idx, s),
           "top-K selection");
        ctx->last_launches += 1;
    } else if (n >= CVB_TOPK_RADIX_MIN && n <= 0x7fffffffLL) { /* large batch: one radix sort (topk.cu) */
        const size_t need = cv_topk_sort_bytes(n);
        CU(grow(&ctx->d_topk_scratch, &ctx->cap_topk_scratch, need), "cudaMalloc(topk scratch)");
        CU(cv_launch_topk_sort(d_ll, n, K, ctx->d_topk_scratch, ctx->cap_topk_scratch, ctx->d_sel_ll,
                               ctx->d_sel_idx, s),
           "top-K sort");
        ctx->last_launches += 12; /* keys, the passes of the radix sort, take */
    } else {
        int ctas = ctx->topk_ctas;
        if ((long long)ctas * 1024 > n) /* small inputs: fewer, fuller slices */
            ctas = (int)((n + 1023) / 1024);
        if (ctas < 1)
            ctas = 1;
        CU(cv_launch_topk(d_ll, n, K, ctx->d_cand_ll, ctx->d_cand_idx, ctas, ctx->d_sel_ll,
                          ctx->d_sel_idx, s),
           "cv_topk_select launch");
        ctx->last_launches += 2;
    }
    const int np = ctx->desc.n_param;
    const bool r_dev = is_device_ptr(out_rows);
    double *dr = r_dev ? out_rows : ctx->d_rows;
    CU(cv_launch_gather_rows(lat, d_params, np, ctx->d_sel_ll, ctx->d_sel_idx, K, dr, s),
       "cv_gather_rows launch");
    ctx->last_launches += 1; /* the row gather */
    if (!r_dev) /* the caller synchronises the stream before it returns */
        CU(cudaMemcpyAsync(out_rows, dr, (size_t)K * (1 + np) * sizeof(double), cudaMemcpyDeviceToHost, s),
           "cudaMemcpyAsync(rows)");
    return CVB_OK;
}

extern "C" int cvb_topk(cvb_ctx *ctx, int64_t n_points, const double *ll, const double *params,
                        int k_best, double *out_rows, void *stream)
{
    if (!ctx)
        return CVB_EINVAL;
    if (n_points < 0 || k_best < 1 || !out_rows || (n_points > 0 && (!ll || !params)))
        return fail(ctx, CVB_EINVAL, "bad arguments to cvb_topk");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    const int np = ctx->desc.n_param;
    ctx->last_launches = 0;
    if (int rc = order_enter(ctx, s))
        return rc;
    const double *dl = ll, *dp = params;
    if (n_points > 0 && !is_device_ptr(ll)) {
        CU(grow(&ctx->d_ll, &ctx->cap_ll, (size_t)n_points), "cudaMalloc(loglik staging)");
        if (ctx->poison)
            if (int rc = poison_fill(ctx, ctx->d_ll, (size_t)n_points, s))
                return rc;
        CU(cudaMemcpyAsync(ctx->d_ll, ll, (size_t)n_points * sizeof(double), cudaMemcpyHostToDevice, s),
           "cudaMemcpyAsync(ll)");
        dl = ctx->d_ll;
    }
    if (n_points > 0 && !is_device_ptr(params)) {
        CU(grow(&ctx->d_params, &ctx->cap_params, (size_t)n_points * np), "cudaMalloc(params staging)");
        CU(cudaMemcpyAsync(ctx->d_params, params, (size_t)n_points * np * sizeof(double),
                           cudaMemcpyHostToDevice, s),
           "cudaMemcpyAsync(params)");
        dp = ctx->d_params;
    }
    CvLattice lat;
    memset(&lat, 0, sizeof(lat));
    if (int rc = topk_device(ctx, lat, dl, dp, n_points, k_best, out_rows, s))
        return rc;
    if (int rc = order_leave(ctx, s))
        return rc;
    if (!is_device_ptr(out_rows))
        CU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}

/* ---- lattice ------------------------------------------------------------------------------ */
/* slices with host output from this size on are evaluated in parts (measured on cfg3, 10^6 points: two parts cost
 * 0.11 ms of a 1.7 ms call on one GPU -- shorter K1 / K2p launches leave SMs idle at their ends) */
#define CVB_LATTICE_PART_MIN ((int64_t)1 << 22)

/* The set-up of a lattice call (cvb_lattice_eval, cvb_lattice_profile): the stream ordering of the
 * context, the axes and the slice checked, the axes on the device, `lat` and the host axes filled in. */
static int lattice_setup(cvb_ctx *ctx, const int32_t *axis_len, const double *axis_values, int64_t first,
                         int64_t stride, int64_t block, int64_t count, cudaStream_t s, CvLattice &lat,
                         const double **axes_host)
{
    const int np = ctx->desc.n_param;
    ctx->timed_chunks = 0;
    ctx->last_launches = 0;
    if (int rc = order_enter(ctx, s))
        return rc;
    size_t total_vals = 0;
    double total_pts = 1.0;
    for (int a = 0; a < np; a++) {
        if (axis_len[a] < 1)
            return fail(ctx, CVB_EINVAL, "empty lattice axis");
        total_vals += (size_t)axis_len[a];
        total_pts *= (double)axis_len[a];
    }
    if (count > 0) {
        const int64_t last_run = (count - 1) / block, last_in = (count - 1) % block;
        if (((double)first + (double)last_run * (double)stride) * (double)block + (double)last_in >= total_pts)
            return fail(ctx, CVB_EINVAL, "lattice slice runs past the end of the lattice");
    }
    CU(grow(&ctx->d_axes, &ctx->cap_axes, total_vals), "cudaMalloc(axes)");
    CU(cudaMemcpyAsync(ctx->d_axes, axis_values, total_vals * sizeof(double), cudaMemcpyHostToDevice, s),
       "cudaMemcpyAsync(axes)");
    memset(&lat, 0, sizeof(lat));
    lat.enabled = 1;
    lat.n_axes = np;
    size_t at = 0;
    for (int a = 0; a < np; a++) {
        lat.len[a] = axis_len[a];
        lat.axis[a] = ctx->d_axes + at;
        at += (size_t)axis_len[a];
    }
    lat.first = first;
    lat.stride = stride;
    lat.block = block;
    for (int a = 0; a < CV_MAX_PARAMS; a++)
        axes_host[a] = nullptr;
    at = 0;
    for (int a = 0; a < np; a++) {
        axes_host[a] = axis_values + at;
        at += (size_t)axis_len[a];
    }
    return CVB_OK;
}

/* Where a lattice call's values go: `out_dev` (device) or else the context's staging buffer, which is
 * grown to `count` values; under COVEST_B200_POISON the staging and the term-by-term scratch are filled. */
static int lattice_values(cvb_ctx *ctx, double *out_dev, int64_t count, cudaStream_t s, double **dl)
{
    *dl = out_dev;
    if (!*dl) {
        CU(grow(&ctx->d_ll, &ctx->cap_ll, (size_t)(count > 0 ? count : 1)), "cudaMalloc(loglik staging)");
        *dl = ctx->d_ll;
    }
    if (ctx->poison) {
        if (int rc = poison_fill(ctx, out_dev ? nullptr : ctx->d_ll, (size_t)(count > 0 ? count : 1), s))
            return rc;
        if (int rc = poison_fill(ctx, ctx->faith.scratch, faith_scratch_doubles(ctx), s))
            return rc;
    }
    return CVB_OK;
}

extern "C" int cvb_lattice_eval(cvb_ctx *ctx, const int32_t *axis_len, const double *axis_values,
                                int64_t first, int64_t stride, int64_t block, int64_t count,
                                double *out_ll, int k_best, double *out_rows, void *stream)
{
    if (!ctx)
        return CVB_EINVAL;
    if (!axis_len || !axis_values || first < 0 || stride < 1 || block < 1 || count < 0)
        return fail(ctx, CVB_EINVAL, "bad lattice arguments");
    if (k_best < 0 || (k_best > 0 && !out_rows))
        return fail(ctx, CVB_EINVAL, "k_best > 0 needs out_rows");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    const int np = ctx->desc.n_param;
    CvLattice lat;
    const double *axes_host[CV_MAX_PARAMS];
    if (int rc = lattice_setup(ctx, axis_len, axis_values, first, stride, block, count, s, lat, axes_host))
        return rc;
    const bool l_dev = out_ll && is_device_ptr(out_ll);
    double *dl = nullptr;
    if (int rc = lattice_values(ctx, l_dev ? out_ll : nullptr, count, s, &dl))
        return rc;
    bool need_sync = false, side_copy = false;
    /* A long slice whose values go to host memory is evaluated in parts of whole runs (and whole
     * (coverage, error_rate) groups), so that the values of a part travel while the next part is
     * evaluated: at 8 bytes per point the copy is otherwise up to a third of the call (cfg5: 100 MB per
     * rank; and the ranks of a box finish together and share the way to host memory). */
    int64_t part = 0;
    if (out_ll && !l_dev && count >= CVB_LATTICE_PART_MIN) {
        int64_t unit = block;
        if (block == 1 && stride == 1 && np == 5)
            unit = (int64_t)axis_len[2] * axis_len[3] * axis_len[4];
        /* parts of about 2^21 points, at most eight */
        int64_t n_parts = count >> 21;
        n_parts = n_parts < 2 ? 2 : n_parts > 8 ? 8 : n_parts;
        const int64_t want = (count + n_parts - 1) / n_parts;
        if (unit >= 1 && unit <= want && (block > 1 || first % unit == 0))
            part = (want + unit - 1) / unit * unit;
    }
    if (part > 0) {
        if (!ctx->copy_stream)
            CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
        if (!ctx->copy_ev)
            CU(cudaEventCreateWithFlags(&ctx->copy_ev, cudaEventDisableTiming), "cudaEventCreate");
        if (!ctx->copy_done)
            CU(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming), "cudaEventCreate");
        for (int64_t off = 0; off < count; off += part) {
            const int64_t n_part = count - off < part ? count - off : part;
            CvLattice lp = lat;
            lp.first = first + (off / block) * stride;
            int rc = launch_loglik(ctx, lp, axes_host, nullptr, n_part, 1, dl + off, nullptr, s);
            if (rc != CVB_OK)
                return rc;
            CU(cudaEventRecord(ctx->copy_ev, s), "cudaEventRecord");
            CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev, 0), "cudaStreamWaitEvent");
            CU(cudaMemcpyAsync(out_ll + off, dl + off, (size_t)n_part * sizeof(double), cudaMemcpyDeviceToHost,
                               ctx->copy_stream),
               "cudaMemcpyAsync(loglik)");
        }
        CU(cudaEventRecord(ctx->copy_done, ctx->copy_stream), "cudaEventRecord");
        side_copy = true;
        need_sync = true;
    } else if (count > 0) {
        int rc = launch_loglik(ctx, lat, axes_host, nullptr, count, 1, dl, nullptr, s);
        if (rc != CVB_OK)
            return rc;
    }
    if (out_ll && !l_dev && count > 0 && part == 0) {
        cudaStream_t cs = s;
        if (k_best > 0 && count >= (1 << 16)) { /* the values leave next to the top-K, on a stream of their own */
            if (!ctx->copy_stream)
                CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
            if (!ctx->copy_ev)
                CU(cudaEventCreateWithFlags(&ctx->copy_ev, cudaEventDisableTiming), "cudaEventCreate");
            if (!ctx->copy_done)
                CU(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming), "cudaEventCreate");
            CU(cudaEventRecord(ctx->copy_ev, s), "cudaEventRecord");
            CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->copy_ev, 0), "cudaStreamWaitEvent");
            cs = ctx->copy_stream;
            side_copy = true;
        }
        CU(cudaMemcpyAsync(out_ll, dl, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, cs),
           "cudaMemcpyAsync(loglik)");
        if (side_copy)
            CU(cudaEventRecord(ctx->copy_done, cs), "cudaEventRecord");
        need_sync = true;
    }
    if (k_best > 0) {
        int rc = topk_device(ctx, lat, dl, nullptr, count, k_best, out_rows, s);
        if (rc != CVB_OK)
            return rc;
        need_sync = need_sync || !is_device_ptr(out_rows);
    }
    if (side_copy)
        CU(cudaStreamWaitEvent(s, ctx->copy_done, 0), "cudaStreamWaitEvent");
    if (int rc = order_leave(ctx, s))
        return rc;
    if (need_sync)
        CU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}

extern "C" int cvb_lattice_profile(cvb_ctx *ctx, const int32_t *axis_len, const double *axis_values,
                                   int64_t first, int64_t stride, int64_t block, int64_t count,
                                   uint32_t keep_mask, double *out_rows, void *stream)
{
    if (!ctx)
        return CVB_EINVAL;
    if (!axis_len || !axis_values || first < 0 || stride < 1 || block < 1 || count < 0)
        return fail(ctx, CVB_EINVAL, "bad lattice arguments");
    if (!out_rows)
        return fail(ctx, CVB_EINVAL, "out_rows is NULL");
    const int np = ctx->desc.n_param;
    if (keep_mask == 0)
        return fail(ctx, CVB_EINVAL, "keep_mask is 0: a profile keeps at least one axis");
    if (keep_mask >> np)
        return fail(ctx, CVB_EINVAL, "keep_mask has a bit at or above n_param");
    int64_t n_seg = 1; /* an empty axis is refused by lattice_setup */
    for (int a = 0; a < np; a++)
        if (((keep_mask >> a) & 1) && axis_len[a] > 0 && __builtin_mul_overflow(n_seg, (int64_t)axis_len[a], &n_seg))
            return fail(ctx, CVB_EINVAL, "the number of segments (product of the kept axis lengths) overflows int64");
    int64_t row_bytes = 0;
    if (__builtin_mul_overflow(n_seg, (int64_t)((1 + np) * sizeof(double)), &row_bytes))
        return fail(ctx, CVB_EINVAL, "the rows of the segments overflow an int64 byte count");
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaStream_t s = stream ? (cudaStream_t)stream : ctx->stream;
    CvLattice lat;
    const double *axes_host[CV_MAX_PARAMS];
    if (int rc = lattice_setup(ctx, axis_len, axis_values, first, stride, block, count, s, lat, axes_host))
        return rc;
    double *dl = nullptr;
    if (int rc = lattice_values(ctx, nullptr, count, s, &dl))
        return rc;
    if (count > 0)
        if (int rc = launch_loglik(ctx, lat, axes_host, nullptr, count, 1, dl, nullptr, s))
            return rc;
    CU(grow(&ctx->d_seg_key, &ctx->cap_seg_key, (size_t)n_seg), "cudaMalloc(segment keys)");
    CU(grow(&ctx->d_seg_best, &ctx->cap_seg_best, (size_t)n_seg), "cudaMalloc(segment indices)");
    const bool r_dev = is_device_ptr(out_rows);
    double *dr = out_rows;
    if (!r_dev) {
        CU(grow(&ctx->d_seg_rows, &ctx->cap_seg_rows, (size_t)n_seg * (1 + np)), "cudaMalloc(segment rows)");
        dr = ctx->d_seg_rows;
        if (ctx->poison)
            if (int rc = poison_fill(ctx, dr, (size_t)n_seg * (1 + np), s))
                return rc;
    }
    CU(cv_launch_lattice_profile(lat, keep_mask, dl, count, n_seg, ctx->d_seg_key, ctx->d_seg_best, dr, ctx->n_sm, s),
       "lattice profile launch");
    ctx->last_launches += count > 0 ? 4 : 2;
    if (!r_dev)
        CU(cudaMemcpyAsync(out_rows, dr, (size_t)row_bytes, cudaMemcpyDeviceToHost, s), "cudaMemcpyAsync(rows)");
    if (int rc = order_leave(ctx, s))
        return rc;
    if (!r_dev) /* one synchronisation, and only when the rows went to host memory */
        CU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}

extern "C" int cvb_merge_rows(const double *rows, int n_rows, int n_cols, int k_best, double *out_rows,
                              void *stream)
{
    if (!rows || !out_rows || n_rows < 0 || n_rows > 2048 || n_cols < 1 || k_best < 1)
        return CVB_EINVAL;
    if (!is_device_ptr(rows) || !is_device_ptr(out_rows))
        return CVB_EINVAL;
    cudaError_t e = cv_launch_merge_rows(rows, n_rows, n_cols, k_best, out_rows, (cudaStream_t)stream);
    return e == cudaSuccess ? CVB_OK : CVB_ECUDA;
}

/* ---- path selection and facts about the last evaluation -------------------------------------- */
extern "C" int cvb_set_path(cvb_ctx *ctx, int mode)
{
    if (!ctx)
        return CVB_EINVAL;
    if (mode < 0 || mode > 5)
        return fail(ctx, CVB_EINVAL, "path mode must be 0 (auto), 1 (per-point), 2 (factored), 3 (factored, GEMM), "
                                     "4 (factored, prefix kernel) or 5 (term by term)");
    ctx->path_mode = mode;
    return CVB_OK;
}

extern "C" int cvb_last_path_info(cvb_ctx *ctx, double *out, int n_out)
{
    if (!ctx || !out || n_out < 1)
        return CVB_EINVAL;
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    double v[CVB_PATH_INFO_LEN] = {0};
    v[0] = ctx->last_path;
    {
        unsigned long long fixed = 0; /* waits for the work queued on the device */
        CU(cudaMemcpy(&fixed, ctx->d_fixed, sizeof(fixed), cudaMemcpyDeviceToHost), "cudaMemcpy");
        v[9] = (double)fixed;
    }
    if (ctx->last_path >= 2) {
        v[10] = (double)ctx->fw.analytic;
        v[11] = (double)(ctx->slots.nsteps * 64 - (ctx->slots.sum_line >= 0 ? 32 : 0));
        const CvFactorWork &w = ctx->fw;
        v[1] = (double)w.n_groups;
        v[2] = (double)w.n_tiles;
        v[3] = (double)w.n_items;
        v[4] = (double)w.w_doubles;
        v[8] = (double)w.n_runs;
        if (w.timed && w.ev[0]) {
            float ms = 0.f;
            CU(cudaEventSynchronize(w.ev[3]), "cudaEventSynchronize");
            CU(cudaEventElapsedTime(&ms, w.ev[0], w.ev[1]), "cudaEventElapsedTime");
            v[5] = ms; /* keys, sort, group tables (includes one host synchronisation) */
            CU(cudaEventElapsedTime(&ms, w.ev[1], w.ev[2]), "cudaEventElapsedTime");
            v[6] = ms; /* profiles (and the tiles of all but the last group range) */
            CU(cudaEventElapsedTime(&ms, w.ev[2], w.ev[3]), "cudaEventElapsedTime");
            v[7] = ms; /* tiles of the last group range */
        }
    }
    for (int i = 0; i < n_out && i < CVB_PATH_INFO_LEN; i++)
        out[i] = v[i];
    return CVB_OK;
}

/* ---- roofline probe ----------------------------------------------------------------------- */
extern "C" int cvb_fp64_peak(cvb_ctx *ctx, int kind, int reps, double *out_tflops)
{
    if (!ctx || !out_tflops || (kind < 0 || kind > 2))
        return ctx ? fail(ctx, CVB_EINVAL, "bad arguments to cvb_fp64_peak") : CVB_EINVAL;
    CU(cudaSetDevice(ctx->device), "cudaSetDevice");
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a), "cudaEventCreate");
    CU(cudaEventCreate(&b), "cudaEventCreate");
    double best = 0.0, flop = 0.0;
    if (reps < 1)
        reps = 1;
    for (int rep = 0; rep < reps + 1; rep++) { /* first pass warms up */
        CU(cudaEventRecord(a, ctx->stream), "cudaEventRecord");
        CU(cv_launch_peak_probe(kind, ctx->n_sm * 8, 4096, ctx->d_sink, &flop, ctx->stream),
           "cv_peak_probe launch");
        CU(cudaEventRecord(b, ctx->stream), "cudaEventRecord");
        CU(cudaEventSynchronize(b), "cudaEventSynchronize");
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, a, b), "cudaEventElapsedTime");
        if (rep > 0 && ms > 0.f) {
            double tf = flop / (ms * 1e-3) / 1e12;
            if (tf > best)
                best = tf;
        }
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *out_tflops = best;
    return CVB_OK;
}

/* ---- k-mer counting (kmers.cu) ------------------------------------------------------------ */
#define CVB_KMER_STAGE ((int64_t)64 << 20) /* bytes of one of the two pinned staging buffers of host input */

struct cvb_kmer_table {
    int device = 0;
    int n_sm = 0;
    CvkTable t = {};
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr; /* host -> device copies of staged parts */
    cudaEvent_t copied[2] = {nullptr, nullptr};   /* the copy out of pinned[b] has finished */
    cudaEvent_t consumed[2] = {nullptr, nullptr}; /* the kernel reading staged[b] has finished */
    unsigned char *pinned[2] = {nullptr, nullptr};
    unsigned char *staged[2] = {nullptr, nullptr};
    long long *d_hist = nullptr; /* histogram staging when the output is host memory */
    size_t cap_hist = 0;
    long long *h_words = nullptr; /* pinned: CVK_STATE_WORDS words read back */
    cudaEvent_t order_ev = nullptr; /* as cvb_ctx: a call on another stream waits for the previous call */
    cudaStream_t last_stream = nullptr;
    bool order_valid = false;
    std::string err;
};

static int kfail(cvb_kmer_table *t, int code, const std::string &msg)
{
    if (t)
        t->err = msg;
    else
        g_create_error = msg;
    return code;
}

#define KU(call, what)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return kfail(t, CVB_ECUDA, std::string(what) + ": " + cudaGetErrorString(e_));   \
    } while (0)

static int kmer_enter(cvb_kmer_table *t, void *stream, cudaStream_t *s)
{
    KU(cudaSetDevice(t->device), "cudaSetDevice");
    *s = stream ? (cudaStream_t)stream : t->stream;
    if (t->order_valid && t->last_stream != *s)
        KU(cudaStreamWaitEvent(*s, t->order_ev, 0), "cudaStreamWaitEvent");
    return CVB_OK;
}

static int kmer_leave(cvb_kmer_table *t, cudaStream_t s)
{
    if (!t->order_ev)
        KU(cudaEventCreateWithFlags(&t->order_ev, cudaEventDisableTiming), "cudaEventCreate");
    KU(cudaEventRecord(t->order_ev, s), "cudaEventRecord");
    t->last_stream = s;
    t->order_valid = true;
    return CVB_OK;
}

extern "C" const char *cvb_kmer_last_error(const cvb_kmer_table *t)
{
    return t ? t->err.c_str() : g_create_error.c_str();
}

extern "C" void cvb_kmer_table_destroy(cvb_kmer_table *t)
{
    if (!t)
        return;
    cudaSetDevice(t->device);
    if (t->stream)
        cudaStreamSynchronize(t->stream);
    if (t->copy_stream)
        cudaStreamSynchronize(t->copy_stream);
    for (int b = 0; b < 2; b++) {
        if (t->copied[b])
            cudaEventDestroy(t->copied[b]);
        if (t->consumed[b])
            cudaEventDestroy(t->consumed[b]);
        if (t->pinned[b])
            cudaFreeHost(t->pinned[b]);
        if (t->staged[b])
            cudaFree(t->staged[b]);
    }
    if (t->h_words)
        cudaFreeHost(t->h_words);
    void *bufs[] = {t->t.slots, t->t.state, t->d_hist};
    for (void *p : bufs)
        if (p)
            cudaFree(p);
    if (t->order_ev)
        cudaEventDestroy(t->order_ev);
    if (t->copy_stream)
        cudaStreamDestroy(t->copy_stream);
    if (t->stream)
        cudaStreamDestroy(t->stream);
    delete t;
}

extern "C" int cvb_kmer_table_create(int k, int64_t capacity, int part, int n_parts, int device,
                                     cvb_kmer_table **out)
{
    cvb_kmer_table *t = nullptr; /* errors before the table exists go to the thread-local slot */
    if (!out)
        return kfail(t, CVB_EINVAL, "out is NULL");
    *out = nullptr;
    if (k < 1 || k > 31)
        return kfail(t, CVB_EINVAL, "k must lie in [1, 31], not " + std::to_string(k));
    if (capacity < 1 || (capacity & (capacity - 1)) || capacity > ((int64_t)1 << 36))
        return kfail(t, CVB_EINVAL, "capacity must be a power of two in [1, 2^36], not " + std::to_string(capacity));
    if (n_parts < 1 || n_parts > 65536 || part < 0 || part >= n_parts)
        return kfail(t, CVB_EINVAL, "need 0 <= part < n_parts <= 65536, not part " + std::to_string(part) +
                                        " of " + std::to_string(n_parts));
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return kfail(t, CVB_ECUDA, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0") +
                                       " (libcovest_b200 has no CPU path)");
    }
    if (device < 0 || device >= n_dev)
        return kfail(t, CVB_EINVAL, "device ordinal out of range");
    if ((e = cudaSetDevice(device)) != cudaSuccess)
        return kfail(t, CVB_ECUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    t = new cvb_kmer_table();
    t->device = device;
    t->t.k = k;
    t->t.mask = (unsigned long long)capacity - 1;
    const unsigned long long reserve = capacity / 8 > 1 ? (unsigned long long)capacity / 8 : 1;
    t->t.limit = (unsigned long long)capacity - reserve;
    t->t.part = (unsigned int)part;
    t->t.n_parts = (unsigned int)n_parts;
    int rc = CVB_OK;
    do {
        cudaDeviceProp prop;
        if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
            break;
        t->n_sm = prop.multiProcessorCount;
        if (prop.major < 10) {
            rc = kfail(nullptr, CVB_ECUDA, std::string("device is ") + prop.name + "; this library holds sm_100a code only");
            break;
        }
        if ((e = cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking)) != cudaSuccess)
            break;
        if ((e = cudaMalloc((void **)&t->t.slots, (size_t)capacity * sizeof(CvkSlot))) != cudaSuccess) {
            rc = kfail(nullptr, CVB_ENOMEM, "cudaMalloc of " + std::to_string(capacity) + " slots (" +
                                                std::to_string((size_t)capacity * sizeof(CvkSlot)) + " bytes): " +
                                                cudaGetErrorString(e));
            cudaGetLastError();
            break;
        }
        if ((e = cudaMalloc((void **)&t->t.state, CVK_STATE_WORDS * sizeof(unsigned long long))) != cudaSuccess)
            break;
        if ((e = cudaMallocHost((void **)&t->h_words, CVK_STATE_WORDS * sizeof(long long))) != cudaSuccess)
            break;
        if ((e = cvk_launch_clear(t->t, t->n_sm, t->stream)) != cudaSuccess)
            break;
        e = cudaStreamSynchronize(t->stream);
    } while (0);
    if (rc == CVB_OK && e != cudaSuccess)
        rc = kfail(nullptr, CVB_ECUDA, std::string("k-mer table setup: ") + cudaGetErrorString(e));
    if (rc != CVB_OK) {
        cvb_kmer_table_destroy(t);
        return rc;
    }
    *out = t;
    return CVB_OK;
}

extern "C" int cvb_kmer_clear(cvb_kmer_table *t, void *stream)
{
    if (!t)
        return CVB_EINVAL;
    cudaStream_t s;
    if (int rc = kmer_enter(t, stream, &s))
        return rc;
    KU(cvk_launch_clear(t->t, t->n_sm, s), "k-mer clear launch");
    return kmer_leave(t, s);
}

/* the two pinned and two device staging buffers of host input, made on first use */
static int kmer_staging(cvb_kmer_table *t)
{
    if (t->copy_stream)
        return CVB_OK;
    for (int b = 0; b < 2; b++) {
        KU(cudaMallocHost((void **)&t->pinned[b], CVB_KMER_STAGE), "cudaMallocHost(k-mer staging)");
        KU(cudaMalloc((void **)&t->staged[b], CVB_KMER_STAGE), "cudaMalloc(k-mer staging)");
        KU(cudaEventCreateWithFlags(&t->copied[b], cudaEventDisableTiming), "cudaEventCreate");
        KU(cudaEventCreateWithFlags(&t->consumed[b], cudaEventDisableTiming), "cudaEventCreate");
    }
    KU(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    return CVB_OK;
}

extern "C" int cvb_kmer_count(cvb_kmer_table *t, const uint8_t *seq, int64_t n, void *stream)
{
    if (!t)
        return CVB_EINVAL;
    if (n < 0 || (n > 0 && !seq))
        return kfail(t, CVB_EINVAL, "need n >= 0 and a buffer");
    cudaStream_t s;
    if (int rc = kmer_enter(t, stream, &s))
        return rc;
    if (n == 0)
        return kmer_leave(t, s);
    if (is_device_ptr(seq)) {
        KU(cvk_launch_count(t->t, seq, n, t->n_sm, s), "k-mer count launch");
        return kmer_leave(t, s);
    }
    if (int rc = kmer_staging(t))
        return rc;
    /* Parts of at most CVB_KMER_STAGE bytes; each after the first repeats the k - 1 bytes before it, so
     * that every window of the buffer lies whole in exactly one part.  The host copies part i into
     * pinned[i % 2] while the device copies and counts part i - 1. */
    const int64_t halo = t->t.k - 1;
    int64_t start = 0;
    for (int64_t i = 0; start < n; i++) {
        const int b = (int)(i & 1);
        const int64_t lo = i == 0 ? 0 : start - halo;
        const int64_t hi = std::min(n, lo + CVB_KMER_STAGE);
        if (i >= 2)
            KU(cudaEventSynchronize(t->copied[b]), "cudaEventSynchronize");
        memcpy(t->pinned[b], seq + lo, (size_t)(hi - lo));
        if (i >= 2)
            KU(cudaStreamWaitEvent(t->copy_stream, t->consumed[b], 0), "cudaStreamWaitEvent");
        KU(cudaMemcpyAsync(t->staged[b], t->pinned[b], (size_t)(hi - lo), cudaMemcpyHostToDevice, t->copy_stream),
           "cudaMemcpyAsync(k-mer part)");
        KU(cudaEventRecord(t->copied[b], t->copy_stream), "cudaEventRecord");
        KU(cudaStreamWaitEvent(s, t->copied[b], 0), "cudaStreamWaitEvent");
        KU(cvk_launch_count(t->t, t->staged[b], hi - lo, t->n_sm, s), "k-mer count launch");
        KU(cudaEventRecord(t->consumed[b], s), "cudaEventRecord");
        start = hi;
    }
    if (int rc = kmer_leave(t, s))
        return rc;
    KU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}

extern "C" int cvb_kmer_stats(cvb_kmer_table *t, int64_t out[4], void *stream)
{
    if (!t)
        return CVB_EINVAL;
    if (!out)
        return kfail(t, CVB_EINVAL, "out is NULL");
    cudaStream_t s;
    if (int rc = kmer_enter(t, stream, &s))
        return rc;
    KU(cudaMemsetAsync(t->t.state + CVK_DISTINCT, 0, 3 * sizeof(unsigned long long), s), "cudaMemsetAsync");
    KU(cvk_launch_stats(t->t, t->n_sm, s), "k-mer stats launch");
    const bool dev = is_device_ptr(out);
    KU(cudaMemcpyAsync(dev ? (void *)out : (void *)t->h_words, t->t.state, 4 * sizeof(int64_t),
                       dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s),
       "cudaMemcpyAsync(stats)");
    if (int rc = kmer_leave(t, s))
        return rc;
    if (!dev) {
        KU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
        memcpy(out, t->h_words, 4 * sizeof(int64_t));
    }
    return CVB_OK;
}

extern "C" int cvb_kmer_histogram(cvb_kmer_table *t, int64_t n_bins, int64_t *out_hist, void *stream)
{
    if (!t)
        return CVB_EINVAL;
    if (n_bins < 1 || !out_hist)
        return kfail(t, CVB_EINVAL, "need n_bins >= 1 and an output buffer");
    cudaStream_t s;
    if (int rc = kmer_enter(t, stream, &s))
        return rc;
    /* a table that dropped a k-mer has no right histogram: read the count first (one synchronisation) */
    KU(cudaMemcpyAsync(t->h_words + CVK_DROPPED, t->t.state + CVK_DROPPED, sizeof(long long), cudaMemcpyDeviceToHost, s),
       "cudaMemcpyAsync(dropped)");
    KU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    if (int rc = kmer_leave(t, s))
        return rc;
    const long long dropped = t->h_words[CVK_DROPPED];
    if (dropped)
        return kfail(t, CVB_ENOMEM, "the k-mer table is full: " + std::to_string(dropped) +
                                        " k-mers were dropped (a larger table or more parts holds them)");
    const bool dev = is_device_ptr(out_hist);
    long long *dh = (long long *)out_hist;
    if (!dev) {
        KU(grow(&t->d_hist, &t->cap_hist, (size_t)n_bins), "cudaMalloc(histogram)");
        dh = t->d_hist;
    }
    KU(cudaMemsetAsync(dh, 0, (size_t)n_bins * sizeof(long long), s), "cudaMemsetAsync(histogram)");
    KU(cvk_launch_histogram(t->t, n_bins, dh, t->n_sm, s), "k-mer histogram launch");
    if (!dev)
        KU(cudaMemcpyAsync(out_hist, dh, (size_t)n_bins * sizeof(long long), cudaMemcpyDeviceToHost, s),
           "cudaMemcpyAsync(histogram)");
    if (int rc = kmer_leave(t, s))
        return rc;
    if (!dev)
        KU(cudaStreamSynchronize(s), "cudaStreamSynchronize");
    return CVB_OK;
}
