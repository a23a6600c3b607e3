/*
 * covest_b200.h -- C ABI of libcovest_b200.so, the B200 (sm_100a) implementation of CovEst's
 * likelihood hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / CUDA types.  The caller in
 * the reference is Python (covest/models.py); the binding a maintainer would add is a ctypes stub
 * (INTEGRATION.md shows it; covest_b200/_capi.py is this repo's own).  Reference lines are relative
 * to the upstream mhozza/covest tree.
 *
 * Conventions
 *   - every function returns 0 on success and a negative CVB_E* code on failure; the message is
 *     available from cvb_last_error(ctx) (ctx may be NULL for the error of a failed create);
 *   - the caller owns every buffer it passes; a context owns device copies of the histogram and
 *     the tables derived from it;
 *   - buffer arguments documented "host or device" are inspected with cudaPointerGetAttributes:
 *     device pointers are used in place, host pointers are staged through context-owned device
 *     buffers (the copies are part of the call);
 *   - `stream` is a cudaStream_t passed as void* (NULL = the context's own stream; name the default
 *     stream with cudaStreamLegacy, (void*)1).  Calls with
 *     host buffers return after the results are in the host buffer (one stream synchronisation per
 *     call); calls where all buffers are device pointers only enqueue work on the stream -- with one
 *     exception: cvb_loglik_batch / cvb_loglik_topk on an explicit point array that takes the
 *     factored path (cvb_set_path) synchronise the stream once, because the general plan reads the
 *     group and tile counts back to size its workspace.  cvb_lattice_eval never does: the plan of a
 *     lattice follows from its axes;
 *   - a context is bound to one device and is not re-entrant; its calls share scratch memory, so a
 *     call issued on a different stream than the previous call of the same context first waits
 *     (on the device) for that call's work; distinct contexts are independent;
 *   - there is no CPU fallback: without a CUDA device every call fails with CVB_ECUDA.
 */
#ifndef COVEST_B200_H
#define COVEST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define CVB_API __attribute__((visibility("default")))
#else
#define CVB_API
#endif

#define CVB_OK 0
#define CVB_EINVAL (-1) /* bad argument */
#define CVB_ECUDA (-2)  /* CUDA runtime error (cvb_last_error has cudaGetErrorString) */
#define CVB_ENOMEM (-3)

#define CVB_MODEL_BASIC 0   /* covest/models.py:17  BasicModel   params (coverage, error_rate) */
#define CVB_MODEL_REPEATS 1 /* covest/models.py:173 RepeatsModel params + (q1, q2, q) */

typedef struct cvb_ctx cvb_ctx;

/* Replaces the state BasicModel.__init__ / RepeatsModel.__init__ keep (covest/models.py:19-31,
 * :175-183).
 *   k, r        k-mer size and read length
 *   max_error   number of error classes S actually summed (models.py:28-31: min(k+1, max_error))
 *   n_bins      len(hist); bin_j[b] / bin_h[b] are the keys and counts of `hist` in dict order
 *   tail        models.py:27
 *   threshold   models.py:183 (repeats only); NaN = None (no cut-off)
 *   bounds      n_param x 2 doubles (lo, hi) as models.py:23 / :179; NaN = open end
 *   comb        max_error doubles comb[s] = C(k,s) * 3**s exactly as the host computed them
 *               (models.py:25 uses scipy's floating comb); NULL = computed here in long double
 *   pow3        max_error doubles 3 ** -s as the host computed them (models.py:77); NULL = here
 *   device      CUDA device ordinal
 */
CVB_API int cvb_ctx_create(int model_kind, int k, int r, int max_error, int n_bins, const int32_t *bin_j,
                   const double *bin_h, double tail, double threshold, const double *bounds,
                   const double *comb, const double *pow3, int device, cvb_ctx **out_ctx);

CVB_API void cvb_ctx_destroy(cvb_ctx *ctx);

CVB_API const char *cvb_last_error(const cvb_ctx *ctx);

/* Replaces compute_loglikelihood (models.py:100-107) mapped over a batch, i.e.
 * compute_loglikelihood_multi (models.py:109-117): out_ll[i] = loglikelihood of params row i
 * (row-major n_points x n_param), arguments clipped to the bounds first (fit_to_bounds,
 * models.py:60-69).  params / out_ll: host or device. */
CVB_API int cvb_loglik_batch(cvb_ctx *ctx, int64_t n_points, const double *params, double *out_ll,
                     void *stream);

/* Replaces compute_probabilities (models.py:81-98, :211-242) over a batch: out_p is row-major
 * n_points x n_bins, column b pairs with bin_j[b].  clip = 0 evaluates at the arguments as given
 * (what compute_probabilities does), clip = 1 clips first.  out_ll may be NULL.
 * params / out_p / out_ll: host or device. */
CVB_API int cvb_probs_batch(cvb_ctx *ctx, int64_t n_points, const double *params, int clip, double *out_p,
                    double *out_ll, void *stream);

/* The K best rows of a batch already evaluated: out_rows is row-major K x (1 + n_param),
 * (loglik, params...), best first; ties resolved towards the lower index, NaN never preferred;
 * rows beyond n_points are (-inf, NaN...).  Replaces the arg-max over Pool.map results in
 * covest/grid.py:61-69 and covest/covest.py:69-78.  All buffers host or device. */
CVB_API int cvb_topk(cvb_ctx *ctx, int64_t n_points, const double *ll, const double *params, int k_best,
             double *out_rows, void *stream);

/* cvb_loglik_batch followed by cvb_topk in one call: the batch is staged once, out_ll may be NULL
 * (only the best rows are wanted: what one round of covest/grid.py:56-69 consumes). */
CVB_API int cvb_loglik_topk(cvb_ctx *ctx, int64_t n_points, const double *params, double *out_ll,
                            int k_best, double *out_rows, void *stream);

/* Merge of best-row blocks, the step after the all-gather of a multi-GPU round (the arg-max over
 * the Pool.map results of covest/grid.py:61-69 when the candidates were split over ranks): `rows`
 * holds n_rows <= 2048 rows of n_cols doubles (column 0 = log-likelihood), out_rows receives the
 * k_best best, best first.  Order: larger log-likelihood first (NaN as -inf), ties by the other
 * columns in ascending lexicographic order (NaN last), so the result does not depend on the number
 * of ranks.  Device buffers only; the work is enqueued on `stream` (NULL = the legacy default
 * stream).  Needs no context; returns 0 or a negative error code. */
CVB_API int cvb_merge_rows(const double *rows, int n_rows, int n_cols, int k_best, double *out_rows,
                           void *stream);

/* A Cartesian lattice of candidate points generated on the device (no host->device parameter
 * traffic): n_param axes, axis a has axis_len[a] values stored consecutively in axis_values
 * (host), last axis fastest -- the order of itertools.product in covest/grid.py:33.  The call
 * takes runs of `block` consecutive lattice indices: point i is the lattice index
 * (first + (i / block) * stride) * block + i % block.  block = 1 is the strided slice
 * first + i * stride; block = the number of (q1, q2, q) combinations hands whole
 * (coverage, error_rate) groups to a rank, which is how the ranks of a multi-GPU run shard a
 * repeats-model lattice (each group's bin profiles are then computed on one rank only).
 * Evaluates `count` points; out_ll (host or device, may be NULL) receives them; if k_best > 0,
 * out_rows (host or device) receives the k_best best rows as in cvb_topk.  With a host out_ll a
 * slice of 2^22 points or more is evaluated in parts of about 2^21 points (whole runs, whole
 * (coverage, error_rate) groups): the values of a part travel while the next part is evaluated;
 * values and rows are those of one evaluation. */
CVB_API int cvb_lattice_eval(cvb_ctx *ctx, const int32_t *axis_len, const double *axis_values,
                     int64_t first, int64_t stride, int64_t block, int64_t count, double *out_ll,
                     int k_best, double *out_rows, void *stream);

/* The best point of every segment of a lattice slice: the building block of a profile likelihood
 * (for each value of the kept parameters, the best log-likelihood over the others).  The lattice and
 * the slice are those of cvb_lattice_eval (same arguments, same values).  Bit a of keep_mask set keeps
 * axis a; the segment of a point is the mixed-radix number of its kept-axis digits in axis order, the
 * last kept axis fastest, and n_seg is the product of the kept axes' lengths.  out_rows (host or
 * device) receives n_seg rows of (1 + n_param) doubles, row-major: for each segment (loglik, params...)
 * of its best slice point in the order of cvb_topk -- larger value first, NaN as -inf, -0 tied with +0,
 * ties to the lower lattice index -- with the value cvb_topk reports for it (a NaN as -inf) and the
 * axis values bit for bit.  A segment with no point in the slice gets (-inf, NaN...); a segment whose
 * points are all -inf or NaN gets -inf and the axis values of its lowest lattice index.  For strictly
 * increasing axes "lower lattice index" and "lexicographically smaller params" are the same, which is
 * the tie-break of cvb_merge_rows: per-rank rows of a sharded lattice merge segment by segment into
 * the rows of one call.  With a device out_rows the call only enqueues work; with a host out_rows it
 * synchronises the stream once.  CVB_EINVAL for keep_mask == 0, a bit at or above n_param, or an n_seg
 * (or its rows' byte count) that does not fit an int64. */
CVB_API int cvb_lattice_profile(cvb_ctx *ctx, const int32_t *axis_len, const double *axis_values,
                                int64_t first, int64_t stride, int64_t block, int64_t count,
                                uint32_t keep_mask, double *out_rows, void *stream);

/* Measures the FP64 roofline denominator on the context's device: kind 0 = dependent-free DFMA
 * chains, kind 1 = DMMA m8n8k4 chains, kind 2 = both at once (half of the warps each), all register
 * resident.  *out_tflops = best of `reps`. */
CVB_API int cvb_fp64_peak(cvb_ctx *ctx, int kind, int reps, double *out_tflops);

/* Device time (ms, CUDA events on the launch stream) of the dominant kernel of the most recent
 * cvb_loglik_batch / cvb_probs_batch / cvb_lattice_eval call, and how many kernels that call
 * launched.  Timing is only recorded after cvb_set_timing(ctx, 1). */
CVB_API int cvb_set_timing(cvb_ctx *ctx, int enabled);
CVB_API int cvb_last_kernel_ms(cvb_ctx *ctx, double *out_ms, int *out_launches);

/* Evaluation path of the repeats model.  A batch is evaluated either point by point
 * (cv_loglik_kernel: one warp per point, reference models.py:211-242 term by term) or *factored*:
 * the per-copy-number bin profiles sum_s a_os * tp(o * l_s, j) -- the inner sum of models.py:236 --
 * are computed once per distinct (coverage, error_rate) of the batch and contracted with the copy
 * weights b(o) of every point (models.py:193-208) -- by an FP64 tensor-core GEMM, or, when points
 * of a (c, e) group also share q (lattices: grid.py:25-33, :95-98), by the *prefix kernel*: b(o) is
 * geometric beyond o = 2 (models.py:196-208), so one running sum over the copy numbers serves every
 * cut-off of such a q-run.  mode 0 = automatic (factored for batches of >= 2048 points with >= 12
 * points per distinct (c, e); prefix kernel at >= 4 points per q-run), 1 = per-point only,
 * 2 = factored whenever the model supports it, 3 = factored with the GEMM, 4 = factored with the
 * prefix kernel, 5 = every point term by term in the reference's order of operations (the kernel
 * that otherwise re-evaluates only points with subnormal bin probabilities; slow, a check).  The environment variable COVEST_B200_PATH=direct|factored|gemm|prefix|auto sets
 * the initial mode.  The factored path holds the repeats model with max_error <= 32 only: for the
 * basic model and for max_error > 32, modes 0 and 2-4 run the per-point kernel.  Per-bin
 * probabilities (cvb_probs_batch) always use the per-point kernel. */
CVB_API int cvb_set_path(cvb_ctx *ctx, int mode);

/* Facts about the most recent evaluation: out[0] = path used (1 per-point, 2 factored with the
 * GEMM, 3 factored with the prefix kernel); for the factored path out[1] = distinct (c, e) groups,
 * out[2] = tiles, out[3] = profile items (16 copy numbers each), out[4] = doubles of profile
 * workspace, out[5..7] = device ms of the planning kernels, the profile kernel and the GEMM /
 * prefix kernel (after cvb_set_timing(ctx, 1)), out[8] = q-runs (0 when the GEMM ordering ran);
 * out[9] = points of the call that were re-evaluated term by term because a bin with a count had a
 * probability in the subnormal range, where the reference's per-term roundings decide the value
 * (reading it waits for the device); out[10] = 1 when the plan of the batch came from lattice axes
 * (no sort, nothing read back); out[11] = slots of a profile row in the factored path: 64 per line
 * of the histogram tables that holds a bin with a count, plus 32 sums over all other lines when
 * there are any (a bin without a count enters the result through the mass only). */
#define CVB_PATH_INFO_LEN 12
CVB_API int cvb_last_path_info(cvb_ctx *ctx, double *out, int n_out);

/* number of model parameters of the context (2 or 5), number of SMs of its device */
CVB_API int cvb_n_param(const cvb_ctx *ctx);
CVB_API int cvb_device_sm_count(const cvb_ctx *ctx);
CVB_API const char *cvb_version(void);

/* ---- k-mer counting (DESIGN.md section 11) ------------------------------------------------------
 * The step before an estimate: canonical k-mers of sequence bytes counted in a device hash table,
 * and the abundance histogram a context is created from.  A table has its own handle (a likelihood
 * context needs a histogram to exist) and follows the conventions above: 0 or a negative CVB_E*,
 * the message from cvb_kmer_last_error(t) (t may be NULL for a failed create), `stream` as void*
 * (NULL = the table's own stream), host or device buffers, and one synchronisation per call with a
 * host buffer.  Calls of one table on different streams are ordered as those of a context.
 *
 * The table is open-addressed with linear probing over `capacity` (a power of two, at most 2^36)
 * 16-byte slots: a uint64 key, the 2-bit packed canonical k-mer (the smaller of the k-mer and its
 * reverse complement, A=0 C=1 G=2 T=3), and a uint64 count.  At most capacity - max(1, capacity / 8)
 * slots are ever occupied; a k-mer that finds no room then is *dropped* (counted, not inserted).
 * With n_parts > 1 the table holds only the k-mers of part `part`, chosen by hash bits of the key
 * that do not pick its slot: tables of parts 0..n_parts-1 together hold every k-mer once. */
typedef struct cvb_kmer_table cvb_kmer_table;

/* CVB_EINVAL for k outside [1, 31], a capacity that is not a power of two in [1, 2^36] and part
 * outside [0, n_parts); CVB_ENOMEM when the device cannot hold the slots.  The table starts empty. */
CVB_API int cvb_kmer_table_create(int k, int64_t capacity, int part, int n_parts, int device,
                                  cvb_kmer_table **out);
CVB_API void cvb_kmer_table_destroy(cvb_kmer_table *t);
CVB_API const char *cvb_kmer_last_error(const cvb_kmer_table *t);

/* empties the table and zeroes its statistics */
CVB_API int cvb_kmer_clear(cvb_kmer_table *t, void *stream);

/* Counts every window of k consecutive bases of seq[0, n) (host or device).  A base is one of
 * ACGTacgt; any other byte (N, IUPAC codes, a separator between reads) ends the windows through it.
 * Nothing is kept between calls: a k-mer across two calls is not counted, so cut at read
 * boundaries.  A host buffer is staged through two pinned buffers of the table; the copy of one part
 * overlaps the counting of the previous one. */
CVB_API int cvb_kmer_count(cvb_kmer_table *t, const uint8_t *seq, int64_t n, void *stream);

/* out (host or device) = {distinct k-mers, total k-mers (sum of counts), largest count, dropped
 * k-mers} of the table (of its part). */
CVB_API int cvb_kmer_stats(cvb_kmer_table *t, int64_t out[4], void *stream);

/* out_hist[j - 1] (host or device, n_bins >= 1 entries) = number of distinct k-mers seen exactly j
 * times; counts above n_bins go into out_hist[n_bins - 1].  Reads the dropped count first, so the call
 * always synchronises the stream once; if anything was dropped it returns CVB_ENOMEM with the count in
 * the message and leaves out_hist as it was. */
CVB_API int cvb_kmer_histogram(cvb_kmer_table *t, int64_t n_bins, int64_t *out_hist, void *stream);

/* Bumped whenever a signature or the meaning of an argument changes; a binding compares it with
 * the version it was written against before it calls anything else (covest_b200/_capi.py). */
#define CVB_ABI_VERSION 2
CVB_API int cvb_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif
