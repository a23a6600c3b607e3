/*
 * kernels.h -- launch interface between the C-ABI (capi.cu) and the sm_100a kernels (kernels.cu).
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "cvpoint.h"

/* A Cartesian lattice of parameter points generated on the device, decoded with the LAST axis
 * varying fastest (the order of itertools.product, which grid.py:33 uses for its candidate
 * grids).  A launch takes runs of `block` consecutive lattice indices: point i is the lattice
 * index (first + (i / block) * stride) * block + i % block -- with block = 1 the strided slice
 * first + i * stride, with block = the number of (q1, q2, q) combinations whole (c, e) groups. */
struct CvLattice {
    int enabled;
    int n_axes;
    int len[CV_MAX_PARAMS];
    const double *axis[CV_MAX_PARAMS]; /* device pointers */
    long long first, stride, block;
};

/* K1/K2: log-likelihood (and optionally the per-bin probabilities) of n_points points.
 * `params` (device, row-major n_points x n_param) is ignored when lat.enabled.
 * `counter` is a device word the persistent warps draw point indices from; zeroed here.
 * `smem_max` is cudaDevAttrMaxSharedMemoryPerBlockOptin of the device. */
cudaError_t cv_launch_loglik(const CvModelDesc &m, const CvLattice &lat, const double *params,
                             long long n_points, int clip, double *out_ll, double *out_probs,
                             unsigned long long *counter, int n_sm, int smem_max, cudaStream_t stream);

/* K3: rows of the K largest log-likelihoods (ties: lower index first; NaN never selected before
 * a number).  out_idx/out_ll: device, K entries, descending (missing entries: -inf, -1).
 * cand_*: device scratch, n_cta * K entries. */
cudaError_t cv_launch_topk(const double *ll, long long n_points, int K, double *cand_ll,
                           long long *cand_idx, int n_cta, double *out_ll, long long *out_idx,
                           cudaStream_t stream);

/* K3 for large batches (topk.cu): the same selection by one stable descending radix sort of
 * order-preserving keys.  `scratch`: device, cv_topk_sort_bytes(n) bytes. */
size_t cv_topk_sort_bytes(long long n);
/* merge of best-row blocks of several ranks: n <= 2048 rows of c doubles -> the k best, device buffers */
cudaError_t cv_launch_merge_rows(const double *rows, int n, int c, int k, double *out, cudaStream_t stream);

/* large n, K <= 1024: radix selection (topk.cu) */
size_t cv_topk_select_bytes(void);
bool cv_topk_select_fits(long long n, int K);
cudaError_t cv_launch_topk_radix_select(const double *ll, long long n, int K, void *scratch, int n_sm,
                                        double *out_ll, long long *out_idx, cudaStream_t stream);

cudaError_t cv_launch_topk_sort(const double *ll, long long n, int K, void *scratch, size_t scratch_bytes,
                                double *out_ll, long long *out_idx, cudaStream_t stream);

/* gathers rows (ll, params...) for selected indices; params from a buffer or from the lattice */
cudaError_t cv_launch_gather_rows(const CvLattice &lat, const double *params, int n_param,
                                  const double *sel_ll, const long long *sel_idx, int K,
                                  double *out_rows, cudaStream_t stream);

/* Best row per segment of a lattice slice (profile.cu): `ll` (device, n values) are the values of the
 * slice points of `lat`; the segment of a point is the mixed-radix number of the digits of the axes set
 * in keep_mask (axis order, last kept axis fastest).  out_rows (device, n_seg x (1 + n_axes)) receives
 * per segment (value, axis values...) of its best point: larger value first, NaN as -inf, -0 tied with
 * +0, ties to the lower lattice index; (-inf, NaN...) for a segment without a point.  seg_key /
 * seg_best: device scratch of n_seg words each, initialised here. */
cudaError_t cv_launch_lattice_profile(const CvLattice &lat, unsigned int keep_mask, const double *ll, long long n,
                                      long long n_seg, unsigned long long *seg_key, unsigned long long *seg_best,
                                      double *out_rows, int n_sm, cudaStream_t stream);

/* Register-resident FP64 micro-benchmarks for the roofline denominator (DESIGN.md section 6):
 * kind 0 = DFMA chains, kind 1 = DMMA m8n8k4 chains.  Returns flop executed. */
cudaError_t cv_launch_peak_probe(int kind, int n_cta, int iters, double *sink, double *flop,
                                 cudaStream_t stream);

/* dynamic shared memory of a cv_loglik_kernel CTA given the opt-in limit of the device */
int cv_loglik_smem_bytes(const CvModelDesc &m, int smem_max);
