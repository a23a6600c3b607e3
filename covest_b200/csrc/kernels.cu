/*
 * kernels.cu -- hand-written sm_100a kernels of the CovEst likelihood path.
 *
 *   cv_loglik_kernel   K1/K2: one WARP per parameter point, up to 16 warps in the one CTA of an SM
 *                      (persistent warps drawing point indices from a device counter), phases of
 *                      cvpoint.h separated by __syncwarp() -- no CTA-wide barrier after the row
 *                      tables are staged.  FP64 throughout; the inner loop is one DFMA per
 *                      (mixture term, bin) with operands read from shared memory as 16-byte pairs.
 *   cv_topk_select     K3: deterministic top-K of the log-likelihoods.
 *   cv_gather_rows     (ll, params...) rows of the selected points.
 *   cv_peak_probe      register-resident DFMA / DMMA chains: the measured FP64 roofline.
 *
 * Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 (covest_b200/build.py)
 */
#include "kernels.h"

#include "kdevice.h"

__device__ __forceinline__ CvPartial cv_partial_shfl_down(const CvPartial &p, int delta)
{
    CvPartial q;
    q.sum = __shfl_down_sync(CV_FULL_MASK, p.sum, delta);
    q.mass_h = __shfl_down_sync(CV_FULL_MASK, p.mass_h, delta);
    q.mass_l = __shfl_down_sync(CV_FULL_MASK, p.mass_l, delta);
    return q;
}

/* All blocks of one point: for every block the tiles of mixture terms are prepared (one term per
 * lane) and contracted into the lane's accumulators, then the block is finished bin by bin. */
template <int NA>
__device__ __forceinline__ void cv_point_blocks(int lane, const CvModelDesc &m, CvWarpMem &M,
                                                CvPartial &part, double *probs_row)
{
    const int S = m.n_err;
    const int cpg = cv_copies_per_group(S);
    for (int blk = 0; blk < m.n_blocks; blk++) {
        const CvLaneGroup G = cv_lane_group(lane, m, blk, M);
        double acc[4 * NA];
#pragma unroll
        for (int i = 0; i < 4 * NA; i++)
            acc[i] = 0.0;
        /* passes of 32 copy numbers: lane i holds b(first + i); the copies before the first
         * lane that reports the cut-off are evaluated (models.py:185-191) */
        for (int first = 1;; first += 32) {
            double b;
            bool stop = cv_w_copy_pass(lane, m, M, first, &b);
            const unsigned stop_mask = __ballot_sync(CV_FULL_MASK, stop);
            const int nlive = stop_mask ? __ffs(stop_mask) - 1 : 32;
            for (int g = 0; g < nlive; g += cpg) {
                const int ncop = min(cpg, nlive - g);
                const int nterms = ncop * S;
                cv_w_mass(lane, m, first + g, nterms, S, M);
                __syncwarp();
                for (int sub = 0; sub < nterms; sub += CV_CT) {
                    int src = g + (sub + lane) / S; /* the lane that holds this term's b(o) */
                    double bt = __shfl_sync(CV_FULL_MASK, b, src < 31 ? src : 31);
                    const CvTerm tm = cv_w_term(lane, m, first + g, nterms, S, sub, bt, M);
                    cv_w_prep<NA>(lane, m, blk, tm, M);
                    __syncwarp();
                    const int nkg = (min(CV_CT, nterms - sub) + 3) >> 2;
                    cv_w_fused<NA>(lane, G, 0, nkg, *M.fx, acc);
                    __syncwarp();
                }
            }
            if (stop_mask)
                break;
        }
        cv_w_spill<NA>(lane, *M.fx, acc);
        __syncwarp();
        cv_w_epilogue<NA>(lane, m, blk, min(CV_GB, m.n_groups - blk * CV_GB), *M.fx, part, probs_row);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(32 * CV_WARPS_MAX, 1)
cv_loglik_kernel(const __grid_constant__ CvModelDesc m, const __grid_constant__ CvLattice lat,
                 const double *__restrict__ params, long long n_points, int clip,
                 double *__restrict__ out_ll, double *__restrict__ out_probs,
                 unsigned long long *counter, int groups_staged)
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
    __syncthreads(); /* the only CTA-wide barrier: from here on every warp is on its own */

    for (;;) {
        long long point = 0;
        if (lane == 0)
            point = (long long)atomicAdd(counter, 1ULL);
        point = __shfl_sync(CV_FULL_MASK, point, 0);
        if (point >= n_points)
            break;
        double row[CV_MAX_PARAMS];
        if (lat.enabled) {
            cv_lattice_point(lat, point, row);
        } else {
#pragma unroll
            for (int i = 0; i < CV_MAX_PARAMS; i++)
                row[i] = i < m.n_param ? params[point * m.n_param + i] : 0.0;
        }
        __syncwarp(); /* the previous point's readers of the working set are done */
        cv_w_header(lane, m, row, clip, M);
        __syncwarp();

        CvPartial part = {0.0, 0.0, 0.0};
        double *probs_row = out_probs ? out_probs + point * (long long)m.n_bins : nullptr;
        switch (m.na) {
        case 1: cv_point_blocks<1>(lane, m, M, part, probs_row); break;
        case 2: cv_point_blocks<2>(lane, m, M, part, probs_row); break;
        case 4: cv_point_blocks<4>(lane, m, M, part, probs_row); break;
        default: cv_point_blocks<8>(lane, m, M, part, probs_row); break;
        }
        /* warp reduction of the partial sums in a fixed order */
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            CvPartial q = cv_partial_shfl_down(part, d);
            cv_partial_merge(part, q);
        }
        if (lane == 0)
            out_ll[point] = cv_point_finish(m, part);
    }
}

/* warps per CTA and staged groups that fit the shared memory of an SM */
static void cv_loglik_config(const CvModelDesc &m, int smem_max, int *n_warps, int *groups_staged,
                             size_t *smem_bytes)
{
    const size_t wb = cv_warp_bytes(m.n_err);
    const int groups = m.n_blocks * CV_GB;
    const size_t tab = (size_t)groups * CV_GD * sizeof(double);
    long long w = ((long long)smem_max - (long long)tab) / (long long)wb;
    if (w > CV_WARPS_MAX)
        w = CV_WARPS_MAX;
    if (w < 1)
        w = 0; /* the group tables do not fit next to one warp: the caller reports it */
    *n_warps = (int)w;
    *groups_staged = groups;
    *smem_bytes = tab + (size_t)w * wb;
}

int cv_loglik_smem_bytes(const CvModelDesc &m, int smem_max)
{
    int w, r;
    size_t b;
    cv_loglik_config(m, smem_max, &w, &r, &b);
    return w < 1 ? -1 : (int)b;
}

cudaError_t cv_launch_loglik(const CvModelDesc &m, const CvLattice &lat, const double *params,
                             long long n_points, int clip, double *out_ll, double *out_probs,
                             unsigned long long *counter, int n_sm, int smem_max, cudaStream_t stream)
{
    int n_warps, groups_staged;
    size_t smem;
    cv_loglik_config(m, smem_max, &n_warps, &groups_staged, &smem);
    if (n_warps < 1)
        return cudaErrorInvalidConfiguration; /* ctx_create refuses such histograms */
    /* per device, and cheap: set on every launch */
    cudaError_t e = cudaFuncSetAttribute(cv_loglik_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess)
        return e;
    if (n_points <= 0)
        return cudaSuccess;
    e = cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream);
    if (e != cudaSuccess)
        return e;
    /* one persistent CTA per SM; a small batch is spread over the SMs first (fewer warps per CTA) */
    if (n_points < (long long)n_sm * n_warps) {
        int w = (int)((n_points + n_sm - 1) / n_sm);
        smem -= (size_t)(n_warps - w) * cv_warp_bytes(m.n_err);
        n_warps = w;
    }
    long long ctas = (n_points + n_warps - 1) / n_warps;
    int grid = (int)(ctas < n_sm ? ctas : n_sm);
    cv_loglik_kernel<<<grid, 32 * n_warps, smem, stream>>>(m, lat, params, n_points, clip, out_ll,
                                                           out_probs, counter, groups_staged);
    return cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------- */
/* K3: top-K.  Total order: larger ll first, then lower index; NaN counts as -inf.              */
/* ------------------------------------------------------------------------------------------- */
struct CvKey {
    double v;
    long long i;
};

__device__ __forceinline__ bool cv_key_before(const CvKey &a, const CvKey &b)
{
    return a.v > b.v || (a.v == b.v && a.i < b.i);
}

__device__ __forceinline__ double cv_key_value(double v) { return (v != v) ? -INFINITY : v; }

/* Each CTA selects the K best keys of its slice [cta * chunk, ...) of (vals, idxs).  idxs may be
 * null (index = position).  Output: out_v/out_i[cta * K + k], descending; missing = (-inf, -1)
 * ordered last (index LLONG_MAX internally). */
__global__ void __launch_bounds__(256)
cv_topk_select(const double *__restrict__ vals, const long long *__restrict__ idxs, long long n,
               long long chunk, int K, double *__restrict__ out_v, long long *__restrict__ out_i)
{
    __shared__ CvKey s_best[8];
    __shared__ CvKey s_prev;
    const int tid = threadIdx.x;
    long long lo = (long long)blockIdx.x * chunk;
    long long hi = lo + chunk < n ? lo + chunk : n;
    CvKey prev = {INFINITY, -1}; /* before every real key */
    for (int k = 0; k < K; k++) {
        CvKey best = {-INFINITY, 0x7fffffffffffffffLL};
        for (long long p = lo + tid; p < hi; p += blockDim.x) {
            CvKey c = {cv_key_value(vals[p]), idxs ? idxs[p] : p};
            if (c.i < 0)
                continue; /* padding of an earlier stage */
            if (cv_key_before(prev, c) && cv_key_before(c, best))
                best = c;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            CvKey o;
            o.v = __shfl_down_sync(CV_FULL_MASK, best.v, d);
            o.i = __shfl_down_sync(CV_FULL_MASK, best.i, d);
            if (cv_key_before(o, best))
                best = o;
        }
        if ((tid & 31) == 0)
            s_best[tid >> 5] = best;
        __syncthreads();
        if (tid == 0) {
            CvKey b = s_best[0];
            for (int w = 1; w < (int)(blockDim.x >> 5); w++)
                if (cv_key_before(s_best[w], b))
                    b = s_best[w];
            s_prev = b;
            bool none = (b.i == 0x7fffffffffffffffLL);
            out_v[(long long)blockIdx.x * K + k] = none ? -INFINITY : b.v;
            out_i[(long long)blockIdx.x * K + k] = none ? -1 : b.i;
        }
        __syncthreads();
        prev = s_prev;
        __syncthreads();
    }
}

cudaError_t cv_launch_topk(const double *ll, long long n_points, int K, double *cand_ll,
                           long long *cand_idx, int n_cta, double *out_ll, long long *out_idx,
                           cudaStream_t stream)
{
    if (n_cta < 1)
        n_cta = 1;
    long long chunk = (n_points + n_cta - 1) / n_cta;
    if (chunk < 1)
        chunk = 1;
    cv_topk_select<<<n_cta, 256, 0, stream>>>(ll, nullptr, n_points, chunk, K, cand_ll, cand_idx);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        return e;
    long long n2 = (long long)n_cta * K;
    cv_topk_select<<<1, 256, 0, stream>>>(cand_ll, cand_idx, n2, n2, K, out_ll, out_idx);
    return cudaGetLastError();
}

__global__ void cv_gather_rows(const __grid_constant__ CvLattice lat, const double *__restrict__ params,
                               int n_param, const double *__restrict__ sel_ll,
                               const long long *__restrict__ sel_idx, int K,
                               double *__restrict__ out_rows)
{
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K)
        return;
    double *o = out_rows + (long long)k * (1 + n_param);
    long long i = sel_idx[k];
    o[0] = sel_ll[k];
    if (i < 0) {
        for (int a = 0; a < n_param; a++)
            o[1 + a] = NAN;
        return;
    }
    if (lat.enabled) {
        double row[CV_MAX_PARAMS];
        cv_lattice_point(lat, i, row);
        for (int a = 0; a < n_param; a++)
            o[1 + a] = row[a];
    } else {
        for (int a = 0; a < n_param; a++)
            o[1 + a] = params[i * n_param + a];
    }
}

cudaError_t cv_launch_gather_rows(const CvLattice &lat, const double *params, int n_param,
                                  const double *sel_ll, const long long *sel_idx, int K,
                                  double *out_rows, cudaStream_t stream)
{
    cv_gather_rows<<<(K + 127) / 128, 128, 0, stream>>>(lat, params, n_param, sel_ll, sel_idx, K,
                                                        out_rows);
    return cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------- */
/* FP64 peak probes                                                                             */
/* ------------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(256) cv_peak_probe_dfma(int iters, double *sink)
{
    double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-9 * blockIdx.x;
    double x0 = 0.1, x1 = 0.2, x2 = 0.3, x3 = 0.4, x4 = 0.5, x5 = 0.6, x6 = 0.7, x7 = 0.8;
    double y0 = 0.15, y1 = 0.25, y2 = 0.35, y3 = 0.45, y4 = 0.55, y5 = 0.65, y6 = 0.75, y7 = 0.85;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            x0 = __fma_rn(x0, a, b);
            x1 = __fma_rn(x1, a, b);
            x2 = __fma_rn(x2, a, b);
            x3 = __fma_rn(x3, a, b);
            x4 = __fma_rn(x4, a, b);
            x5 = __fma_rn(x5, a, b);
            x6 = __fma_rn(x6, a, b);
            x7 = __fma_rn(x7, a, b);
            y0 = __fma_rn(y0, a, b);
            y1 = __fma_rn(y1, a, b);
            y2 = __fma_rn(y2, a, b);
            y3 = __fma_rn(y3, a, b);
            y4 = __fma_rn(y4, a, b);
            y5 = __fma_rn(y5, a, b);
            y6 = __fma_rn(y6, a, b);
            y7 = __fma_rn(y7, a, b);
        }
    }
    double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7)) + ((y0 + y1) + (y2 + y3)) +
               ((y4 + y5) + (y6 + y7));
    if (s == 12345.678)
        sink[0] = s;
}

__device__ __forceinline__ void cv_dmma_m8n8k4(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) cv_peak_probe_dmma(int iters, double *sink)
{
    double a = 1e-3 * (threadIdx.x & 7), b = 1e-3 * (threadIdx.x & 3);
    double c[16];
#pragma unroll
    for (int i = 0; i < 16; i++)
        c[i] = 0.0;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++)
            cv_dmma_m8n8k4(c[2 * u], c[2 * u + 1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; i++)
        s += c[i];
    if (s == 12345.678)
        sink[0] = s;
}

/* Even warps run the DMMA chain, odd warps the DFMA chain: do the two share execution units? */
__global__ void __launch_bounds__(256) cv_peak_probe_mixed(int iters, double *sink)
{
    double s = 0.0;
    if ((threadIdx.x >> 5) & 1) {
        double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-9 * blockIdx.x;
        double x[16];
#pragma unroll
        for (int i = 0; i < 16; i++)
            x[i] = 0.1 + 0.05 * i;
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int u = 0; u < 8; u++)
#pragma unroll
                for (int j = 0; j < 16; j++)
                    x[j] = __fma_rn(x[j], a, b);
        }
#pragma unroll
        for (int i = 0; i < 16; i++)
            s += x[i];
    } else {
        double a = 1e-3 * (threadIdx.x & 7), b = 1e-3 * (threadIdx.x & 3);
        double c[16];
#pragma unroll
        for (int i = 0; i < 16; i++)
            c[i] = 0.0;
        for (int i = 0; i < iters; i++) {
#pragma unroll
            for (int u = 0; u < 8; u++)
                cv_dmma_m8n8k4(c[2 * u], c[2 * u + 1], a, b);
        }
#pragma unroll
        for (int i = 0; i < 16; i++)
            s += c[i];
    }
    if (s == 12345.678)
        sink[0] = s;
}

cudaError_t cv_launch_peak_probe(int kind, int n_cta, int iters, double *sink, double *flop,
                                 cudaStream_t stream)
{
    if (kind == 0) {
        cv_peak_probe_dfma<<<n_cta, 256, 0, stream>>>(iters, sink);
        *flop = 2.0 * 16.0 * 8.0 * (double)iters * 256.0 * (double)n_cta;
    } else if (kind == 1) {
        cv_peak_probe_dmma<<<n_cta, 256, 0, stream>>>(iters, sink);
        /* one m8n8k4 = 8*8*4 FMA per warp */
        *flop = 2.0 * 256.0 * 8.0 * (double)iters * 8.0 * (double)n_cta;
    } else {
        /* four DFMA warps (16 x 8 FMA per thread and iteration) + four DMMA warps (8 MMAs) */
        cv_peak_probe_mixed<<<n_cta, 256, 0, stream>>>(iters, sink);
        *flop = (2.0 * 16.0 * 8.0 * 128.0 + 2.0 * 256.0 * 8.0 * 4.0) * (double)iters * (double)n_cta;
    }
    return cudaGetLastError();
}
