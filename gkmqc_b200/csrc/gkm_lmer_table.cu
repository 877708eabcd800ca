/* gkm_lmer_table.cu -- sm_100a kernels of the L-mer table (the arithmetic: gkm_lmer_table.h; DESIGN.md 4.5).
 *
 * Build (once per model, on every GPU of the problem):
 *   gkm_idx_sort_keys       every L-mer of both strands of the SV columns -> key, radix-sorted by code (the index build's
 *                           own first steps, gkm_index.cu)
 *   gkm_lt_beta_kernel      beta_c = alpha_c / |c|
 *   gkm_lt_s_kernel         one thread per run of equal codes: S[code] = the run's sum of beta_c * wt
 *   gkm_lt_transform_kernel one launch per base t, one thread per group of four codes that differ only in base t
 *   gkm_lt_combine_kernel   T[u] = sum_m w[m] A_m[u]
 * Use:
 *   gkm_lt_export_kernel    T in lexicographic L-mer order
 *   gkm_lt_score_kernel     one thread per row: its forward L-mers, read from the packed planes like the index row kernel
 *                           builds its query, looked up in T
 *   gkm_lt_subst_kernel     single-base substitutions (gkm_lmer_subst.h, DESIGN.md 4.6): one CTA per block of consecutive
 *                           sites, one warp per site
 */
#include <cuda_runtime.h>

#include "gkm_index_dev.h"
#include "gkm_internal.h"
#include "gkm_lmer_table.h"
#include "gkm_lmer_table_dev.h"
#include "gkm_lmer_subst.h"

__global__ void __launch_bounds__(256)
gkm_lt_beta_kernel(const double *__restrict__ alpha, const double *__restrict__ norm, int ncols, double *__restrict__ beta)
{
    const int c = (int) (blockIdx.x * blockDim.x + threadIdx.x);
    if (c < ncols) beta[c] = gkm_lt_beta(alpha[c], norm[c]);
}

/* the head of every run of equal codes sums the run; long runs (homopolymers) cost that one thread a serial loop */
__global__ void __launch_bounds__(256)
gkm_lt_s_kernel(const unsigned long long *__restrict__ keys, uint32_t P, const double *__restrict__ beta, double *__restrict__ S)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const uint32_t code = (uint32_t) (keys[i] >> 32);
    if (i > 0 && (uint32_t) (keys[i - 1] >> 32) == code) return;
    double s = 0.0;
    for (uint32_t j = i; j < P; j++) {
        const unsigned long long k = keys[j];
        if ((uint32_t) (k >> 32) != code) break;
        s = gkm_lt_s_add(s, beta[(uint32_t) (k >> 8) & 0xFFFFFFu], (uint32_t) k & 0xFFu);
    }
    S[code] = s;
}

/* consecutive threads take consecutive groups: for t > 0 their codes are consecutive too, for t = 0 each thread reads
 * four consecutive doubles; either way a warp reads whole sectors */
__global__ void __launch_bounds__(256)
gkm_lt_transform_kernel(double *__restrict__ A, uint32_t ngroups, int L, int d, int t)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngroups) return;
    uint32_t b[4];
    gkm_lt_group(g, t, L, b);
    gkm_lt_step(A, (size_t) ngroups * 4, d, b);
}

struct gkm_lt_w { double w[GKM_MAX_L + 1]; };

__global__ void __launch_bounds__(256)
gkm_lt_combine_kernel(const double *__restrict__ A, uint32_t n, int d, const __grid_constant__ gkm_lt_w w, double *__restrict__ T)
{
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u < n) T[u] = gkm_lt_combine(A, n, d, w.w, u);
}

__global__ void __launch_bounds__(256)
gkm_lt_export_kernel(const double *__restrict__ T, uint32_t n, int L, double *__restrict__ out)
{
    const uint32_t lex = blockIdx.x * blockDim.x + threadIdx.x;
    if (lex < n) out[lex] = T[gkm_lt_lex_code(lex, L)];
}

template <bool WEIGHTED>
__global__ void __launch_bounds__(128)
gkm_lt_score_kernel(const double *__restrict__ T, const uint32_t *__restrict__ planes, const int32_t *__restrict__ lens,
                    const uint8_t *__restrict__ wend, int W, int L, const double *__restrict__ norm, int row0, int nrows,
                    double *__restrict__ out)
{
    const int r = (int) (blockIdx.x * blockDim.x + threadIdx.x);
    if (r >= nrows) return;
    const int a = row0 + r, nq = lens[a] - L + 1;
    const uint32_t *pl = planes + (size_t) a * 3 * (size_t) W;
    const uint8_t *we = WEIGHTED ? wend + (size_t) a * 32 * (size_t) W + (size_t) (L - 1) : nullptr;
    const uint32_t mask = (1u << L) - 1u;
    double s = 0.0;
#pragma unroll 4
    for (int i = 0; i < nq; i++) {
        const uint32_t x = gkm_idx_code(idx_window(pl, W, i, mask), idx_window(pl + W, W, i, mask), L);
        s = gkm_lt_row_add(s, WEIGHTED ? (uint32_t) we[i] : 1u, __ldg(T + x));
    }
    out[r] = gkm_lt_row_end(s, norm[a]);
}

/* Sites [s0, s0 + GKM_LS_SITES) of the launch go to one CTA, which walks them in runs of equal rows.  Per run it stages the
 * row: the plane windows and weights of both strands, T[code] of the forward windows and the prefix sums of the score
 * (thread 0, in gkm_lt_score_kernel's order).  Then each warp takes a site: lanes stride over the partner windows and
 * count into the warp's GKM_LS_ACC shared counters, and lane v < 4 finishes base v.  Repeated rows in one block are staged
 * once; a site list in row order (an ISM) stages each row once per block. */
#define GKM_LS_THREADS 128
#define GKM_LS_SITES 64

struct gkm_ls_add {
    __device__ __forceinline__ void operator()(uint32_t *a, uint32_t v) const { atomicAdd(a, v); }
};

/* dynamic shared memory: X0, X1 [2 nmax] words, PRE [nmax + 1], TX [nmax] doubles, WT [2 nmax] bytes */
static unsigned gkm_ls_smem(int nmax) { return (unsigned) (16 * nmax + 8 * (nmax + 1) + 8 * nmax + 2 * nmax + 16); }

template <bool WEIGHTED>
__global__ void __launch_bounds__(GKM_LS_THREADS)
gkm_lt_subst_kernel(const double *__restrict__ T, const uint32_t *__restrict__ planes, const int32_t *__restrict__ lens,
                    const uint8_t *__restrict__ wend, int W, int L, int d, const __grid_constant__ gkm_lt_w w,
                    const int32_t *__restrict__ H, int hrow0, int nmax, const int *__restrict__ row,
                    const int *__restrict__ pos, long long nsites, double *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t *X0 = reinterpret_cast<uint32_t *>(smem), *X1 = X0 + 2 * nmax;
    double *PRE = reinterpret_cast<double *>(X1 + 2 * nmax), *TX = PRE + nmax + 1;
    uint8_t *WT = reinterpret_cast<uint8_t *>(TX + nmax);
    __shared__ uint32_t sAcc[GKM_LS_THREADS / 32][GKM_LS_ACC];
    const int tid = (int) threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t mask = (1u << L) - 1u;
    const long long s0 = (long long) blockIdx.x * GKM_LS_SITES;
    const long long s1 = s0 + GKM_LS_SITES < nsites ? s0 + GKM_LS_SITES : nsites;
    uint32_t *acc = sAcc[warp];
    for (long long i = s0; i < s1;) {
        const int r = row[i];
        long long j = i + 1;
        while (j < s1 && row[j] == r) j++;
        const int len = lens[r], n = len - L + 1;
        const uint32_t *pl = planes + (size_t) r * 3 * (size_t) W;
        for (int k = tid; k < 2 * n; k += GKM_LS_THREADS) {
            const int lo = k < n ? k : len + k - n;
            const uint32_t x0 = idx_window(pl, W, lo, mask), x1 = idx_window(pl + W, W, lo, mask);
            X0[k] = x0; X1[k] = x1;
            WT[k] = WEIGHTED ? wend[(size_t) r * 32 * (size_t) W + (size_t) (lo + L - 1)] : (uint8_t) 1;
            if (k < n) TX[k] = __ldg(T + gkm_idx_code(x0, x1, L));
        }
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
            PRE[0] = s;
            for (int k = 0; k < n; k++) { s = gkm_lt_row_add(s, WT[k], TX[k]); PRE[k + 1] = s; }
        }
        __syncthreads();
        const int32_t *Hr = H + (size_t) (r - hrow0) * (size_t) (d + 1);
        for (long long site = i + warp; site < j; site += GKM_LS_THREADS / 32) {
            const int p = pos[site];
            int flo, fhi, rlo, rhi;
            gkm_ls_changed(p, len, L, &flo, &fhi, &rlo, &rhi);
            for (int k = lane; k < GKM_LS_ACC; k += 32) acc[k] = 0u;
            __syncwarp();
            gkm_ls_site_a(lane, 32, X0, X1, WT, n, p, flo, fhi, rlo, rhi, d, gkm_ls_add(), acc);
            gkm_ls_site_b(lane, 32, X0, X1, WT, n, len, p, flo, fhi, rlo, rhi, d, gkm_ls_add(), acc);
            __syncwarp();
            if (lane < 4) {
                const double norm = gkm_ls_norm(Hr, acc, (uint32_t) lane, d, w.w);
                const double num = gkm_ls_num(T, PRE, TX, X0, X1, WT, n, L, p, flo, fhi, (uint32_t) lane);
                out[(size_t) site * 4 + (size_t) lane] = gkm_lt_row_end(num, norm);
            }
            __syncwarp();
        }
        __syncthreads();
        i = j;
    }
}

static unsigned blocks_of(size_t n, unsigned threads) { return (unsigned) ((n + threads - 1) / threads); }

int gkm_lt_build(const gkm_lt_build_args *a, cudaStream_t st, cudaEvent_t *ev)
{
    const int L = a->keys.L, d = a->d;
    const size_t n = (size_t) 1 << (2 * L);
    cudaError_t e;
    if ((e = cudaMemsetAsync(a->A, 0, (size_t) (d + 1) * n * sizeof(double), st)) != cudaSuccess) goto fail;
    if (ev && (e = cudaEventRecord(ev[0], st)) != cudaSuccess) goto fail;
    if (a->keys.P > 0) {
        const unsigned long long *sorted;
        if ((e = gkm_idx_sort_keys(&a->keys, st, &sorted)) != cudaSuccess) goto fail;
        const int nc = a->keys.ce - a->keys.cb;
        gkm_lt_beta_kernel<<<blocks_of((size_t) nc, 256), 256, 0, st>>>(a->alpha, a->norm, nc, a->beta);
        gkm_lt_s_kernel<<<blocks_of(a->keys.P, 256), 256, 0, st>>>(sorted, (uint32_t) a->keys.P, a->beta, a->A);
    }
    if (ev && (e = cudaEventRecord(ev[1], st)) != cudaSuccess) goto fail;
    for (int t = 0; t < L; t++) gkm_lt_transform_kernel<<<blocks_of(n / 4, 256), 256, 0, st>>>(a->A, (uint32_t) (n / 4), L, d, t);
    if (ev && (e = cudaEventRecord(ev[2], st)) != cudaSuccess) goto fail;
    {
        gkm_lt_w w;
        for (int m = 0; m <= GKM_MAX_L; m++) w.w[m] = m <= d ? a->w[m] : 0.0;
        gkm_lt_combine_kernel<<<blocks_of(n, 256), 256, 0, st>>>(a->A, (uint32_t) n, d, w, a->T);
    }
    if (ev && (e = cudaEventRecord(ev[3], st)) != cudaSuccess) goto fail;
    if ((e = cudaGetLastError()) != cudaSuccess) goto fail;
    return 0;
fail:
    gkm_set_error("CUDA: L-mer table build: %s", cudaGetErrorString(e));
    return 1;
}

int gkm_lt_export(const double *T, int L, double *out, cudaStream_t st)
{
    const size_t n = (size_t) 1 << (2 * L);
    gkm_lt_export_kernel<<<blocks_of(n, 256), 256, 0, st>>>(T, (uint32_t) n, L, out);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table export: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}

int gkm_lt_score(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L,
                 const double *norm, int row0, int nrows, double *out, cudaStream_t st)
{
    if (wend) gkm_lt_score_kernel<true><<<blocks_of((size_t) nrows, 128), 128, 0, st>>>(T, planes, lens, wend, W, L, norm, row0, nrows, out);
    else gkm_lt_score_kernel<false><<<blocks_of((size_t) nrows, 128), 128, 0, st>>>(T, planes, lens, wend, W, L, norm, row0, nrows, out);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table scores: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}

int gkm_lt_subst(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L, int d,
                 const double *w, const int32_t *H, int hrow0, int maxlen, const int *row, const int *pos, long long nsites,
                 double *out, cudaStream_t st)
{
    if (nsites <= 0) return 0;
    gkm_lt_w wc;
    for (int m = 0; m <= GKM_MAX_L; m++) wc.w[m] = m <= d ? w[m] : 0.0;
    const int nmax = maxlen - L + 1;
    const unsigned smem = gkm_ls_smem(nmax);
    const void *fn = wend ? (const void *) gkm_lt_subst_kernel<true> : (const void *) gkm_lt_subst_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned) ((nsites + GKM_LS_SITES - 1) / GKM_LS_SITES);
        if (wend) gkm_lt_subst_kernel<true><<<grid, GKM_LS_THREADS, smem, st>>>(T, planes, lens, wend, W, L, d, wc, H, hrow0, nmax, row, pos, nsites, out);
        else gkm_lt_subst_kernel<false><<<grid, GKM_LS_THREADS, smem, st>>>(T, planes, lens, wend, W, L, d, wc, H, hrow0, nmax, row, pos, nsites, out);
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table substitutions: %s", cudaGetErrorString(e)); return 1; }
    return 0;
}
