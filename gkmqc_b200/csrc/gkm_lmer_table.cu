/* gkm_lmer_table.cu -- the L-mer table (the arithmetic: gkm_lmer_table.h; DESIGN.md 4.5): its sm_100a kernels and the
 * entry points of the ABI that build, export and score through it.
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
#include "gkm_dev.h"
#include "gkm_lmer_table.h"
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

/* On stream st, from the sorted keys of the SV columns [cb, ce) and their alpha and norm |c| (device, [ce - cb]): beta (device,
 * [ce - cb]), S and its transform in A (device, [d + 1][4^L]), and the combine with w[0..d] (host) into T (device, [4^L]).
 * ev = NULL or four events recorded before S, between the phases and behind the combine.  The functions that launch
 * return the first CUDA error; their callers word it. */
static cudaError_t gkm_lt_build(const gkm_idx_build_args *keys, int d, const double *alpha, const double *norm, double *beta, double *A,
                                double *T, const double *w, cudaStream_t st, cudaEvent_t *ev)
{
    const int L = keys->L;
    const size_t n = (size_t) 1 << (2 * L);
    cudaError_t e;
    if ((e = cudaMemsetAsync(A, 0, (size_t) (d + 1) * n * sizeof(double), st)) != cudaSuccess) return e;
    if (ev && (e = cudaEventRecord(ev[0], st)) != cudaSuccess) return e;
    if (keys->P > 0) {
        const unsigned long long *sorted;
        if ((e = gkm_idx_sort_keys(keys, st, &sorted)) != cudaSuccess) return e;
        const int nc = keys->ce - keys->cb;
        gkm_lt_beta_kernel<<<blocks_of((size_t) nc, 256), 256, 0, st>>>(alpha, norm, nc, beta);
        gkm_lt_s_kernel<<<blocks_of(keys->P, 256), 256, 0, st>>>(sorted, (uint32_t) keys->P, beta, A);
    }
    if (ev && (e = cudaEventRecord(ev[1], st)) != cudaSuccess) return e;
    for (int t = 0; t < L; t++) gkm_lt_transform_kernel<<<blocks_of(n / 4, 256), 256, 0, st>>>(A, (uint32_t) (n / 4), L, d, t);
    if (ev && (e = cudaEventRecord(ev[2], st)) != cudaSuccess) return e;
    {
        gkm_lt_w wc;
        for (int m = 0; m <= GKM_MAX_L; m++) wc.w[m] = m <= d ? w[m] : 0.0;
        gkm_lt_combine_kernel<<<blocks_of(n, 256), 256, 0, st>>>(A, (uint32_t) n, d, wc, T);
    }
    if (ev && (e = cudaEventRecord(ev[3], st)) != cudaSuccess) return e;
    return cudaGetLastError();
}

/* out[lex] = T[code of lex], 4^L values (device buffers) */
static cudaError_t gkm_lt_export(const double *T, int L, double *out, cudaStream_t st)
{
    const size_t n = (size_t) 1 << (2 * L);
    gkm_lt_export_kernel<<<blocks_of(n, 256), 256, 0, st>>>(T, (uint32_t) n, L, out);
    return cudaGetLastError();
}

/* out[r] = (sum over the forward L-mers of row row0 + r of wt * T[code]) / norm[row0 + r], r < nrows; wend = NULL: unit weights */
static cudaError_t gkm_lt_score(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L,
                                const double *norm, int row0, int nrows, double *out, cudaStream_t st)
{
    const auto kernel = wend ? gkm_lt_score_kernel<true> : gkm_lt_score_kernel<false>;
    kernel<<<blocks_of((size_t) nrows, 128), 128, 0, st>>>(T, planes, lens, wend, W, L, norm, row0, nrows, out);
    return cudaGetLastError();
}

/* out[4 i + v] = (numerator of the row row[i] with base pos[i] replaced by v) / its norm, i < nsites (gkm_lmer_subst.h):
 * H = the rows' self histograms, [rows][d + 1] int32 from row hrow0; w[0..d] host; maxlen = the longest row of the
 * problem; row, pos, out device buffers.  Sites of one row are best consecutive: each block of 64 stages a row once per run. */
static cudaError_t gkm_lt_subst(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L, int d,
                                const double *w, const int32_t *H, int hrow0, int maxlen, const int *row, const int *pos, long long nsites,
                                double *out, cudaStream_t st)
{
    gkm_lt_w wc;
    for (int m = 0; m <= GKM_MAX_L; m++) wc.w[m] = m <= d ? w[m] : 0.0;
    const int nmax = maxlen - L + 1;
    const unsigned smem = gkm_ls_smem(nmax);
    const auto kernel = wend ? gkm_lt_subst_kernel<true> : gkm_lt_subst_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute((const void *) kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned) ((nsites + GKM_LS_SITES - 1) / GKM_LS_SITES);
        kernel<<<grid, GKM_LS_THREADS, smem, st>>>(T, planes, lens, wend, W, L, d, wc, H, hrow0, nmax, row, pos, nsites, out);
        e = cudaGetLastError();
    }
    return e;
}

/* ---- entry points of the ABI ---- */
/* the folded model: one copy of T on every GPU of the problem it was built from */
struct gkmb200_lmer_table {
    gkm_parameter param;       /* of that problem: scoring needs the same (type, L, k, d, M, H) */
    int ndev;
    int dev[GKM_MAX_DEV];      /* the problem's GPUs, in its slot order */
    double *T[GKM_MAX_DEV];    /* 4^L doubles per GPU, in code order (gkm_idx_code) */
    double build_ms[3];        /* device time of S, the transform and the combine on the first GPU (CUDA events) */
};

/* one GPU's copy: sorted keys of the columns -> S -> transform -> T.  Everything but T is freed before returning. */
static int lmer_table_slice(gkmb200_lmer_table *t, gkmb200_problem *p, int slot, int col0, int ncols, const double *alpha)
{
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[slot]];
    const gkm_image *im = &ds->img[slot];
    const int L = p->param.L, d = p->param.d;
    const size_t n = (size_t) 1 << (2 * L);
    gkm_idx_build_args a;
    memset(&a, 0, sizeof(a));
    uint32_t *offs = NULL;
    size_t sbytes = 0;
    const int kr = column_keys_prepare(p, im, col0, col0 + ncols, &a, &offs, &sbytes);
    if (kr == 2) gkm_set_error("L-mer table: %zu postings, more than the key sort takes", a.P);
    if (kr) return 1;
    gkm_dbuf<char> scratch(g);
    gkm_dbuf<uint32_t> d_offs(g);
    gkm_dbuf<double> d_alpha(g), beta(g), A(g), T(g);
    cudaEvent_t ev[4] = { NULL, NULL, NULL, NULL };
    int rc = 0;
    cudaError_t e = scratch.alloc(sbytes);
    if (e == cudaSuccess) e = d_offs.alloc((size_t) ncols);
    if (e == cudaSuccess) e = d_alpha.alloc((size_t) ncols);
    if (e == cudaSuccess) e = beta.alloc((size_t) ncols);
    if (e == cudaSuccess) e = A.alloc((size_t) (d + 1) * n);
    if (e == cudaSuccess) e = T.alloc(n);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_offs, offs, (size_t) ncols * 4, cudaMemcpyHostToDevice, g->sc);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_alpha, alpha, (size_t) ncols * sizeof(double), cudaMemcpyHostToDevice, g->sc);
    for (int i = 0; i < 4 && e == cudaSuccess && slot == 0; i++) e = cudaEventCreate(&ev[i]);
    if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table buffers (%zu bytes of planes): %s", (size_t) (d + 2) * n * sizeof(double), cudaGetErrorString(e)); rc = 1; }
    if (!rc) {
        a.offs = d_offs; a.scratch = scratch;
        e = gkm_lt_build(&a, d, d_alpha, im->sqnorm + col0, beta, A, T, p->w, g->sc, slot == 0 ? ev : NULL);
        if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table build: %s", cudaGetErrorString(e)); rc = 1; }
    }
    /* pageable sources: wait for the build before letting go of them */
    e = cudaStreamSynchronize(g->sc);
    if (e != cudaSuccess && !rc) { gkm_set_error("CUDA: L-mer table build failed: %s", cudaGetErrorString(e)); rc = 1; }
    if (!rc && slot == 0) {
        for (int i = 0; i < 3; i++) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
            t->build_ms[i] = ms;
        }
    }
    for (int i = 0; i < 4; i++) if (ev[i]) cudaEventDestroy(ev[i]);
    free(offs);
    if (!rc) t->T[slot] = T.release();
    return rc;
}

static void lmer_table_release(gkmb200_lmer_table *t)
{
    for (int i = 0; i < t->ndev; i++) {
        if (!t->T[i]) continue;
        if (cudaSetDevice(t->dev[i]) == cudaSuccess) cudaFree(t->T[i]);
        else cudaGetLastError();
        t->T[i] = NULL;
    }
}

extern "C" gkmb200_lmer_table *gkmb200_lmer_table_new(gkmb200_problem *p, int col0, int ncols, const double *alpha)
{
    if (!p || !alpha) { gkm_set_error("null argument"); return NULL; }
    const gkm_parameter *pa = &p->param;
    if (pa->kernel_type == 3 || pa->kernel_type == 5) {
        gkm_set_error("kernel type %d is an RBF kernel, not linear in the gkm features: it has no L-mer table", pa->kernel_type);
        return NULL;
    }
    if (col0 < 0 || ncols < 1 || col0 > p->n - ncols) { gkm_set_error("columns [%d,+%d) outside the problem (n=%d)", col0, ncols, p->n); return NULL; }
    if (ncols > GKM_LT_MAX_COLS) { gkm_set_error("L-mer table of %d columns: at most %d", ncols, GKM_LT_MAX_COLS); return NULL; }
    if (gkm_lt_bytes(pa->L, pa->d) > GKM_LT_MAX_BYTES) {
        gkm_set_error("L-mer table at L=%d d=%d needs %llu bytes per GPU, more than %llu", pa->L, pa->d, gkm_lt_bytes(pa->L, pa->d), GKM_LT_MAX_BYTES);
        return NULL;
    }
    gkmb200_lmer_table *t = (gkmb200_lmer_table *) calloc(1, sizeof(*t));
    if (!t) { gkm_set_error("out of memory"); return NULL; }
    t->param = *pa;
    pthread_mutex_lock(&g_lock);
    int rc = upload_locked(p, 0);
    if (!rc) {
        t->ndev = p->dev->ndev;
        for (int i = 0; i < t->ndev; i++) t->dev[i] = p->dev->dev[i];
        rc = for_each_gpu(p->dev, [&](int slot) { return lmer_table_slice(t, p, slot, col0, ncols, alpha); });
    }
    if (rc) lmer_table_release(t);
    pthread_mutex_unlock(&g_lock);
    if (rc) { free(t); return NULL; }
    return t;
}

extern "C" void gkmb200_lmer_table_free(gkmb200_lmer_table *t)
{
    if (!t) return;
    pthread_mutex_lock(&g_lock);
    lmer_table_release(t);
    pthread_mutex_unlock(&g_lock);
    free(t);
}

extern "C" int gkmb200_lmer_table_build_ms(const gkmb200_lmer_table *t, double *out)
{
    if (!t || !out) { gkm_set_error("null argument"); return 1; }
    memcpy(out, t->build_ms, sizeof(t->build_ms));
    return 0;
}

extern "C" int gkmb200_lmer_table_get(gkmb200_lmer_table *t, double *out)
{
    if (!t || !out) { gkm_set_error("null argument"); return 1; }
    const size_t n = (size_t) 1 << (2 * t->param.L);
    pthread_mutex_lock(&g_lock);
    int rc = 0;
    {
        gkm_gpu *g = &g_gpu[t->dev[0]];
        gkm_dbuf<double> d_out(g);
        cudaError_t e = cudaSetDevice(t->dev[0]);
        if (e == cudaSuccess) e = d_out.alloc(n);
        if (e == cudaSuccess) e = gkm_lt_export(t->T[0], t->param.L, d_out, g->sc);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, g->sc);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc);
        if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table export: %s", cudaGetErrorString(e)); rc = 1; }
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* one GPU's slice of the rows of q */
static int lmer_scores_slice(const gkmb200_lmer_table *t, gkmb200_problem *q, int slot, int row0, int nrows, double bias, double *out)
{
    if (nrows <= 0) return 0;
    gkm_gpu *g = &g_gpu[q->dev->dev[slot]];
    const gkm_image *im = &q->dev->img[slot];
    gkm_dbuf<double> d_out(g);
    cudaError_t e = d_out.alloc((size_t) nrows);
    if (e == cudaSuccess) e = gkm_lt_score(t->T[slot], im->planes, im->lens, q->weighted ? im->wend : NULL, q->Wmax, q->param.L, im->sqnorm, row0, nrows, d_out, g->sc);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, (size_t) nrows * sizeof(double), cudaMemcpyDeviceToHost, g->sc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc);
    if (e != cudaSuccess) { gkm_set_error("CUDA: L-mer table scores: %s", cudaGetErrorString(e)); return 1; }
    __atomic_fetch_add(&q->stats.launches, 1, __ATOMIC_RELAXED);
    for (int i = 0; i < nrows; i++) out[i] += bias; /* as decision_slice adds it */
    return 0;
}

/* the checks of every use of a table on a problem q: the same (type, L, k, d, M, H) before anything is done ... */
static int lmer_table_params_match(const gkmb200_lmer_table *t, const gkmb200_problem *q)
{
    const gkm_parameter *a = &t->param, *b = &q->param;
    if (a->kernel_type != b->kernel_type || a->L != b->L || a->k != b->k || a->d != b->d || a->M != b->M || a->H != b->H) {
        gkm_set_error("problem (type %d, L=%d, k=%d, d=%d, M=%d, H=%g) does not match the L-mer table (type %d, L=%d, k=%d, d=%d, M=%d, H=%g)",
                      b->kernel_type, b->L, b->k, b->d, b->M, b->H, a->kernel_type, a->L, a->k, a->d, a->M, a->H);
        return 0;
    }
    return 1;
}

/* ... and, under g_lock, q uploaded to the table's GPUs in the table's slot order */
static int lmer_table_upload(const gkmb200_lmer_table *t, gkmb200_problem *q)
{
    if (upload_locked(q, 0)) return 1;
    int same = q->dev->ndev == t->ndev;
    for (int i = 0; same && i < t->ndev; i++) same = q->dev->dev[i] == t->dev[i];
    if (!same) { gkm_set_error("the problem lives on other GPUs than the L-mer table (%d against %d)", q->dev->ndev, t->ndev); return 1; }
    return 0;
}

extern "C" int gkmb200_lmer_table_scores(gkmb200_lmer_table *t, gkmb200_problem *q, int row0, int nrows, double bias, double *out)
{
    if (!t || !q || !out) { gkm_set_error("null argument"); return 1; }
    if (!lmer_table_params_match(t, q)) return 1;
    if (row0 < 0 || nrows < 0 || row0 > q->n - nrows) { gkm_set_error("rows [%d,+%d) outside the problem (n=%d)", row0, nrows, q->n); return 1; }
    if (nrows == 0) return 0;
    pthread_mutex_lock(&g_lock);
    q->stats.launches = 0;
    int rc = lmer_table_upload(t, q);
    if (!rc) rc = for_each_gpu_share(q->dev, nrows, 8, [&](int slot, long long b, long long e) {
        return lmer_scores_slice(t, q, slot, row0 + (int) b, (int) (e - b), bias, out + b);
    });
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* sites per launch of the substitution kernel: 16 MB of sites and 64 MB of results on the device, whatever nsites is */
#define GKM_LS_CHUNK ((long long) 1 << 21)

/* one GPU's slice of the sites, in chunks of GKM_LS_CHUNK */
static int lmer_subst_slice(const gkmb200_lmer_table *t, gkmb200_problem *q, int slot, long long nsites, const int *row, const int *pos,
                            double bias, double *out)
{
    if (nsites <= 0) return 0;
    gkm_gpu *g = &g_gpu[q->dev->dev[slot]];
    const gkm_image *im = &q->dev->img[slot];
    const long long cap = nsites < GKM_LS_CHUNK ? nsites : GKM_LS_CHUNK;
    gkm_dbuf<int> d_row(g), d_pos(g);
    gkm_dbuf<int32_t> d_H(g);
    gkm_dbuf<double> d_out(g);
    size_t hcap = 0;
    int rc = 0;
    cudaError_t e = d_row.alloc((size_t) cap);
    if (e == cudaSuccess) e = d_pos.alloc((size_t) cap);
    if (e == cudaSuccess) e = d_out.alloc((size_t) cap * 4);
    for (long long c0 = 0; e == cudaSuccess && !rc && c0 < nsites; c0 += cap) {
        const long long nc = nsites - c0 < cap ? nsites - c0 : cap;
        int rmin = row[c0], rmax = row[c0];
        for (long long i = c0; i < c0 + nc; i++) { rmin = row[i] < rmin ? row[i] : rmin; rmax = row[i] > rmax ? row[i] : rmax; }
        const size_t hbytes = (size_t) (rmax - rmin + 1) * (size_t) q->nbins * sizeof(int32_t);
        if (hbytes > hcap) {
            if ((e = cudaStreamSynchronize(g->sc)) != cudaSuccess) break;
            if ((e = d_H.alloc(hbytes / sizeof(int32_t))) != cudaSuccess) break;
            hcap = hbytes;
        }
        if ((e = cudaMemcpyAsync(d_row, row + c0, (size_t) nc * sizeof(int), cudaMemcpyHostToDevice, g->sc)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(d_pos, pos + c0, (size_t) nc * sizeof(int), cudaMemcpyHostToDevice, g->sc)) != cudaSuccess) break;
        /* H(r, r) of the rows [rmin, rmax]: the upload's diagonal launch, with histograms kept (the diagonal: entry (r, r)
         * lands at row r - row_base) */
        gkm_kparams kp;
        fill_kparams(q, im, GKM_MODE_DIAG, &kp);
        kp.hist = d_H;
        const int diag = launch_diag_rows(q, im, g, rmin, rmax + 1, kp);
        if (diag < 0) { rc = 1; break; }
        __atomic_fetch_add(&q->stats.launches, diag + 1, __ATOMIC_RELAXED);
        e = gkm_lt_subst(t->T[slot], im->planes, im->lens, q->weighted ? im->wend : NULL, q->Wmax, q->param.L, q->param.d, q->w,
                         d_H, rmin, q->maxlen, d_row, d_pos, nc, d_out, g->sc);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out + 4 * c0, d_out, (size_t) nc * 4 * sizeof(double), cudaMemcpyDeviceToHost, g->sc);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc);
    }
    if (e != cudaSuccess && !rc) { gkm_set_error("CUDA: L-mer table substitutions: %s", cudaGetErrorString(e)); rc = 1; }
    cudaStreamSynchronize(g->sc); /* the pageable sources and the buffers stay until the stream has drained */
    if (!rc) for (long long i = 0; i < 4 * nsites; i++) out[i] += bias; /* as lmer_scores_slice adds it */
    return rc;
}

extern "C" int gkmb200_lmer_table_substitutions(gkmb200_lmer_table *t, gkmb200_problem *q, long long nsites, const int *row, const int *pos,
                                                double bias, double *out)
{
    if (!t || !q) { gkm_set_error("null argument"); return 1; }
    if (nsites < 0) { gkm_set_error("%lld sites", nsites); return 1; }
    if (nsites > 0 && (!row || !pos || !out)) { gkm_set_error("null argument"); return 1; }
    if (!lmer_table_params_match(t, q)) return 1;
    for (long long i = 0; i < nsites; i++) {
        if (row[i] < 0 || row[i] >= q->n) { gkm_set_error("site %lld: row %d outside the problem (n=%d)", i, row[i], q->n); return 1; }
        if (pos[i] < 0 || pos[i] >= q->len[row[i]]) {
            gkm_set_error("site %lld: position %d outside row %d (length %d)", i, pos[i], row[i], q->len[row[i]]);
            return 1;
        }
    }
    if (nsites == 0) return 0;
    pthread_mutex_lock(&g_lock);
    q->stats.launches = 0;
    int rc = lmer_table_upload(t, q);
    if (!rc) rc = for_each_gpu_share(q->dev, nsites, 1, [&](int slot, long long b, long long e) {
        return lmer_subst_slice(t, q, slot, e - b, row + b, pos + b, bias, out + 4 * b);
    });
    pthread_mutex_unlock(&g_lock);
    return rc;
}

