/* gkm_b200.h -- extended C-ABI of gkmkern_pylib.so (B200 / sm_100a gkm kernel engine).
 *
 * gkm_abi.h holds the entry points the reference exports (src/libgkm.h); this
 * header adds what a GPU engine needs that the reference's ABI cannot express:
 * in-memory sequences (SURVEY.md 8f/f2), the rectangular test x SV shape without
 * abusing one row per call (libgkm.c:1156), raw integer histograms for parity
 * checks (the reference keeps them private, libgkm.c:568-588), fused decision
 * values (8f/f1, what gkmsvm.py:109,118 does with the slice), tile sharding over
 * processes, device timing.  Plain pointers and sizes only.
 *
 * Every function returns 0 on success unless stated otherwise; on failure
 * gkmb200_last_error() describes why.  Compute entry points FAIL when no
 * sm_100 device is visible: there is no CPU fallback.
 */
#ifndef GKM_B200_H_INCLUDED
#define GKM_B200_H_INCLUDED

#include "gkm_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gkmb200_problem gkmb200_problem;

typedef struct gkmb200_stats {
    double kernel_ms;        /* device time of the histogram kernels of the last compute call (CUDA events) */
    double wall_ms;          /* host wall time of the last compute call */
    double upload_ms;        /* pack + H2D + sqnorm of the last upload */
    long long launches;      /* kernel launches of the last call on this problem, over all its GPUs: an upload, a compute
                              * call, decision values, or (on the scored problem) L-mer table scores and substitutions.
                              * An upload or index build the call made is included (pack 1, sqnorm 1 per diagonal step,
                              * index 5 per column block).  Decision values: one per row block of 8 192 rows (index: one per
                              * column block per 2 368 rows); scores: one per GPU share; substitutions: per batch of 2^21
                              * sites, the diagonal launches of its rows plus one */
    long long entries;       /* kernel entries produced by the last compute call */
    long long lmer_pairs;    /* L-mer pair comparisons those entries stand for */
    long long h2d_bytes;     /* bytes copied host->device by the last upload */
    long long d2h_bytes;     /* bytes copied device->host by the last compute call */
    int devices;             /* GPUs used */
    int kernel_variant;      /* 1 = lmer (XOR/LOP3/POPC per pair), 2 = diag (bit-sliced diagonals), 3 = mma (tcgen05), 4 = index */
    int shard_rank, shard_world; /* the call computed only the chunks of shard rank/world (1 = everything) */
    int copy_threads;        /* host threads that copied finished chunks into the caller's rows */
    int thp_chunks;          /* always 0: the transparent-huge-page hint on the destination rows is retired (no gain measured) */
    float scatter_ms;        /* host time spent in that copy (page faults of a fresh matrix included), slowest GPU thread */
    float wait_ms;           /* host time spent waiting for the GPU, slowest GPU thread */
} gkmb200_stats;

/* ---- process-wide ---- */
const char *gkmb200_last_error(void);
int gkmb200_abi_version(void);
int gkmb200_device_count(void);                      /* visible CUDA devices of compute capability 10.x; 0 if none */
int gkmb200_set_devices(const int *ids, int n);      /* default: env GKM_DEVICES ("0,1,.."), else all */
int gkmb200_set_option(const char *key, const char *value); /* "kernel" = auto|lmer|diag|mma|index ; "max_L" = 12|16 ; "chunk_mb", "index_cols", "index_split" = auto|equal|greedy, "index_wide" */
void gkmb200_set_verbosity(int level);               /* 0..4 like gkmOpt.verbosity */
int gkmb200_trim(void);                              /* give the cached device blocks of every GPU back to the driver */

/* ---- host-only arithmetic of the path (no GPU needed) ---- */
const char *gkmb200_check_parameter(const gkm_parameter *param); /* NULL if ok; the gate of gkmkern_pylib.c:38-64 */
int gkmb200_weights(int kernel_type, int L, int k, double *w);   /* w[0..L]; libgkm.c:107-217 */
int gkmb200_posweights(int nk, int kernel_type, int M, double H, uint8_t *wt, uint8_t *wt_rc); /* libgkm.c:910-932 */

/* ---- problem = parameter set + sequences (ids in insertion order) ---- */
gkmb200_problem *gkmb200_problem_new(const gkm_parameter *param);
void gkmb200_problem_free(gkmb200_problem *p);
int gkmb200_problem_add(gkmb200_problem *p, const char *seq, int len);       /* len < 0: strlen. returns the id or -1 */
int gkmb200_problem_add_block(gkmb200_problem *p, const char *bases, long stride, int n, int len); /* n sequences of len bases, stride bytes apart; returns the new size or -1 */
int gkmb200_problem_read_fasta(gkmb200_problem *p, const char *path);        /* records appended, or -1 (libgkm.c:1251) */
int gkmb200_problem_read(gkmb200_problem *p, const char *posfile, const char *negfile); /* n_pos, or -1 (libgkm.c:1316) */
int gkmb200_problem_size(const gkmb200_problem *p);
int gkmb200_problem_seqlen(const gkmb200_problem *p, int i);
const char *gkmb200_problem_sid(const gkmb200_problem *p, int i);            /* FASTA id (libgkm.c:1287-1292) or NULL */
int gkmb200_problem_codes(const gkmb200_problem *p, int i, uint8_t *fwd, uint8_t *rc);   /* 1..4 like gkm_data.seq */
int gkmb200_problem_get_weights(const gkmb200_problem *p, double *w);        /* d+1 values */
int gkmb200_problem_set_shard(gkmb200_problem *p, int rank, int world);      /* this process computes chunk c iff owner(c) == rank */

/* copy the base codes (one byte per base) to every selected GPU, pack them there into the 2-bit plane image
 * (SURVEY.md 8f/f2), compute sqnorm there (libgkm.c:723-759) */
int gkmb200_problem_upload(gkmb200_problem *p);
int gkmb200_problem_sqnorm(gkmb200_problem *p, double *out);                 /* n values */

/* ---- the kernel ---- */
/* triangular matrix into caller rows: rows[a][j] = K(a,j) for j<a, rows[a][a] = 1 (gkmkern_pylib.c:169-221).
 * copy_threads is a lower bound on the host threads that scatter finished chunks into the rows: the library uses
 * the cores of its affinity mask, divided by the ranks of a sharded run (env GKM_COPY_THREADS overrides;
 * gkm_device.cu:gkm_copy_threads_shared) */
int gkmb200_kernel_lower(gkmb200_problem *p, double **rows, int copy_threads);
/* dense block: out[(r-row0)*ld + (c-col0)] = K(r,c).  lower != 0: only c < r is written (and r == c gets 1.0).
 * With the SVs at ids [0,nSV) this is gkmkernel_kernelfunc_batch_all(a, 0, nSV) for a whole batch of rows. */
int gkmb200_kernel_block(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower, double *out, long ld);
/* raw truncated mismatch histograms: hist[((r-row0)*ncols + (c-col0))*(d+1) + m] = H_m(r,c), 32-bit */
int gkmb200_hist_block(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower, int32_t *hist);
/* out[r-row0] = bias + sum_c alpha[c-col0] * K(r,c), reduced on the device */
int gkmb200_decision_values(gkmb200_problem *p, int row0, int nrows, int col0, int ncols,
                            const double *alpha, double bias, double *out);

/* ---- the consumer of the matrix (SURVEY.md 8f/f4): cross-validated C-SVC on the precomputed kernel ---- */
/* One fit = one (train, test) split, like one call of _svm_train_proc in scripts/gkmsvm.py:104-122.
 * train_idx / test_idx hold sequence ids; the training ids of a fit must be grouped by class, label 0 (the
 * negatives) first -- the order libsvm gives them (svm_group_classes) -- and train_y must be +1 for that first
 * class and -1 for the other (libsvm's sub-problem labels); a fit whose training labels lack either is rejected.
 * gkmqc_b200/driver.py prepares both from 0/1 labels. */
typedef struct gkmb200_svm_task {
    long long train_off, test_off; /* first entry of this fit in train_idx / train_y and in test_idx / scores */
    int ntrain, ntest;
} gkmb200_svm_task;

typedef struct gkmb200_svm_fit {
    double rho;    /* libsvm's rho of the sub-problem (sklearn's intercept_ = +rho after its sign flip) */
    double obj;    /* dual objective value */
    double nu;     /* sum(alpha) / ntrain, what gkmsvm.py:120 logs */
    int n_iter;    /* SMO iterations */
    int n_sv;      /* support vectors */
    long long reserved;
} gkmb200_svm_fit;

/* Trains every fit with libsvm's SMO (C-SVC, second-order working-set selection, no shrinking; C, eps = SVC's C and
 * tol; max_iter < 0: libsvm's own ceiling) on the GPU, all fits concurrently, and evaluates their test points:
 * scores[test_off + r] = sklearn's decision_function value (positive = label 1).
 * kmat != NULL: dense symmetric n x n host matrix with ld doubles per row (what computeGkmKernel returns).
 * kmat == NULL: the kernel matrix of problem p is computed on the device and never leaves it (n = problem size).
 * fits[ntasks] and alpha[sum of ntrain] (in training order) may be NULL.
 * = gkmb200_svm_cv_ex with shrinking = 0. */
int gkmb200_svm_cv(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                   const int *train_idx, const signed char *train_y, const int *test_idx,
                   double C, double eps, int max_iter, double *scores, gkmb200_svm_fit *fits, double *alpha);

typedef struct gkmb200_svm_options {
    double C;          /* SVC's C */
    double eps;        /* SVC's tol */
    int max_iter;      /* SVC's max_iter; < 0: libsvm's own ceiling */
    int shrinking;     /* SVC's shrinking: 0 or 1 (anything else is rejected) */
    long long reserved;
} gkmb200_svm_options;

/* what the shrinking heuristic did in one fit (shrinking = 0: {0, ntrain, -1, 0, 0}) */
typedef struct gkmb200_svm_shrink_stats {
    int shrink_passes;   /* calls of libsvm's do_shrinking */
    int min_active;      /* smallest active set those passes left */
    int unshrink_iter;   /* iterations done when the whole gradient was rebuilt near the optimum (Gmax1 + Gmax2 <= 10 eps), or -1 */
    int recon_a;         /* gradient reconstructions looping over the inactive points outside, the free active ones inside */
    int recon_b;         /* gradient reconstructions looping over the free active points outside */
    int reserved;
} gkmb200_svm_shrink_stats;

/* gkmb200_svm_cv with the options of SVC: shrinking = 1 follows sklearn's SVC(shrinking=True) iterate for iterate
 * (libsvm's do_shrinking every min(ntrain, 1000) iterations, its unshrink and gradient reconstructions, the same
 * iteration count, support vectors, dual_coef_ and intercept_).  stats[ntasks] may be NULL. */
int gkmb200_svm_cv_ex(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                      const int *train_idx, const signed char *train_y, const int *test_idx, const gkmb200_svm_options *opt,
                      double *scores, gkmb200_svm_fit *fits, double *alpha, gkmb200_svm_shrink_stats *stats);

/* rows [row0, row0 + nrows) of the resident symmetric matrix of p (all n columns, unit diagonal; ld >= n doubles per row),
 * computed on first use and kept on the device for gkmb200_svm_cv; nrows = 0 only makes it resident.  With several
 * GPUs in one process every GPU writes its chunks straight into the first GPU's matrix (peer stores over NVLink). */
int gkmb200_resident_rows(gkmb200_problem *p, int row0, int nrows, double *out, long ld);

/* ---- the model folded into one weight per L-mer (kernel types 0, 1, 2, 4) ---- */
/* A model f(r) = bias + sum_c alpha[c] K(r, c) of a kernel type that is linear in the gkm features is a table of 4^L
 * weights T: f(r) = bias + (sum over the forward L-mers x of r of wt_r(x) T[x]) / |r|, whatever the number of SVs.
 * T[u] is also the model's weight of the L-mer u: the score of the sequence u (exactly L bases) is T[u] / |u| + bias.
 * The table needs (d + 2) 4^L doubles per GPU while it is built (A_0..A_d and T; 4^L stay); more than
 * GKM_LT_MAX_BYTES (16 GiB: L = 16 always, L = 15 above d = 0) is refused, as are the RBF types 3 and 5 and more than
 * 2^24 columns.  DESIGN.md 4.5. */
typedef struct gkmb200_lmer_table gkmb200_lmer_table;
/* the model sum_c alpha[c - col0] K(., c), c in [col0, col0 + ncols) of p, folded into T[4^L]; built on every GPU of p.
 * NULL on failure (gkmb200_last_error) */
gkmb200_lmer_table *gkmb200_lmer_table_new(gkmb200_problem *p, int col0, int ncols, const double *alpha);
void gkmb200_lmer_table_free(gkmb200_lmer_table *t);
/* out[4^L]: T in lexicographic L-mer order (A, C, G, T = 0..3, first base most significant) */
int gkmb200_lmer_table_get(gkmb200_lmer_table *t, double *out);
/* out[r - row0] = bias + sum_c alpha[c] K(r, c) for r in [row0, row0 + nrows) of q, evaluated through the table.  q may be
 * the problem of the table or another one with the same (type, L, k, d, M, H) on the same GPUs; its rows are cut into
 * one slice per GPU.  Equal to gkmb200_decision_values up to the rounding of two different summation orders. */
int gkmb200_lmer_table_scores(gkmb200_lmer_table *t, gkmb200_problem *q, int row0, int nrows, double bias, double *out);
/* Single-base substitutions (in-silico mutagenesis, variant effects): for the sites i < nsites, with 0 <= row[i] < n and
 * 0 <= pos[i] < len(row[i]), in any order and repeats allowed,
 *   out[4 i + v] = bias + the score of row[i] with base pos[i] replaced by v   (v = A, C, G, T = 0..3).
 * Each entry equals, bit for bit, gkmb200_lmer_table_scores of a problem holding that mutated sequence, its norm as the
 * upload computes it included (and the inf / NaN of a zero norm).  The entry of the row's own base (gkmb200_problem_codes:
 * an N counts as A) is the row's unmutated score.  The norm and the sum are updated, not recomputed: only the <= L windows
 * of each strand that cover the base change (DESIGN.md 4.6).  q as for gkmb200_lmer_table_scores; the sites are cut into
 * one slice per GPU.  Refused: null pointers (when nsites > 0), nsites < 0, a row outside q, a position outside its row,
 * mismatched parameters and other GPUs. */
int gkmb200_lmer_table_substitutions(gkmb200_lmer_table *t, gkmb200_problem *q, long long nsites, const int *row, const int *pos,
                                     double bias, double *out);
/* out[3] = device milliseconds of the table's build on its first GPU: S (keys, sort, run sums), transform, combine */
int gkmb200_lmer_table_build_ms(const gkmb200_lmer_table *t, double *out);

/* the packed image as it lies on GPU 0: planes[n][3][W] (code bit 0, code bit 1, window-end plane E; both strands in one
 * circular string) and, weighted kernel types only, wend[n][32 W]; either may be NULL; out_shape = {n, W} */
int gkmb200_problem_image(gkmb200_problem *p, uint32_t *planes, uint8_t *wend, int *out_shape);

/* ---- measurement ---- */
/* out[3] = {column blocks, columns per block, first column} of the index variant's last compute call on p (zeros: another variant ran) */
int gkmb200_problem_index_layout(const gkmb200_problem *p, int *out);
/* the index variant's column blocks of the last compute call on p, on its first GPU: returns their number (0: another
 * variant ran; -1: error) and fills 8 values per block for the first `max` of them: {first column, end column, slot format
 * (0 P32, 1 C16, 2 W20), postings, sum of squared posting-list lengths, row-kernel builds that ran (bit 2 RANGE + MINB - 1),
 * most dynamic shared memory of one launch, launches} */
int gkmb200_problem_index_blocks(const gkmb200_problem *p, long long *out, int max);
/* out[4] = {variant (1 lmer, 2 diag, 3 mma), TA, TB, dynamic shared memory bytes} of the last bit-sliced, lmer or mma launch
 * made for p on its first GPU (mma: TA = queries per CTA, TB = targets per CTA); zeros if none */
int gkmb200_problem_launch_shape(const gkmb200_problem *p, int *out);
int gkmb200_get_stats(const gkmb200_problem *p, gkmb200_stats *out);
/* `steps` timed passes over the full lower triangle with inputs and outputs resident in HBM;
 * ms_each[steps] = CUDA-event time of each pass; flush_l2 != 0 rewrites a >L2-sized buffer between passes */
int gkmb200_bench_lower_resident(gkmb200_problem *p, int steps, int warmup, int flush_l2, double *ms_each);
/* micro-benchmarks behind the roofline denominators (bench.py), on the first selected GPU:
 *   "lop3" | "shf" | "popc" | "iadd3" | "imad" | "imadhi" | "lop3+imad" | "lop3+popc" | "lop3+imad+popc": 1e9 lane-ops per second;
 *   "gather16": 1e9 random 16-byte gathers per second from a 64 MB (L2-resident) table;
 *   "atoms7" | "atoms14" | "atoms32": 1e9 shared-memory atomic adds per second with ~7 / 14 / 32 of 32 lanes on per instruction */
int gkmb200_microbench(const char *what, double *result);

#ifdef __cplusplus
}
#endif

#endif /* GKM_B200_H_INCLUDED */
