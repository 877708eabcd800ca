/* gkm_internal.h -- host-side internals of gkmkern_pylib.so (C, shared with the .cu files) */
#ifndef GKM_INTERNAL_H_INCLUDED
#define GKM_INTERNAL_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#include "../../include/gkm_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define GKM_MAX_L 16       /* one L-mer fits a 32-bit word (2 bits per base) */
#define GKM_MAX_BINS 16    /* d <= 15 */
#define GKM_MAX_BASES 2047 /* MAX_SEQ_LENGTH - 1, libgkm.c:1294-1299 */

/* ---- logging (gkm_log.c): same look as the reference's clog format "%l %d %t: %m\n" ---- */
enum { GKM_LOG_TRACE = 0, GKM_LOG_DEBUG, GKM_LOG_INFO, GKM_LOG_WARN, GKM_LOG_ERROR };
void gkm_log_set_level(int level);
int gkm_log_get_level(void);
void gkm_log(int level, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
void gkm_set_error(const char *fmt, ...) __attribute__((format(printf, 1, 2)));

/* ---- parameters and weights (gkm_weights.c) ---- */
const char *gkm_param_problem(const gkm_parameter *p, int max_L);
int gkm_calc_weights(int kernel_type, int L, int k, double *w /* L+1 slots */);
void gkm_calc_posweights(int nk, int kernel_type, int M, double H, uint8_t *wt, uint8_t *wt_rc);

/* ---- the problem: sequences, their packed form, and (opaque) device state ---- */
struct gkm_devstate; /* gkm_dev.h */

struct gkmb200_problem {
    gkm_parameter param;
    double w[GKM_MAX_L + 1];
    int nbins;     /* d + 1 */
    int weighted;  /* kernel types 4, 5 */
    int n, cap;
    int npos;      /* set by read_problem */
    int *len;      /* bases per sequence */
    uint8_t *arena;/* forward strands of all sequences back to back, the LETTERS as they were given (either case, anything
                    * else than ACGT counts as A: gkm_base_code): what goes to the GPU, which codes and packs them */
    size_t arena_len, arena_cap;
    size_t *off;   /* first base of sequence i in the arena */
    char **sid;    /* FASTA record ids (first token after '>', libgkm.c:1287-1292); NULL for sequences added in memory */
    int nonacgt;   /* characters mapped to 'A' so far */

    /* shape of the packed image (gkm_shape_problem); the image itself is built ON THE DEVICE from the arena
     * (gkm_device.cu: gkm_pack_kernel).  planes / wend on the host exist only after gkm_pack_problem, which only the CPU
     * emulators of the test tier call; both packers apply the rule of gkm_pack.h. */
    int packed;
    int Wmax;        /* 32-bit words per bit plane = ceil(2*maxlen / 32): both strands in one circular string */
    int Wa;          /* ceil(maxlen / 32): 32-position chunks of a query */
    int maxlen;      /* longest sequence */
    uint32_t *planes;/* [n][3][Wmax]: code bit 0, code bit 1, valid-window-end plane E */
    uint8_t *wend;   /* weighted only: [n][32*Wmax] weight by window END position */
    double *sqnorm;  /* [n], filled by the device */
    int have_sqnorm;   /* computed (or queued) on the devices */
    int host_sqnorm;   /* copied back into sqnorm[] */

    int shard_rank, shard_world;
    struct gkm_devstate *dev;
    gkmb200_stats stats;
};

int gkm_problem_reserve(gkmb200_problem *p, int extra);
void gkm_problem_shard_from_env(gkmb200_problem *p); /* GKM_SHARD="rank/world": gkm_main_pywrapper only */
int gkm_shape_problem(gkmb200_problem *p);   /* Wmax, Wa, sqnorm buffer; no image */
int gkm_pack_problem(gkmb200_problem *p);    /* + the image on the host (CPU emulators only) */
static inline const uint8_t *gkm_letters(const gkmb200_problem *p, int i) { return p->arena + p->off[i]; }
/* A,C,G,T (either case) -> 0..3; anything else counts as 'A' (libgkm.c:864-875).  With the case bit cleared the four letters
 * are 0x41, 0x43, 0x47, 0x54: t = (ch >> 1) & 3 is 0,1,3,2 and t ^ (t >> 1) is 0,1,2,3.  The device packer
 * (gkm_device.cu: gkm_pack_kernel) applies the same rule. */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline uint8_t gkm_base_code(unsigned char ch)
{
    const unsigned u = ch & 0xDFu, t = (ch >> 1) & 3u;
    return (u == 'A' || u == 'C' || u == 'G' || u == 'T') ? (uint8_t) (t ^ (t >> 1)) : (uint8_t) 0;
}
/* positional weight by distance from the centre L-mer (libgkm.c:910-932): tab[dist], dist = 0..GKM_MAX_BASES */
void gkm_posweight_table(int kernel_type, int M, double H, uint8_t *tab);
void gkm_unpack_problem(gkmb200_problem *p);

/* ---- chunk planning (gkm_sched.c), pure host logic ---- */
typedef struct gkm_chunk {
    int row_begin, row_end; /* query rows [row_begin, row_end) */
    int col_begin, col_end; /* target columns computed for these rows */
    long long entries;      /* kernel entries this chunk produces */
} gkm_chunk;

/* split rows [row0,row0+nrows) x cols [col0,col0+ncols) into chunks of whole row tiles.
 * lower != 0: only columns j < row are needed (triangular matrix path).
 * Returns the number of chunks written (<= max_chunks) or -1. */
int gkm_plan_chunks(int row0, int nrows, int col0, int ncols, int lower, int tile_rows,
                    long long max_chunk_bytes, gkm_chunk *out, int max_chunks);
int gkm_plan_chunks_rows(int row0, int nrows, int col0, int ncols, int lower, int tile_rows,
                         long long max_chunk_bytes, int max_rows, gkm_chunk *out, int max_chunks);
/* which chunks belong to shard `rank` of `world` (round-robin by descending cost) */
int gkm_chunk_owner(int chunk_index, int nchunks, int world);
/* the index variant's column blocks: how many, and the width of all but the last in *cols */
int gkm_plan_index_blocks(int span, int cap, int greedy, int *cols);

/* ---- device layer (gkm_device.cu, gkm_compute.cu, gkm_resident.cu, gkm_microbench.cu) ---- */
int gkm_dev_count(void);
int gkm_dev_select(const int *ids, int n);
int gkm_dev_upload(gkmb200_problem *p);            /* planes -> every selected GPU, sqnorm on GPU */
void gkm_dev_release(gkmb200_problem *p);
/* host destinations: either dense `out` (ld doubles per row) or row pointers `rows` (rows[r][c]) */
int gkm_dev_compute(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower,
                    double *out, long ld, double **rows, int32_t *hist, int copy_threads);
int gkm_dev_decision(gkmb200_problem *p, int row0, int nrows, int col0, int ncols,
                     const double *alpha, double bias, double *out);
int gkm_dev_bench_lower(gkmb200_problem *p, int steps, int warmup, int flush_l2, double *ms_each);
int gkm_dev_microbench(const char *what, double *result);
int gkm_dev_svm_cv(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                   const int *train_idx, const signed char *train_y, const int *test_idx,
                   double C, double eps, int max_iter, double *scores, gkmb200_svm_fit *fits, double *alpha);

#ifdef __cplusplus
}
#endif

#endif
