/* gkm_dev.h -- internals shared by the .cu files of the device layer (C++, hidden: none of it is part of the ABI) */
#ifndef GKM_DEV_H_INCLUDED
#define GKM_DEV_H_INCLUDED

#include <cuda_runtime.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "gkm_internal.h"
#include "gkm_index_dev.h"
#include "gkm_mma_kernel.cuh"

#define GKM_MAX_DEV 16
#define GKM_NBUF 4 /* chunks in flight per GPU: kernels run ahead while the host scatters finished ones */

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            gkm_set_error("CUDA: %s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

/* per-GPU resources, created lazily and kept for the life of the process
 * (the ABI has no handle that survives gkm_main_pywrapper, SURVEY.md 8b) */
struct gkm_gpu {
    int id;
    int ready;
    cudaStream_t sc, sc2, sx;  /* compute (two, so that the tail of one chunk overlaps the head of the next), copy */
    cudaEvent_t join;
    cudaEvent_t span0;         /* start of the first kernel of a compute call */
    cudaEvent_t k0[GKM_NBUF], k1[GKM_NBUF];  /* kernel start / end per staging slot */
    cudaEvent_t cdone[GKM_NBUF];             /* D2H complete per staging slot */
    void *d_band[GKM_NBUF];
    size_t band_cap;
    void *h_stage[GKM_NBUF];
    size_t stage_cap;
    void *d_flush;
    /* small cache of device blocks: cudaMalloc/cudaFree per call cost up to a second of host time on
     * this driver (measured: sporadic 0.2-1.3 s inside gkm_main_pywrapper), so image buffers are recycled */
    struct { void *ptr; size_t bytes; } pool[32];
    int npool;
    /* "index" variant: XOR masks of the (L, d) last used on this GPU */
    uint32_t *d_deltas;
    size_t deltas_bytes;
    int delta_L, delta_d, ndelta, ncold;
    int32_t *d_cold[2];   /* cold-bin scratch of the launches on sc / sc2 */
    long long nkernels;   /* histogram kernels launched on this GPU so far (the statistics report differences) */
    size_t cold_cap[2];
};

struct gkm_image {
    uint32_t *planes;
    int32_t *lens;
    uint8_t *wend;
    double *sqnorm;
    uint8_t *codes;     /* device packing: the base codes as uploaded (one byte per base), kept until release */
    uint32_t *pimg;     /* "mma" variant: copy of planes with a 16-byte row pitch, the source of its TMA loads */
    size_t pimg_bytes;
    CUtensorMap tmap;   /* 2-D map over pimg: {P words, n rows}, box {box words, 1 row} */
    gkm_mma_args mma;
    size_t planes_bytes, lens_bytes, wend_bytes, sqnorm_bytes, codes_bytes; /* block sizes as handed out by the pool */
    double *full;       /* resident N x ldfull result (bench, svm consumer) */
    size_t full_ld;
    int full_sym;       /* the resident matrix is complete and symmetric (unit diagonal) */
    /* "index" variant: one inverted index per block of blk_cols columns, built on first use */
    gkm_idx_block *blk;
    int nblk, blk_cols;
    int blk_greedy;       /* the blocks were cut full-size first (index_split) */
    int part_lo, part_hi; /* the column range the blocks partition (that of the call that created them) */
    int shape[4];         /* {variant, TA, TB, dynamic shared memory bytes} of the last bit-sliced, lmer or mma launch (slot 0) */
};

struct gkm_devstate {
    int ndev;
    int dev[GKM_MAX_DEV];
    gkm_image img[GKM_MAX_DEV];
    int variant;        /* kernel variant of the compute call in progress (choose_variant) */
};

#pragma GCC visibility push(hidden)

extern gkm_gpu g_gpu[GKM_MAX_DEV];
extern int g_sel[GKM_MAX_DEV];
extern int g_nsel;
extern pthread_mutex_t g_lock;

/* body(slot) for every GPU slot of ds side by side, with that slot's device current: slot 0 on the caller's thread, the
 * others on threads of their own (on the caller's thread too if one cannot start).  The error text is per thread
 * (gkm_log.c), so a failing slot's is handed over to the caller's. */
template <class F>
static int for_each_gpu(const gkm_devstate *ds, const F &body)
{
    struct slot_run { const F *body; int dev, slot, rc; char err[256]; } run[GKM_MAX_DEV];
    void *(*go)(void *) = [](void *a) -> void * {
        slot_run *r = (slot_run *) a;
        r->rc = 1;
        if (cudaSetDevice(r->dev) != cudaSuccess) gkm_set_error("CUDA: cannot select device %d", r->dev);
        else r->rc = (*r->body)(r->slot);
        if (r->rc) snprintf(r->err, sizeof(r->err), "%s", gkmb200_last_error());
        return NULL;
    };
    pthread_t th[GKM_MAX_DEV];
    int started[GKM_MAX_DEV];
    for (int i = 0; i < ds->ndev; i++) {
        run[i].body = &body; run[i].dev = ds->dev[i]; run[i].slot = i; run[i].rc = 0;
        started[i] = i > 0 && pthread_create(&th[i], NULL, go, &run[i]) == 0;
    }
    go(&run[0]);
    for (int i = 1; i < ds->ndev; i++) { if (started[i]) pthread_join(th[i], NULL); else go(&run[i]); }
    for (int i = 0; i < ds->ndev; i++) if (run[i].rc) { gkm_set_error("%s", run[i].err); return 1; }
    return 0;
}

/* body(slot, begin, end) for one contiguous share of [0, count) per GPU slot: shares of ceil(count / ndev) items rounded up
 * to a multiple of align, the last ones shorter or empty */
template <class F>
static int for_each_gpu_share(const gkm_devstate *ds, long long count, long long align, const F &body)
{
    const long long per = ((count + ds->ndev - 1) / ds->ndev + align - 1) / align * align;
    return for_each_gpu(ds, [&](int slot) {
        const long long b = slot * per < count ? slot * per : count, e = b + per < count ? b + per : count;
        return body(slot, b, e);
    });
}

/* ---- gkm_device.cu ---- */
double now_ms(void);
cudaError_t dev_malloc(gkm_gpu *g, void **out, size_t bytes);
int pool_alloc(gkm_gpu *g, void **out, size_t *got, size_t bytes);
void pool_free(gkm_gpu *g, void *ptr, size_t bytes);
int ensure_selected(void);
int gpu_prepare(gkm_gpu *g, int id, size_t band_bytes, size_t stage_bytes);
int stream_join(gkm_gpu *g, cudaStream_t from, cudaStream_t to);
cudaError_t gpu_drain(gkm_gpu *g, int with_copy_stream);
int upload_locked(gkmb200_problem *p, int need_host);

/* device memory of one GPU for the length of a scope: allocated with dev_malloc, freed on scope exit (with its GPU
 * current) unless release() hands it on */
template <class T>
struct gkm_dbuf {
    gkm_gpu *g;
    T *ptr = nullptr;
    explicit gkm_dbuf(gkm_gpu *gpu) : g(gpu) {}
    gkm_dbuf(const gkm_dbuf &) = delete;
    gkm_dbuf &operator=(const gkm_dbuf &) = delete;
    ~gkm_dbuf() { if (ptr) cudaFree(ptr); }
    cudaError_t alloc(size_t count) /* count elements of T, in place of what the buffer held */
    {
        if (ptr) { cudaFree(ptr); ptr = nullptr; }
        return dev_malloc(g, (void **) &ptr, count * sizeof(T));
    }
    T *release() { T *q = ptr; ptr = nullptr; return q; }
    operator T *() const { return ptr; }
};

/* ---- gkm_launch.cu ---- */
void fill_kparams(const gkmb200_problem *p, const gkm_image *im, int mode, gkm_kparams *kp);
gkm_kparams chunk_kparams(const gkmb200_problem *p, const gkm_image *im, const gkm_chunk *c, int mode);
int launch_hist(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, gkm_kparams kp, cudaStream_t st, int *variant_out);
int launch_diag_rows(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, int r0, int r1, gkm_kparams kp);
int choose_variant(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower);
void release_index(gkm_gpu *g, gkm_image *im);
int column_keys_prepare(const gkmb200_problem *p, const gkm_image *im, int cb, int ce, gkm_idx_build_args *a, uint32_t **offs, size_t *sbytes);

/* ---- gkm_compute.cu ---- */
int plan_chunks(const gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower, int nshare, gkm_chunk **out);

#pragma GCC visibility pop

#endif
