/* gkm_device.cu -- device layer of gkmkern_pylib.so: GPU selection, the resident
 * problem image, kernel launches over chunks of row tiles, and the return path
 * into caller memory.
 *
 * Stands where the reference has its pthread row scheduler and row loop
 * (gkmkern_pylib.c:70-90,169-216 -> libgkm.c:1156): thread t there takes rows
 * t, t+T, ...; here one host thread per GPU takes whole chunks of row tiles, the
 * GPU computes chunk i+1 while chunk i is copied D2H (second stream, pinned
 * staging) and scattered into the caller's rows by `copy_threads` host threads.
 * The caller's matrix is neither pinned nor contiguous (numpy rows with a
 * 120 000-byte stride, gkmsvm.py:75-77), hence the bounce buffer.
 * There is no collective: every chunk depends only on the replicated sequence image.
 */
#include <cuda_runtime.h>
#include <pthread.h>
#include <semaphore.h>
#include <unistd.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "gkm_internal.h"
#include "gkm_options.h"
#include "gkm_lmer_kernel.cuh"
#include "gkm_mma_kernel.cuh"
#include "gkm_index_dev.h"
#include "gkm_svm.h"

#define GKM_MAX_DEV 16
#define GKM_NBUF 4 /* chunks in flight per GPU: kernels run ahead while the host scatters finished ones */
#define GKM_FLUSH_BYTES ((size_t) 256 << 20) /* > 126 MB L2 */
#define GKM_WAVE_ROWS 148 /* rows of one wave of the index variant's row kernel: one CTA per row and SM */

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            gkm_set_error("CUDA: %s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

extern "C" {
const void *gkm_diag_fn_L2(int, int, int);  const void *gkm_diag_fn_L3(int, int, int);  const void *gkm_diag_fn_L4(int, int, int);
const void *gkm_diag_fn_L5(int, int, int);  const void *gkm_diag_fn_L6(int, int, int);  const void *gkm_diag_fn_L7(int, int, int);
const void *gkm_diag_fn_L8(int, int, int);  const void *gkm_diag_fn_L9(int, int, int);  const void *gkm_diag_fn_L10(int, int, int);
const void *gkm_diag_fn_L11(int, int, int); const void *gkm_diag_fn_L12(int, int, int); const void *gkm_diag_fn_L13(int, int, int);
const void *gkm_diag_fn_L14(int, int, int); const void *gkm_diag_fn_L15(int, int, int); const void *gkm_diag_fn_L16(int, int, int);
}

static const void *diag_fn(int L, int nb, int weighted, int d)
{
    switch (L) {
        case 2: return gkm_diag_fn_L2(nb, weighted, d);   case 3: return gkm_diag_fn_L3(nb, weighted, d);
        case 4: return gkm_diag_fn_L4(nb, weighted, d);   case 5: return gkm_diag_fn_L5(nb, weighted, d);
        case 6: return gkm_diag_fn_L6(nb, weighted, d);   case 7: return gkm_diag_fn_L7(nb, weighted, d);
        case 8: return gkm_diag_fn_L8(nb, weighted, d);   case 9: return gkm_diag_fn_L9(nb, weighted, d);
        case 10: return gkm_diag_fn_L10(nb, weighted, d); case 11: return gkm_diag_fn_L11(nb, weighted, d);
        case 12: return gkm_diag_fn_L12(nb, weighted, d); case 13: return gkm_diag_fn_L13(nb, weighted, d);
        case 14: return gkm_diag_fn_L14(nb, weighted, d); case 15: return gkm_diag_fn_L15(nb, weighted, d);
        case 16: return gkm_diag_fn_L16(nb, weighted, d);
        default: return NULL;
    }
}

/* ------------------------------------------------------------------ */
/* per-GPU resources, created lazily and kept for the life of the process
 * (the ABI has no handle that survives gkm_main_pywrapper, SURVEY.md 8b) */
/* ------------------------------------------------------------------ */
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

static gkm_gpu g_gpu[GKM_MAX_DEV];
static int g_sel[GKM_MAX_DEV];
static int g_nsel = -1;
static pthread_mutex_t g_lock = PTHREAD_MUTEX_INITIALIZER;

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

/* give the cached blocks of one GPU back to the driver (current device must be g's) */
static void pool_trim(gkm_gpu *g)
{
    for (int i = 0; i < g->npool; i++) cudaFree(g->pool[i].ptr);
    g->npool = 0;
}

/* cudaMalloc that, when the device is out of memory, first returns this library's own cached blocks (up to 32 blocks
 * of up to 512 MB per GPU would otherwise stand between a long-lived host and a 50k x 50k problem) and tries again */
static cudaError_t dev_malloc(gkm_gpu *g, void **out, size_t bytes)
{
    cudaError_t e = cudaMalloc(out, bytes);
    if (e == cudaErrorMemoryAllocation && g->npool > 0) {
        cudaGetLastError();
        gkm_log(GKM_LOG_DEBUG, "GPU %d: out of memory for %zu bytes, releasing %d cached blocks", g->id, bytes, g->npool);
        pool_trim(g);
        e = cudaMalloc(out, bytes);
    }
    return e;
}

static double now_ms(void)
{
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return 1e3 * (double) t.tv_sec + 1e-6 * (double) t.tv_nsec;
}

extern "C" int gkm_dev_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n && i < GKM_MAX_DEV; i++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

extern "C" int gkmb200_device_count(void) { return gkm_dev_count(); }

extern "C" int gkm_dev_select(const int *ids, int n)
{
    int total = 0;
    if (cudaGetDeviceCount(&total) != cudaSuccess) { cudaGetLastError(); total = 0; }
    if (n < 1 || n > GKM_MAX_DEV) { gkm_set_error("bad device list"); return 1; }
    for (int i = 0; i < n; i++) {
        int major = 0;
        if (ids[i] < 0 || ids[i] >= total ||
            cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, ids[i]) != cudaSuccess || major != 10) {
            gkm_set_error("device %d is not a visible sm_100 GPU", ids[i]);
            return 1;
        }
    }
    for (int i = 0; i < n; i++) g_sel[i] = ids[i];
    g_nsel = n;
    return 0;
}

extern "C" int gkmb200_set_devices(const int *ids, int n) { return gkm_dev_select(ids, n); }

static int ensure_selected(void)
{
    if (g_nsel > 0) return 0;
    const char *env = getenv("GKM_DEVICES");
    if (env && *env) {
        int ids[GKM_MAX_DEV], n = 0;
        const char *s = env;
        while (*s && n < GKM_MAX_DEV) {
            ids[n++] = (int) strtol(s, (char **) &s, 10);
            while (*s == ',' || *s == ' ') s++;
        }
        return gkm_dev_select(ids, n);
    }
    int total = 0, n = 0, ids[GKM_MAX_DEV];
    if (cudaGetDeviceCount(&total) != cudaSuccess) { cudaGetLastError(); total = 0; }
    for (int i = 0; i < total && n < GKM_MAX_DEV; i++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ids[n++] = i;
    }
    if (n == 0) {
        gkm_set_error("no sm_100 (B200) GPU is visible: gkmkern_pylib.so has no CPU fallback");
        return 1;
    }
    return gkm_dev_select(ids, n);
}

static int gpu_prepare(gkm_gpu *g, int id, size_t band_bytes, size_t stage_bytes)
{
    CK(cudaSetDevice(id));
    if (!g->ready) {
        g->id = id;
        CK(cudaStreamCreateWithFlags(&g->sc, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&g->sc2, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&g->join, cudaEventDisableTiming));
        CK(cudaEventCreate(&g->span0));
        CK(cudaStreamCreateWithFlags(&g->sx, cudaStreamNonBlocking));
        for (int i = 0; i < GKM_NBUF; i++) {
            CK(cudaEventCreate(&g->k0[i]));
            CK(cudaEventCreate(&g->k1[i]));
            CK(cudaEventCreateWithFlags(&g->cdone[i], cudaEventDisableTiming));
        }
        g->ready = 1;
    }
    if (band_bytes > g->band_cap) {
        for (int i = 0; i < GKM_NBUF; i++) { if (g->d_band[i]) cudaFree(g->d_band[i]); g->d_band[i] = NULL; }
        g->band_cap = 0;
        for (int i = 0; i < GKM_NBUF; i++) CK(dev_malloc(g, &g->d_band[i], band_bytes));
        g->band_cap = band_bytes;
    }
    if (stage_bytes > g->stage_cap) {
        for (int i = 0; i < GKM_NBUF; i++) { if (g->h_stage[i]) cudaFreeHost(g->h_stage[i]); g->h_stage[i] = NULL; }
        g->stage_cap = 0;
        for (int i = 0; i < GKM_NBUF; i++) CK(cudaMallocHost(&g->h_stage[i], stage_bytes));
        g->stage_cap = stage_bytes;
    }
    return 0;
}

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

/* ------------------------------------------------------------------ */
/* one launch of a histogram kernel over the block described by kp     */
/* ------------------------------------------------------------------ */
/* variant named by the option, without the index (which is decided per compute call, choose_variant) */
static int base_variant(const gkmb200_problem *p)
{
    int v = gkm_opt_kernel();
    if (v == GKM_KERNEL_LMER) return GKM_KERNEL_LMER;
    if (v == GKM_KERNEL_MMA && p->param.d < p->param.L) return GKM_KERNEL_MMA; /* needs >= 1 matching base per hit */
    return GKM_KERNEL_DIAG;
}

static int pick_variant(const gkmb200_problem *p, int mode)
{
    int v = (p->dev && p->dev->variant) ? p->dev->variant : base_variant(p);
    if ((v == GKM_KERNEL_INDEX || v == GKM_KERNEL_MMA) && mode == GKM_MODE_DIAG) v = GKM_KERNEL_DIAG; /* sqnorm: n pairs only */
    return v;
}

/* "index" variant: one row-kernel launch per index block that holds wanted columns */
static int launch_index(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, const gkm_kparams &kp, cudaStream_t st)
{
    int a_max = kp.row_end - 1;
    for (int k = 0; k < im->nblk; k++) {
        const gkm_idx_block *b = &im->blk[k];
        int lo = kp.col_begin > b->cb ? kp.col_begin : b->cb;
        int hi = kp.col_end < b->ce ? kp.col_end : b->ce;
        if (kp.mode == GKM_MODE_LOWER && hi > a_max) hi = a_max; /* columns < row only */
        if (hi <= lo) continue;
        if (!b->built) { gkm_set_error("index block %d is not built", k); return 1; }
        gkm_idx_rowargs ra;
        ra.fmt = b->fmt; ra.tab = b->tab; ra.ovf = b->ovf; ra.deltas = g->d_deltas; ra.ndelta = g->ndelta;
        ra.nslots = 1u << (2 * p->param.L);
        ra.cb = b->cb; ra.blo = lo - b->cb; ra.bhi = hi - b->cb;
        ra.ldh = (ra.bhi - ra.blo + 31) & ~31;
        ra.blk_cols = b->ce - b->cb;
        ra.nblk = im->nblk;
        ra.skew = b->skew;
        ra.maxq = 32 * p->Wa;
        ra.ncold = g->ncold;
        {   /* cold-bin scratch of this stream, grown on demand (the stream is drained before a block is replaced) */
            const int si = (st == g->sc2) ? 1 : 0;
            const size_t need = gkm_idx_cold_bytes(p->nbins, ra.ldh, kp.row_end - kp.row_begin);
            if (need > g->cold_cap[si]) {
                CK(cudaStreamSynchronize(st));
                if (g->d_cold[si]) cudaFree(g->d_cold[si]);
                g->d_cold[si] = NULL; g->cold_cap[si] = 0;
                const size_t want = need + need / 4 + 4096;
                CK(dev_malloc(g, (void **) &g->d_cold[si], want));
                g->cold_cap[si] = want;
            }
            ra.cold = g->d_cold[si];
        }
        if (gkm_idx_rows(&kp, &ra, p->weighted, st)) return 1;
        g->nkernels++;
    }
    return 0;
}

static int pool_alloc(gkm_gpu *g, void **out, size_t *got, size_t bytes);
static void pool_free(gkm_gpu *g, void *ptr, size_t bytes);

/* "mma" variant: the 16-byte-pitched copy of the plane image and the TMA descriptor over it, made on first use */
typedef CUresult (*gkm_encode_tiled_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                        const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int ensure_mma(const gkmb200_problem *p, gkm_image *im, gkm_gpu *g, cudaStream_t st)
{
    if (im->pimg) return 0;
    const size_t n = (size_t) p->n, W3 = 3 * (size_t) p->Wmax;
    const size_t P = (W3 + 3) & ~(size_t) 3;
    static gkm_encode_tiled_fn encode = NULL;
    if (!encode) {
        void *fn = NULL;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn || qres != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            gkm_set_error("mma variant: the driver has no cuTensorMapEncodeTiled");
            return 1;
        }
        encode = (gkm_encode_tiled_fn) fn;
    }
    if (pool_alloc(g, (void **) &im->pimg, &im->pimg_bytes, n * P * 4)) return 1;
    CK(cudaMemsetAsync(im->pimg, 0, n * P * 4, st));
    CK(cudaMemcpy2DAsync(im->pimg, P * 4, im->planes, W3 * 4, W3 * 4, n, cudaMemcpyDeviceToDevice, st));
    im->mma.P = (int) P;
    im->mma.nbox = (int) ((P + GKM_MMA_TMA_BOX - 1) / GKM_MMA_TMA_BOX);
    im->mma.box = (int) ((((P + im->mma.nbox - 1) / im->mma.nbox) + 31) & ~(size_t) 31); /* 128-byte pieces: every box lands 128-byte aligned */
    const int maxnk = p->maxlen - p->param.L + 1;
    im->mma.QA = GKM_MMA_ROWS_CAP / (maxnk > 0 ? maxnk : 1);
    if (im->mma.QA > GKM_MMA_QA) im->mma.QA = GKM_MMA_QA;
    if (im->mma.QA < 1) {
        cudaStreamSynchronize(st);
        pool_free(g, im->pimg, im->pimg_bytes); im->pimg = NULL; /* no half-made image: the next call starts over */
        gkm_set_error("sequence too long for the mma kernel");
        return 1;
    }
    const cuuint64_t gdim[2] = { (cuuint64_t) P, (cuuint64_t) n };
    const cuuint64_t gstr[1] = { (cuuint64_t) P * 4 };
    const cuuint32_t box[2] = { (cuuint32_t) im->mma.box, 1 };
    const cuuint32_t estr[2] = { 1, 1 };
    const CUresult r = encode(&im->tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, im->pimg, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        cudaStreamSynchronize(st); /* the copy into the block must not outlive its owner */
        pool_free(g, im->pimg, im->pimg_bytes); im->pimg = NULL;
        gkm_set_error("mma variant: cuTensorMapEncodeTiled failed (%d)", (int) r);
        return 1;
    }
    return 0;
}

/* the tile shape (TA, TB) of a bit-sliced or lmer launch: the first candidate, in order, whose shared memory
 * bytes(TA, TB) fit `lim`, else the first that fits 220 KB */
template <int N, class F>
static int pick_tile(const int (&cand)[N][2], unsigned lim, const F &bytes, gkm_kparams *kp, unsigned *smem)
{
    for (int pass = 0; pass < 2; pass++)
        for (int i = 0; i < N; i++) {
            const unsigned s = bytes(cand[i][0], cand[i][1]);
            if (s <= (pass == 0 ? lim : 220u * 1024u)) { kp->TA = cand[i][0]; kp->TB = cand[i][1]; *smem = s; return 0; }
        }
    gkm_set_error("sequence too long for shared memory");
    return 1;
}

static int launch_hist(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, gkm_kparams kp, cudaStream_t st, int *variant_out)
{
    const int variant = pick_variant(p, kp.mode);
    const int rows = kp.row_end - kp.row_begin, cols = kp.col_end - kp.col_begin;
    if (rows <= 0 || cols <= 0) return 0;
    if (variant == GKM_KERNEL_INDEX) {
        if (variant_out) *variant_out = variant;
        return launch_index(p, im, g, kp, st);
    }
    const void *fn = NULL;
    unsigned smem = 0, threads = 256;
    void *args[3] = { &kp }; /* each kernel reads the leading entries it takes */
    if (variant == GKM_KERNEL_DIAG) {
        const int nb = gkm_diag_nb(p->param.d);
        fn = diag_fn(p->param.L, nb, p->weighted, p->param.d);
        if (!fn) { gkm_set_error("no diag kernel for L=%d", p->param.L); return 1; }
        /* TB = 32 makes the lane-task count of a uniform-length tile a multiple of the warp size */
        static const int cand[][2] = { {8, 32}, {4, 32}, {4, 16}, {2, 16}, {2, 8}, {2, 4}, {2, 2}, {2, 1} }; /* TA even: queries go in pairs */
        if (pick_tile(cand, 74u * 1024u, [&](int ta, int tb) { return gkm_diag_layout(p->Wmax, p->Wa, ta, tb, nb, p->weighted).total; },
                      &kp, &smem)) return 1;
    } else if (variant == GKM_KERNEL_MMA) {
        gkm_image *imw = const_cast<gkm_image *>(im);
        if (ensure_mma(p, imw, g, st)) return 1;
        if (st == g->sc) { CK(cudaEventRecord(g->join, g->sc)); CK(cudaStreamWaitEvent(g->sc2, g->join, 0)); } /* the other compute stream sees the copy too */
        fn = p->weighted ? (const void *) gkm_mma_kernel<true> : (const void *) gkm_mma_kernel<false>;
        const int maxnk = p->maxlen - p->param.L + 1;
        const int tiles = (im->mma.QA * maxnk + GKM_MMA_M - 1) / GKM_MMA_M;
        smem = gkm_mma_smem_bytes(tiles, gkm_mma_stage_words(im->mma), p->nbins, p->weighted);
        if (smem > 227u * 1024u) { gkm_set_error("sequence too long for the mma kernel"); return 1; }
        kp.TA = im->mma.QA;
        kp.TB = GKM_MMA_TB;
        threads = GKM_MMA_THREADS;
        args[1] = (void *) &im->mma;
        args[2] = (void *) &im->tmap;
    } else {
        fn = p->weighted ? (const void *) gkm_lmer_kernel<true> : (const void *) gkm_lmer_kernel<false>;
        static const int cand[][2] = { {8, 8}, {4, 4}, {2, 2}, {1, 1} };
        if (pick_tile(cand, 100u * 1024u, [&](int ta, int tb) { return gkm_lmer_smem_bytes(p->Wa, ta, tb, p->nbins, p->weighted); },
                      &kp, &smem)) return 1;
    }
    CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    dim3 grid((unsigned) ((cols + kp.TB - 1) / kp.TB), (unsigned) ((rows + kp.TA - 1) / kp.TA), 1);
    /* the diagonal: one CTA per row tile (it finds its own column tile), where the tile shapes allow it */
    if (kp.mode == GKM_MODE_DIAG && variant == GKM_KERNEL_DIAG && kp.TB % kp.TA == 0 && kp.row_begin == kp.col_begin) grid.x = 1;
    if (grid.y > 65535u) { gkm_set_error("chunk has too many row tiles"); return 1; }
    CK(cudaLaunchKernel(fn, grid, dim3(threads, 1, 1), args, smem, st));
    g->nkernels++;
    if (im == &p->dev->img[0]) { /* what gkmb200_problem_launch_shape reports */
        int *s = const_cast<gkm_image *>(im)->shape;
        s[0] = variant; s[1] = kp.TA; s[2] = kp.TB; s[3] = (int) smem;
    }
    if (variant_out) *variant_out = variant;
    return 0;
}

static void fill_kparams(const gkmb200_problem *p, const gkm_image *im, int mode, gkm_kparams *kp)
{
    memset(kp, 0, sizeof(*kp));
    kp->mode = mode;
    kp->planes = im->planes;
    kp->lens = im->lens;
    kp->wend = im->wend;
    kp->sqnorm = im->sqnorm;
    kp->W = p->Wmax;
    kp->WA = p->Wa;
    kp->L = p->param.L;
    kp->d = p->param.d;
    kp->nbins = p->nbins;
    kp->kernel_type = p->param.kernel_type;
    kp->gamma = p->param.gamma;
    for (int m = 0; m < 16; m++) kp->w[m] = (m < p->nbins) ? p->w[m] : 0.0;
}

/* ------------------------------------------------------------------ */
/* upload: packed image to every selected GPU; sqnorm = diagonal of the kernel */
/* ------------------------------------------------------------------ */
/* device blocks come from / go back to a per-GPU free list (current device must be g's) */
static int pool_alloc(gkm_gpu *g, void **out, size_t *got, size_t bytes)
{
    const size_t need = (bytes + 65535) & ~(size_t) 65535;
    int best = -1;
    for (int i = 0; i < g->npool; i++)
        if (g->pool[i].bytes >= need && g->pool[i].bytes <= 4 * need && (best < 0 || g->pool[i].bytes < g->pool[best].bytes)) best = i;
    if (best >= 0) {
        *out = g->pool[best].ptr;
        *got = g->pool[best].bytes;
        g->pool[best] = g->pool[--g->npool];
        return 0;
    }
    CK(dev_malloc(g, out, need));
    *got = need;
    return 0;
}

static void pool_free(gkm_gpu *g, void *ptr, size_t bytes)
{
    if (!ptr) return;
    if (g->npool < 32 && bytes <= ((size_t) 512 << 20)) {
        g->pool[g->npool].ptr = ptr;
        g->pool[g->npool].bytes = bytes;
        g->npool++;
        return;
    }
    cudaFree(ptr);
}

/* ------------------------------------------------------------------ */
/* "index" variant: per-GPU mask list, per-image column-block indexes    */
/* ------------------------------------------------------------------ */
/* columns one index block may hold: what fits shared memory, or less when the option says so */
static int index_block_cap(const gkmb200_problem *p)
{
    int cap = gkm_idx_max_cols(p->nbins, 32 * p->Wa, p->weighted);
    if (p->weighted && cap > GKM_IDX_W20_MAX_COLS) cap = GKM_IDX_W20_MAX_COLS; /* 14-bit columns of the compact weighted slots */
    if (!p->weighted && cap > (GKM_IDX_C16_MAX_COLS & ~31)) cap = GKM_IDX_C16_MAX_COLS & ~31; /* 15-bit columns of the compact slots */
    const int opt = gkm_opt_index_cols();
    /* Default width of a full block: wider blocks mean fewer probes per row, denser slots (longer posting lists: more
     * overflow walks) and less L1 next to the histogram rows.  50k x 300 bp, L = 11, full blocks first: 12 512 columns
     * 672 ms, 16 384 609, 18 432 592, 20 480 586, 22 528 577, 25 024 633 (tools/split_ab2.py).  The option replaces this
     * default, not the limits of the formats. */
    const int lim = opt > 0 ? opt : 22528;
    if (lim < cap) cap = lim;
    return cap;
}

static void release_index(gkm_gpu *g, gkm_image *im)
{
    for (int k = 0; k < im->nblk; k++) {
        pool_free(g, im->blk[k].tab, im->blk[k].tab_bytes);
        pool_free(g, im->blk[k].ovf, im->blk[k].ovf_bytes);
    }
    free(im->blk);
    im->blk = NULL;
    im->nblk = 0;
}

static int ensure_deltas(gkm_gpu *g, int L, int d)
{
    if (g->d_deltas && g->delta_L == L && g->delta_d == d) return 0;
    const long long nd = gkm_idx_delta_count(L, d);
    if (nd <= 0) { gkm_set_error("index variant: too many masks for L=%d d=%d", L, d); return 1; }
    uint32_t *h = (uint32_t *) malloc((size_t) nd * 4);
    if (!h || gkm_idx_deltas(L, d, h, nd) != nd) { free(h); gkm_set_error("index variant: mask list failed"); return 1; }
    if (g->d_deltas) { cudaStreamSynchronize(g->sc); cudaStreamSynchronize(g->sc2); pool_free(g, g->d_deltas, g->deltas_bytes); g->d_deltas = NULL; }
    if (pool_alloc(g, (void **) &g->d_deltas, &g->deltas_bytes, (size_t) nd * 4)) { free(h); return 1; }
    cudaError_t e = cudaMemcpyAsync(g->d_deltas, h, (size_t) nd * 4, cudaMemcpyHostToDevice, g->sc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc); /* h is pageable and freed below */
    free(h);
    if (e != cudaSuccess) { gkm_set_error("CUDA: mask upload: %s", cudaGetErrorString(e)); return 1; }
    g->delta_L = L; g->delta_d = d; g->ndelta = (int) nd; g->ncold = (int) gkm_idx_cold_count(L, d);
    return 0;
}

/* build the indexes of the column blocks that intersect [col_begin, col_end); queued on g->sc */
static int ensure_index(gkmb200_problem *p, gkm_gpu *g, gkm_image *im, int col_begin, int col_end, int greedy, int strict)
{
    const int L = p->param.L;
    if (ensure_deltas(g, L, p->param.d)) return 1;
    /* The blocks partition the column range of the call that created them (the SVs of a scoring problem, all
     * sequences of a kernel matrix); a later call for columns outside that range starts over. */
    if (im->blk && (col_begin < im->part_lo || col_end > im->part_hi || (strict && im->blk_greedy != greedy))) { /* strict: the option names a split */
        cudaStreamSynchronize(g->sc); cudaStreamSynchronize(g->sc2);
        release_index(g, im);
    }
    if (!im->blk) {
        const int cap = index_block_cap(p);
        if (cap <= 0) { gkm_set_error("index variant: sequences too long for shared memory"); return 1; }
        const int span = col_end - col_begin;
        const int nblk = (span + cap - 1) / cap;
        /* equal shares, or -- greedy -- full blocks first and the rest in the last one: in a lower triangle row a probes
         * only the blocks that start below it, so the earlier a block ends the fewer rows pay for the next one */
        int cols = (((span + nblk - 1) / nblk) + 31) & ~31;
        if (cols > cap || greedy) cols = cap & ~31;
        im->blk_greedy = greedy;
        im->blk = (gkm_idx_block *) calloc((size_t) nblk, sizeof(gkm_idx_block));
        if (!im->blk) { gkm_set_error("out of memory"); return 1; }
        im->nblk = nblk;
        im->blk_cols = cols;
        im->part_lo = col_begin;
        im->part_hi = col_end;
        for (int k = 0; k < nblk; k++) {
            im->blk[k].cb = col_begin + k * cols;
            im->blk[k].ce = col_begin + (k + 1) * cols < col_end ? col_begin + (k + 1) * cols : col_end;
        }
    }
    for (int k = 0; k < im->nblk; k++) {
        gkm_idx_block *b = &im->blk[k];
        if (b->built || b->ce <= col_begin || b->cb >= col_end || b->ce <= b->cb) continue;
        const int nc = b->ce - b->cb;
        uint32_t *offs = (uint32_t *) malloc((size_t) nc * 4);
        if (!offs) { gkm_set_error("out of memory"); return 1; }
        size_t P = 0;
        for (int i = 0; i < nc; i++) { offs[i] = (uint32_t) P; P += 2 * (size_t) (p->len[b->cb + i] - L + 1); }
        if (P > 0x7FFFFFF0u) { free(offs); gkm_set_error("index variant: column block too large"); return 1; }
        size_t cub_bytes = 0;
        const size_t sbytes = gkm_idx_scratch_bytes(P, L, &cub_bytes);
        void *scratch = NULL, *d_offs = NULL;
        size_t scratch_got = 0, offs_got = 0;
        /* compact slots unless a limit of theirs is crossed (index_block_cap keeps the blocks below their column limits) */
        b->fmt = gkm_idx_block_fmt(p->weighted, p->param.M, nc, P, gkm_opt_index_wide());
        int rc = pool_alloc(g, (void **) &b->tab, &b->tab_bytes, gkm_idx_tab_bytes(L, b->fmt)) ||
                 pool_alloc(g, (void **) &b->ovf, &b->ovf_bytes, gkm_idx_ovf_bytes(P, b->fmt)) ||
                 pool_alloc(g, &scratch, &scratch_got, sbytes) ||
                 pool_alloc(g, &d_offs, &offs_got, (size_t) nc * 4);
        if (!rc) {
            cudaError_t e = cudaMemcpyAsync(d_offs, offs, (size_t) nc * 4, cudaMemcpyHostToDevice, g->sc);
            if (e != cudaSuccess) { gkm_set_error("CUDA: index offsets: %s", cudaGetErrorString(e)); rc = 1; }
        }
        if (!rc) {
            gkm_idx_build_args a;
            a.planes = im->planes; a.lens = im->lens; a.wend = p->weighted ? im->wend : NULL;
            a.W = p->Wmax; a.L = L; a.cb = b->cb; a.ce = b->ce;
            a.offs = (const uint32_t *) d_offs; a.P = P; a.scratch = scratch; a.cub_bytes = cub_bytes;
            a.fmt = b->fmt; a.tab = b->tab; a.ovf = b->ovf;
            b->sumsq = 0; a.h_sumsq = &b->sumsq;
            rc = gkm_idx_build(&a, g->sc);
        }
        /* pageable source and recycled scratch: wait for the build before letting go of them */
        if (cudaStreamSynchronize(g->sc) != cudaSuccess && !rc) { gkm_set_error("CUDA: index build failed: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
        free(offs);
        pool_free(g, scratch, scratch_got);
        pool_free(g, d_offs, offs_got);
        if (rc) return 1;
        b->skew = (double) b->sumsq / (double) (P ? P : 1);
        gkm_log(GKM_LOG_DEBUG, "index block %d: %zu postings, sum len^2 / postings = %.2f", k, P, b->skew);
        b->built = 1;
        __atomic_fetch_add(&p->stats.launches, 5, __ATOMIC_RELAXED); /* the GPUs of a call build their indexes side by side */
    }
    return 0;
}

/* which kernel variant serves a block of rows x cols; for the index also makes sure that the
 * indexes exist on every GPU.  Called under g_lock after upload_locked. */
static int choose_variant(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower)
{
    gkm_devstate *ds = p->dev;
    const int opt = gkm_opt_kernel();
    int v = base_variant(p);
    double ci = 0.0, cd = 0.0; /* estimates of kernel = auto */
    /* How the columns are cut into index blocks (index_split).  In a lower triangle row a probes only the blocks that start
     * below it: full blocks first, the rest last (50k: 16 384 + 16 384 + 16 384 + 848 columns = 2.03 n row-block probes
     * against 2.5 n for four equal blocks).  Measured (tools/split_ab.py, profiles/r2_index_split_ab.txt): 50k x 50k 672 ->
     * 609 ms with blocks of 16 384, 577 ms with blocks of 22 528; 20k wgkm 244 -> 225 ms.  A rectangle probes every block
     * from every row: equal shares there. */
    const int gopt = gkm_opt_index_greedy();
    const int greedy = gopt >= 0 ? gopt : (lower != 0);
    if ((opt == GKM_KERNEL_AUTO || opt == GKM_KERNEL_INDEX) && nrows > 0 && ncols > 0 &&
        gkm_idx_supported(p->param.L, p->param.d, p->nbins)) {
        const int cap = index_block_cap(p);
        int ok = cap > 0;
        int blocks = 0;
        if (ok) {
            blocks = (ncols + cap - 1) / cap;
            /* at most 8 GiB of slot tables per GPU */
            if ((double) blocks * (double) gkm_idx_tab_bytes(p->param.L, p->weighted ? GKM_IDX_FMT_P32 : GKM_IDX_FMT_C16) > 8.0 * 1073741824.0) ok = 0;
        }
        if (ok && opt == GKM_KERNEL_AUTO) {
            double sum = 0.0;
            for (int i = 0; i < p->n; i++) sum += (double) (p->len[i] - p->param.L + 1);
            const double nq = sum / (double) p->n;
            const long long entries = (long long) nrows * (long long) ncols / (lower ? 2 : 1);
            /* lower: row a probes only the blocks that start below it */
            double eff_blocks = lower ? 0.5 * (double) (blocks + 1) : (double) blocks;
            if (greedy) { /* rows of block k probe k + 1 blocks; all blocks but the last hold cap columns */
                const int capc = cap & ~31;
                double s = 0.0;
                for (int k = 0; k < blocks; k++) s += (double) (k + 1) * (double) ((k + 1) * capc <= ncols ? capc : ncols - k * capc);
                eff_blocks = s / (double) ncols;
            }
            ci = gkm_idx_cost_ms(p->param.L, p->param.d, p->weighted, nrows, nq, eff_blocks, entries, 2.0 * nq * nq);
            cd = gkm_diag_cost_ms(p->param.d, p->weighted, entries, 2.0 * nq * nq);
            ok = ci < cd;
            gkm_log(GKM_LOG_DEBUG, "kernel = auto: index %.2f ms vs diag %.2f ms (estimates)", ci, cd);
        }
        if (ok) v = GKM_KERNEL_INDEX;
    }
    if (v == GKM_KERNEL_INDEX) {
        /* every GPU builds its own copy of the (cheap) index: side by side, one host thread per GPU -- in turn the
         * builds of an 8-GPU call at 50k (4 column blocks each, a stream sync per block) were ~25 ms of host time */
        if (for_each_gpu(ds, [&](int slot) {
                gkm_gpu *g = &g_gpu[ds->dev[slot]];
                if (ensure_index(p, g, &ds->img[slot], col0, col0 + ncols, greedy, gopt >= 0)) return 1;
                CK(cudaEventRecord(g->join, g->sc));
                CK(cudaStreamWaitEvent(g->sc2, g->join, 0));
                return 0;
            })) return 1;
        /* kernel = auto, second look: the cost model above assumes random sequences.  The index build knows better:
         * a list of l postings is met by ~l/2 query L-mers of the same problem, l^2/4 exact-match hits in the lower
         * triangle.  Low-complexity input (thousands of poly-A sequences) makes that term seconds; the bit-sliced
         * kernel does not care what the sequences are. */
        if (opt == GKM_KERNEL_AUTO && lower && row0 == col0 && nrows == ncols) {
            const gkm_image *im = &ds->img[0];
            double sumsq = 0.0;
            for (int k = 0; k < im->nblk; k++)
                if (im->blk[k].built && im->blk[k].ce > col0 && im->blk[k].cb < col0 + ncols) sumsq += (double) im->blk[k].sumsq;
            const double extra = 1e3 * 0.25 * sumsq / 4.1e11;
            if (ci + extra > cd) {
                gkm_log(GKM_LOG_DEBUG, "kernel = auto: long posting lists add ~%.1f ms to the index estimate (%.1f ms): bit-sliced kernel (%.1f ms)", extra, ci, cd);
                v = base_variant(p);
            }
        }
    }
    (void) row0;
    ds->variant = v;
    return 0;
}

static int upload_locked(gkmb200_problem *p, int need_host);

/* the image as it lies on GPU 0 (tests: device packing against the host packer): planes [n][3][W] and, for the
 * weighted kernel types, wend [n][32 W]; either pointer may be NULL.  out_shape = {n, W}. */
extern "C" int gkmb200_problem_image(gkmb200_problem *p, uint32_t *planes, uint8_t *wend, int *out_shape)
{
    if (!p) { gkm_set_error("null problem"); return 1; }
    pthread_mutex_lock(&g_lock);
    int rc = upload_locked(p, 0);
    if (!rc) {
        gkm_devstate *ds = p->dev;
        gkm_gpu *g = &g_gpu[ds->dev[0]];
        const size_t n = (size_t) p->n, W = (size_t) p->Wmax;
        if (out_shape) { out_shape[0] = p->n; out_shape[1] = p->Wmax; }
        do {
            if (cudaSetDevice(ds->dev[0]) != cudaSuccess || cudaStreamSynchronize(g->sc) != cudaSuccess) { rc = 1; break; }
            if (planes && cudaMemcpy(planes, ds->img[0].planes, n * 3 * W * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { rc = 1; break; }
            if (wend && p->weighted && cudaMemcpy(wend, ds->img[0].wend, n * 32 * W, cudaMemcpyDeviceToHost) != cudaSuccess) { rc = 1; break; }
        } while (0);
        if (rc) gkm_set_error("CUDA: image read-back: %s", cudaGetErrorString(cudaGetLastError()));
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* how the last compute call of this problem cut its columns for the index variant: out = {number of column blocks,
 * columns per block, first column}; {0, 0, 0} when another variant ran.  For tests and the bench's parity rows. */
extern "C" int gkmb200_problem_index_layout(const gkmb200_problem *p, int *out)
{
    if (!p || !out) { gkm_set_error("null argument"); return 1; }
    out[0] = out[1] = out[2] = 0;
    pthread_mutex_lock(&g_lock);
    if (p->dev && p->dev->variant == GKM_KERNEL_INDEX && p->dev->img[0].blk) {
        out[0] = p->dev->img[0].nblk; out[1] = p->dev->img[0].blk_cols; out[2] = p->dev->img[0].part_lo;
    }
    pthread_mutex_unlock(&g_lock);
    return 0;
}

/* {variant, TA, TB, dynamic shared memory bytes} of the last bit-sliced, lmer or mma launch made for this problem on its
 * first GPU (mma: TA = queries per CTA, TB = 8); zeros if none.  For tests: which tile shape a problem ran. */
extern "C" int gkmb200_problem_launch_shape(const gkmb200_problem *p, int *out)
{
    if (!p || !out) { gkm_set_error("null argument"); return 1; }
    out[0] = out[1] = out[2] = out[3] = 0;
    pthread_mutex_lock(&g_lock);
    if (p->dev)
        for (int i = 0; i < 4; i++) out[i] = p->dev->img[0].shape[i];
    pthread_mutex_unlock(&g_lock);
    return 0;
}

/* drop every cached device block of every GPU (long-lived hosts that change L or n) */
extern "C" int gkmb200_trim(void)
{
    pthread_mutex_lock(&g_lock);
    for (int i = 0; i < GKM_MAX_DEV; i++) {
        gkm_gpu *g = &g_gpu[i];
        if (!g->ready || cudaSetDevice(g->id) != cudaSuccess) { cudaGetLastError(); continue; }
        cudaStreamSynchronize(g->sc); cudaStreamSynchronize(g->sc2); cudaStreamSynchronize(g->sx);
        pool_trim(g);
    }
    pthread_mutex_unlock(&g_lock);
    return 0;
}

extern "C" void gkm_dev_release(gkmb200_problem *p)
{
    if (!p || !p->dev) return;
    gkm_devstate *ds = p->dev;
    for (int i = 0; i < ds->ndev; i++) {
        if (cudaSetDevice(ds->dev[i]) != cudaSuccess) { cudaGetLastError(); continue; }
        gkm_gpu *g = &g_gpu[ds->dev[i]];
        gkm_image *im = &ds->img[i];
        /* nothing of this problem may still be running when its blocks are recycled */
        if (g->ready) { cudaStreamSynchronize(g->sc); cudaStreamSynchronize(g->sc2); cudaStreamSynchronize(g->sx); }
        pool_free(g, im->planes, im->planes_bytes);
        pool_free(g, im->lens, im->lens_bytes);
        pool_free(g, im->wend, im->wend_bytes);
        pool_free(g, im->sqnorm, im->sqnorm_bytes);
        pool_free(g, im->codes, im->codes_bytes);
        pool_free(g, im->pimg, im->pimg_bytes);
        release_index(g, im);
        cudaFree(im->full);
    }
    free(ds);
    p->dev = NULL;
}

/* ------------------------------------------------------------------ */
/* packing on the device (SURVEY.md 8f/f2): base codes -> the image of 3 */
/* ------------------------------------------------------------------ */
/* What gkm_seq.c:pack_worker does on the host (it stays there for the CPU emulators of the test tier), one CTA per
 * sequence, one warp per 32-position word of the circular string.  The input is the sequence TEXT, one byte per base as
 * the FASTA file or the caller spelled it: the letter -> code rule (A,C,G,T in either case -> 0..3, anything else -> A,
 * libgkm.c:864-875; gkm_base_code) is applied here.  Layout: forward strand at [0, len), reverse complement
 * (3 - code, mirrored: libgkm.c:878-888) at [len, 2 len), zero padding; plane bits by warp ballot; E = positions at
 * which an L-mer of either strand may end; wend[j] = positional weight of the L-mer ending at j, looked up by its
 * distance from the centre L-mer in a table the host computed with the reference's expression (libgkm.c:910-932) --
 * no exp() on the device, so the bytes are the host's. */
template <bool WEIGHTED>
__global__ void __launch_bounds__(128)
gkm_pack_kernel(const uint8_t *__restrict__ codes, const unsigned long long *__restrict__ off, const int32_t *__restrict__ lens,
                int W, int L, const uint8_t *__restrict__ wtab, uint32_t *__restrict__ planes, uint8_t *__restrict__ wend)
{
    const int i = (int) blockIdx.x;
    const int len = lens[i], nk = len - L + 1, centre = nk / 2;
    const uint8_t *c = codes + off[i];
    const int lane = (int) threadIdx.x & 31;
    for (int wi = (int) threadIdx.x >> 5; wi < W; wi += 4) {
        const int j = wi * 32 + lane;
        uint32_t code = 0;
        int s = -1; /* start index (forward-strand numbering of wt[]) of the L-mer that ends at j, if any */
        if (j < len) {
            code = gkm_base_code(c[j]);
            if (j >= L - 1) s = j - (L - 1);
        } else if (j < 2 * len) {
            code = 3u - gkm_base_code(c[2 * len - 1 - j]);
            const int rel = j - len;
            if (rel >= L - 1) s = nk - 1 - (rel - (L - 1)); /* wt_rc[t] = wt[nk - 1 - t] */
        }
        const uint32_t p0 = __ballot_sync(0xFFFFFFFFu, code & 1u), p1 = __ballot_sync(0xFFFFFFFFu, code & 2u);
        const uint32_t pe = __ballot_sync(0xFFFFFFFFu, s >= 0);
        if (lane == 0) {
            uint32_t *pl = planes + (size_t) i * 3 * (size_t) W;
            pl[wi] = p0; pl[W + wi] = p1; pl[2 * W + wi] = pe;
        }
        if (WEIGHTED) wend[(size_t) i * 32 * (size_t) W + (size_t) j] = (s >= 0) ? wtab[abs(centre - s)] : (uint8_t) 0;
    }
}

/* bring sqnorm back to the host (only the ABI functions that expose it need that) */
static int fetch_sqnorm(gkmb200_problem *p)
{
    if (p->host_sqnorm) return 0;
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[0]];
    CK(cudaSetDevice(ds->dev[0]));
    CK(cudaMemcpyAsync(p->sqnorm, ds->img[0].sqnorm, (size_t) p->n * sizeof(double), cudaMemcpyDeviceToHost, g->sc));
    CK(cudaStreamSynchronize(g->sc));
    p->host_sqnorm = 1;
    return 0;
}

/* need_host = 0: everything is only queued; later kernels are stream-ordered behind it */
static int upload_locked(gkmb200_problem *p, int need_host)
{
    if (p->dev && p->packed && p->have_sqnorm) return need_host ? fetch_sqnorm(p) : 0;
    if (ensure_selected()) return 1;
    const double t0 = now_ms();
    gkm_dev_release(p);
    const int pack_host = gkm_opt_pack_host();
    if (pack_host ? gkm_pack_problem(p) : gkm_shape_problem(p)) return 1;
    uint8_t wtab[GKM_MAX_BASES + 1];
    if (!pack_host && p->weighted) gkm_posweight_table(p->param.kernel_type, p->param.M, p->param.H, wtab);
    gkm_devstate *ds = (gkm_devstate *) calloc(1, sizeof(gkm_devstate));
    if (!ds) { gkm_set_error("out of memory"); return 1; }
    p->dev = ds;
    ds->ndev = g_nsel;
    const size_t n = (size_t) p->n, W = (size_t) p->Wmax;
    long long h2d = 0;
    for (int i = 0; i < ds->ndev; i++) {
        ds->dev[i] = g_sel[i];
        gkm_gpu *g = &g_gpu[g_sel[i]];
        if (gpu_prepare(g, g_sel[i], 0, 0)) return 1;
        gkm_image *im = &ds->img[i];
        if (pool_alloc(g, (void **) &im->planes, &im->planes_bytes, n * 3 * W * sizeof(uint32_t))) return 1;
        if (pool_alloc(g, (void **) &im->lens, &im->lens_bytes, n * sizeof(int32_t))) return 1;
        if (pool_alloc(g, (void **) &im->sqnorm, &im->sqnorm_bytes, n * sizeof(double))) return 1;
        CK(cudaMemcpyAsync(im->lens, p->len, n * sizeof(int32_t), cudaMemcpyHostToDevice, g->sc));
        h2d += (long long) (n * sizeof(int32_t));
        if (p->weighted && pool_alloc(g, (void **) &im->wend, &im->wend_bytes, n * 32 * W)) return 1;
        if (pack_host) {
            CK(cudaMemcpyAsync(im->planes, p->planes, n * 3 * W * sizeof(uint32_t), cudaMemcpyHostToDevice, g->sc));
            h2d += (long long) (n * 3 * W * sizeof(uint32_t));
            if (p->weighted) {
                CK(cudaMemcpyAsync(im->wend, p->wend, n * 32 * W, cudaMemcpyHostToDevice, g->sc));
                h2d += (long long) (n * 32 * W);
            }
        } else {
            /* one byte per base goes up (3 MB at 10k x 300 bp; the packed image of a weighted problem was 8.3 MB) and the
             * GPU packs: codes | offsets | weight table in one block */
            const size_t off_at = (p->arena_len + 15) & ~(size_t) 15, tab_at = off_at + n * sizeof(unsigned long long);
            if (pool_alloc(g, (void **) &im->codes, &im->codes_bytes, tab_at + sizeof(wtab))) return 1;
            CK(cudaMemcpyAsync(im->codes, p->arena, p->arena_len, cudaMemcpyHostToDevice, g->sc));
            CK(cudaMemcpyAsync(im->codes + off_at, p->off, n * sizeof(unsigned long long), cudaMemcpyHostToDevice, g->sc));
            if (p->weighted) CK(cudaMemcpyAsync(im->codes + tab_at, wtab, sizeof(wtab), cudaMemcpyHostToDevice, g->sc));
            h2d += (long long) (p->arena_len + n * sizeof(unsigned long long) + (p->weighted ? sizeof(wtab) : 0));
            const unsigned long long *d_off = (const unsigned long long *) (im->codes + off_at);
            if (p->weighted) gkm_pack_kernel<true><<<(unsigned) n, 128, 0, g->sc>>>(im->codes, d_off, im->lens, (int) W, p->param.L, im->codes + tab_at, im->planes, im->wend);
            else gkm_pack_kernel<false><<<(unsigned) n, 128, 0, g->sc>>>(im->codes, d_off, im->lens, (int) W, p->param.L, NULL, im->planes, NULL);
            CK(cudaGetLastError());
            p->stats.launches++;
        }
        /* sqnorm: Kraw(a,a) by the same kernel in diagonal mode, in blocks of 1024 rows */
        gkm_kparams kp;
        fill_kparams(p, im, GKM_MODE_DIAG, &kp);
        kp.sqnorm_out = im->sqnorm;
        /* the bit-sliced kernel covers the diagonal with one column of CTAs, 8 rows each: one launch for up to
         * 131 070 rows (grid.y <= 65 535 row tiles of at least 2 rows; it was 10 launches of 32 x 128 CTAs at 10k,
         * 1.8 ms of device time) */
        const int step = (pick_variant(p, GKM_MODE_DIAG) == GKM_KERNEL_DIAG) ? 131070 : 1024;
        for (int r = 0; r < p->n; r += step) {
            kp.row_begin = kp.col_begin = kp.row_base = kp.col_base = r;
            kp.row_end = kp.col_end = (r + step < p->n) ? r + step : p->n;
            if (launch_hist(p, im, g, kp, g->sc, NULL)) return 1;
            p->stats.launches++;
        }
        CK(cudaEventRecord(g->join, g->sc));            /* the second compute stream starts behind sqnorm too */
        CK(cudaStreamWaitEvent(g->sc2, g->join, 0));
    }
    p->have_sqnorm = 1;
    p->host_sqnorm = 0;
    if (need_host && fetch_sqnorm(p)) return 1;
    p->stats.upload_ms = now_ms() - t0;
    p->stats.h2d_bytes = h2d;
    p->stats.devices = ds->ndev;
    gkm_log(GKM_LOG_DEBUG, "uploaded %d sequences (%d words/plane) to %d GPU(s) in %.2f ms", p->n, p->Wmax, ds->ndev, p->stats.upload_ms);
    return 0;
}

extern "C" int gkm_dev_upload(gkmb200_problem *p)
{
    pthread_mutex_lock(&g_lock);
    p->stats.launches = 0;
    int r = upload_locked(p, 1);
    pthread_mutex_unlock(&g_lock);
    return r;
}

/* ------------------------------------------------------------------ */
/* compute: chunks -> GPUs -> pinned staging -> caller memory           */
/* ------------------------------------------------------------------ */
struct gkm_job {
    gkmb200_problem *p;
    const gkm_chunk *chunks;
    const int *owned;
    int nowned;
    int next;               /* atomic cursor into owned[] */
    int row0, col0, ncols, lower;
    double *out; long ld;   /* dense destination ... */
    double **rows;          /* ... or row pointers (absolute column index) */
    int32_t *hist;          /* dense histogram destination (tests) */
    int copy_threads;
};

struct gkm_scatter {
    const gkm_job *job;
    const gkm_chunk *c;
    const double *src;
    int t, nt;
};

static void *scatter_worker(void *arg)
{
    const gkm_scatter *s = (const gkm_scatter *) arg;
    const gkm_job *job = s->job;
    const gkm_chunk *c = s->c;
    const int width = c->col_end - c->col_begin;
    /* contiguous rows per thread, not interleaved ones: the destination rows are first-touch memory, and threads that
     * fault pages of the same 2 MB region in turn queue on its page-table lock (every chunk took 1.0-1.6 ms whatever
     * its size: 24 MB or 2.8 MB) */
    const int per = (c->row_end - c->row_begin + s->nt - 1) / s->nt;
    const int r_lo = c->row_begin + s->t * per;
    const int r_hi = r_lo + per < c->row_end ? r_lo + per : c->row_end;
    for (int r = r_lo; r < r_hi; r++) {
        int hi = c->col_end;
        if (job->lower && hi > r) hi = r;
        const int ncopy = hi - c->col_begin;
        double *dst = job->rows ? job->rows[r] + c->col_begin
                                : job->out + (size_t) (r - job->row0) * (size_t) job->ld + (size_t) (c->col_begin - job->col0);
        if (ncopy > 0) memcpy(dst, s->src + (size_t) (r - c->row_begin) * (size_t) width, (size_t) ncopy * sizeof(double));
        if (job->lower && r >= job->col0 && r < job->col0 + job->ncols) {
            if (job->rows) job->rows[r][r] = 1.0;                 /* gkmkern_pylib.c:219-221 */
            else job->out[(size_t) (r - job->row0) * (size_t) job->ld + (size_t) (r - job->col0)] = 1.0;
        }
    }
    return NULL;
}

/* The scatter team of one device thread: created once per compute call and joined before it returns (no thread of
 * the library outlives gkm_main_pywrapper, SURVEY.md 8b).  One pthread_create per helper and CHUNK was 0.5 ms of
 * pure overhead per chunk with 16 threads (25-35 chunks per call: a third of the time spent "scattering"). */
struct gkm_team {
    int nthreads;          /* helpers + the device thread itself */
    int pending, quit;
    gkm_scatter task;      /* job, chunk, source of the task in progress (t is per helper) */
    sem_t start[64];       /* one per helper: a broadcast on one condition variable woke them one after the other
                            * through its mutex, 0.7 ms per chunk with 15 helpers */
    sem_t done;
    pthread_t th[64];
    int started[64];
    struct gkm_team_arg { gkm_team *team; int t; } arg[64];
};

static void *team_worker(void *a)
{
    gkm_team *tm = ((gkm_team::gkm_team_arg *) a)->team;
    const int t = ((gkm_team::gkm_team_arg *) a)->t;
    for (;;) {
        while (sem_wait(&tm->start[t]) != 0) { /* EINTR */ }
        if (__atomic_load_n(&tm->quit, __ATOMIC_ACQUIRE)) return NULL;
        gkm_scatter sc = tm->task;
        sc.t = t;
        if (t < sc.nt) scatter_worker(&sc);
        if (__atomic_sub_fetch(&tm->pending, 1, __ATOMIC_ACQ_REL) == 0) sem_post(&tm->done);
    }
}

static void team_start(gkm_team *tm, int nthreads)
{
    memset(tm, 0, sizeof(*tm));
    sem_init(&tm->done, 0, 0);
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 64) nthreads = 64;
    tm->nthreads = 1;
    for (int t = 1; t < nthreads; t++) {
        const int id = tm->nthreads;
        sem_init(&tm->start[id], 0, 0);
        tm->arg[id].team = tm; tm->arg[id].t = id;
        tm->started[id] = (pthread_create(&tm->th[id], NULL, team_worker, &tm->arg[id]) == 0);
        if (tm->started[id]) tm->nthreads++; /* like the reference: a thread that cannot start just is not there */
        else sem_destroy(&tm->start[id]);
    }
}

static void team_stop(gkm_team *tm)
{
    __atomic_store_n(&tm->quit, 1, __ATOMIC_RELEASE);
    for (int t = 1; t < tm->nthreads; t++) sem_post(&tm->start[t]);
    for (int t = 1; t < tm->nthreads; t++) { pthread_join(tm->th[t], NULL); sem_destroy(&tm->start[t]); }
    sem_destroy(&tm->done);
}

static void scatter_chunk(gkm_team *tm, const gkm_job *job, const gkm_chunk *c, const double *src)
{
    int nt = tm->nthreads;
    if (nt > c->row_end - c->row_begin) nt = c->row_end - c->row_begin;
    if (nt < 1) nt = 1;
    gkm_scatter sc;
    sc.job = job; sc.c = c; sc.src = src; sc.t = 0; sc.nt = nt;
    if (nt > 1) {
        tm->task = sc;
        __atomic_store_n(&tm->pending, tm->nthreads - 1, __ATOMIC_RELEASE);
        for (int t = 1; t < tm->nthreads; t++) sem_post(&tm->start[t]);
    }
    scatter_worker(&sc);
    if (nt > 1) while (sem_wait(&tm->done) != 0) { /* EINTR */ }
}

struct gkm_devthread {
    gkm_job *job;
    int slot;          /* index into devstate */
    double kernel_ms;
    double scatter_ms, wait_ms; /* host time of this device thread spent copying into caller rows / waiting for the GPU */
    long long launches, d2h_bytes, entries;
    int variant;
};

static int dev_issue(gkm_devthread *dt, gkm_gpu *g, const gkm_image *im, const gkm_chunk *c, int buf, int32_t *d_hist)
{
    gkm_job *job = dt->job;
    gkm_kparams kp;
    fill_kparams(job->p, im, job->lower ? GKM_MODE_LOWER : GKM_MODE_RECT, &kp);
    kp.row_begin = kp.row_base = c->row_begin;
    kp.row_end = c->row_end;
    kp.col_begin = kp.col_base = c->col_begin;
    kp.col_end = c->col_end;
    const int width = c->col_end - c->col_begin;
    kp.out = (double *) g->d_band[buf];
    kp.ld = width;
    kp.hist = d_hist;
    kp.hist_cols = width;
    cudaStream_t st = (buf & 1) ? g->sc2 : g->sc;
    CK(cudaEventRecord(g->k0[buf], st));
    const long long k_before = g->nkernels;
    if (launch_hist(job->p, im, g, kp, st, &dt->variant)) return 1;
    dt->launches += g->nkernels - k_before; /* kernels, not chunks: the index variant launches one per column block */
    CK(cudaEventRecord(g->k1[buf], st));
    CK(cudaStreamWaitEvent(g->sx, g->k1[buf], 0));
    const size_t bytes = (size_t) (c->row_end - c->row_begin) * (size_t) width * sizeof(double);
    if (bytes) CK(cudaMemcpyAsync(g->h_stage[buf], g->d_band[buf], bytes, cudaMemcpyDeviceToHost, g->sx));
    CK(cudaEventRecord(g->cdone[buf], g->sx));
    dt->d2h_bytes += (long long) bytes;
    dt->entries += c->entries;
    return 0;
}

static int dev_thread_run(gkm_devthread *dt, gkm_team *team_p)
{
    gkm_job *job = dt->job;
    gkmb200_problem *p = job->p;
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[dt->slot]];
    const gkm_image *im = &ds->img[dt->slot];
    size_t maxbytes = 0, maxhist = 0;
    for (int i = 0; i < job->nowned; i++) {
        const gkm_chunk *c = &job->chunks[job->owned[i]];
        size_t cells = (size_t) (c->row_end - c->row_begin) * (size_t) (c->col_end - c->col_begin);
        if (cells * 8 > maxbytes) maxbytes = cells * 8;
        if (cells * 4 * (size_t) p->nbins > maxhist) maxhist = cells * 4 * (size_t) p->nbins;
    }
    if (gpu_prepare(g, ds->dev[dt->slot], maxbytes, maxbytes)) return 1;
    gkm_team &team = *team_p;
    int32_t *d_hist = NULL, *h_hist = NULL;
    if (job->hist) {
        CK(dev_malloc(g, (void **) &d_hist, maxhist ? maxhist : 4));
        h_hist = (int32_t *) malloc(maxhist ? maxhist : 4);
        if (!h_hist) { cudaFree(d_hist); gkm_set_error("out of memory"); return 1; }
    }
    /* up to `depth` chunks are in flight: slot s holds chunk inslot[s]; the oldest is retired (D2H done ->
     * scattered into the caller's rows) while the GPU works on the younger ones.  Histogram dumps (tests)
     * run one chunk at a time: they share a single device buffer. */
    const int depth = job->hist ? 1 : GKM_NBUF;
    int inslot[GKM_NBUF];
    int head = 0, inflight = 0, rc = 0;
    const double tb0 = now_ms();
    double t_wait = 0.0, t_scatter = 0.0, t_issue = 0.0, t_lastsync = tb0;
    if (cudaEventRecord(g->span0, g->sc) != cudaSuccess) { gkm_set_error("CUDA: event record failed"); return 1; }
    while (!rc && inflight < depth) {
        const int nxt = __atomic_fetch_add(&job->next, 1, __ATOMIC_RELAXED);
        if (nxt >= job->nowned) break;
        const int s = (head + inflight) % GKM_NBUF;
        inslot[s] = nxt;
        rc = dev_issue(dt, g, im, &job->chunks[job->owned[nxt]], s, d_hist);
        inflight++;
    }
    t_issue += now_ms() - tb0;
    while (!rc && inflight > 0) {
        const int s = head % GKM_NBUF;
        const gkm_chunk *c = &job->chunks[job->owned[inslot[s]]];
        const double tw0 = now_ms();
        if (cudaEventSynchronize(g->cdone[s]) != cudaSuccess) {
            gkm_set_error("CUDA: kernel or copy failed: %s", cudaGetErrorString(cudaGetLastError()));
            rc = 1;
            break;
        }
        float ms = 0.f;
        /* device time of the call so far: first kernel start -> end of this chunk's kernel (chunks overlap) */
        if (cudaEventElapsedTime(&ms, g->span0, g->k1[s]) == cudaSuccess && ms > dt->kernel_ms) dt->kernel_ms = ms;
        t_lastsync = now_ms();
        t_wait += t_lastsync - tw0;
        if (job->out || job->rows) scatter_chunk(&team, job, c, (const double *) g->h_stage[s]);
        t_scatter += now_ms() - t_lastsync;
        gkm_log(GKM_LOG_TRACE, "chunk rows [%d, %d) x %d columns: waited %.3f ms, scattered in %.3f ms", c->row_begin, c->row_end,
                c->col_end - c->col_begin, t_lastsync - tw0, now_ms() - t_lastsync);
        if (job->hist) {
            const int width = c->col_end - c->col_begin, nb = p->nbins;
            const size_t cells = (size_t) (c->row_end - c->row_begin) * (size_t) width;
            if (cudaMemcpy(h_hist, d_hist, cells * 4 * (size_t) nb, cudaMemcpyDeviceToHost) != cudaSuccess) {
                gkm_set_error("CUDA: histogram copy failed: %s", cudaGetErrorString(cudaGetLastError()));
                rc = 1;
                break;
            }
            for (int r = c->row_begin; r < c->row_end; r++) {
                int hi = c->col_end;
                if (job->lower && hi > r) hi = r;
                for (int cc = c->col_begin; cc < hi; cc++)
                    memcpy(job->hist + ((size_t) (r - job->row0) * (size_t) job->ncols + (size_t) (cc - job->col0)) * (size_t) nb,
                           h_hist + ((size_t) (r - c->row_begin) * (size_t) width + (size_t) (cc - c->col_begin)) * (size_t) nb,
                           (size_t) nb * 4);
            }
        }
        head++;
        inflight--;
        const int nxt = __atomic_fetch_add(&job->next, 1, __ATOMIC_RELAXED);
        if (nxt < job->nowned) {
            const int ns = (head + inflight) % GKM_NBUF;
            inslot[ns] = nxt;
            const double ti0 = now_ms();
            rc = dev_issue(dt, g, im, &job->chunks[job->owned[nxt]], ns, d_hist);
            t_issue += now_ms() - ti0;
            inflight++;
        }
    }
    dt->scatter_ms = t_scatter; dt->wait_ms = t_wait;
    gkm_log(GKM_LOG_DEBUG, "GPU %d: %.2f ms in all: issue %.2f, waiting for chunks %.2f, scatter %.2f = %.1f GB/s with %d threads "
            "(after the last chunk arrived: %.2f)",
            ds->dev[dt->slot], now_ms() - tb0, t_issue, t_wait, t_scatter, t_scatter > 0 ? (double) dt->entries * 8e-6 / t_scatter : 0.0,
            team.nthreads, now_ms() - t_lastsync);
    if (rc) cudaDeviceSynchronize();
    if (d_hist) cudaFree(d_hist);
    free(h_hist);
    return rc;
}

static long long plan_budget(const gkmb200_problem *p, long long total_cells, int ndev)
{
    long long cap = (long long) gkm_opt_chunk_mb() << 20;
    long long want = total_cells * 8 / (16LL * ndev * p->shard_world);
    if (want < (4LL << 20)) want = 4LL << 20;
    return want < cap ? want : cap;
}

/* The chunks of rows [row0, +nrows) x columns [col0, +ncols) in *out (malloc'd; the caller frees it), for nshare GPUs.
 * The index variant costs the same for every row, so its chunks are whole waves of rows, at most 4 of them; the
 * others take 16-row tiles, at most 65 520 rows (grid.y <= 65 535 row tiles).  Returns the count, or -1. */
static int plan_chunks(const gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower, int nshare, gkm_chunk **out)
{
    const int by_rows = (p->dev->variant == GKM_KERNEL_INDEX);
    const int maxc = nrows / 16 + 2;
    const long long total_cells = (long long) nrows * ncols / (lower ? 2 : 1);
    *out = (gkm_chunk *) malloc(sizeof(gkm_chunk) * (size_t) maxc);
    const int nchunks = *out ? gkm_plan_chunks_rows(row0, nrows, col0, ncols, lower, by_rows ? GKM_WAVE_ROWS : 16, plan_budget(p, total_cells, nshare),
                                                    by_rows ? 4 * GKM_WAVE_ROWS : 65520, *out, maxc) : -1;
    if (nchunks < 0) gkm_set_error("chunk planning failed");
    return nchunks;
}

/* Host threads that scatter finished chunks into the caller's rows.  The reference's `nthreads` (default 1 in
 * bin/gkmqc.py:107,162) is its number of COMPUTE threads; here the only host work that scales with it is the copy-out,
 * which is first-touch page faults of the caller's fresh matrix (100 000 of them at 10k, 2.4 million at 50k; ~2 us
 * each on this host: tools/pagefault_probe.c).  So the request is a lower bound and the library uses the cores this
 * process may run on (its affinity mask: cgroup-, slurm- and taskset-aware).  Round 1 capped that at 16; the 8-GPU box
 * has 32 cores and the cap left half of them idle (VERDICT r1).  GKM_COPY_THREADS overrides. */
#include <sched.h>
static int host_cores(void)
{
    int avail = 0;
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0) avail = CPU_COUNT(&set);
    if (avail < 1) avail = (int) sysconf(_SC_NPROCESSORS_ONLN);
    return avail < 1 ? 1 : avail;
}

/* threads of one process that shares the box with `world - 1` others (one process per GPU) */
extern "C" int gkm_copy_threads_shared(int requested, int world)
{
    const char *e = getenv("GKM_COPY_THREADS");
    if (e && atoi(e) > 0) return atoi(e) > 64 ? 64 : atoi(e);
    if (world < 1) world = 1;
    int n = host_cores() / world;
    if (n < requested) n = requested;
    if (n < 1) n = 1;
    return n > 64 ? 64 : n;
}

extern "C" int gkm_copy_threads(int requested) { return gkm_copy_threads_shared(requested, 1); }

extern "C" int gkm_dev_compute(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower,
                               double *out, long ld, double **rows, int32_t *hist, int copy_threads)
{
    if (!p) { gkm_set_error("null problem"); return 1; }
    if (row0 < 0 || col0 < 0 || nrows < 0 || ncols < 0 || row0 + nrows > p->n || col0 + ncols > p->n) {
        gkm_set_error("block [%d,+%d) x [%d,+%d) outside the problem (n=%d)", row0, nrows, col0, ncols, p->n);
        return 1;
    }
    /* the ranks of a sharded run (one process per GPU) share the cores of the box */
    copy_threads = gkm_copy_threads_shared(copy_threads, p->shard_world);
    pthread_mutex_lock(&g_lock);
    const double t0 = now_ms();
    p->stats.launches = 0;
    /* Chunks are issued in ascending row order.  Round 1 issued the widest rows first so that the call ends on the smallest
     * copy; that saves < 1 ms at 10k and costs the weighted kernel types dearly (wgkm 10k x 300 bp: device span 59.0
     * against 47.3 ms; gkmQC's default, 600-bp windows: 312 against 237 ms; unit weights: equal) --
     * profiles/r2_chunk_order_carveout_ab.txt. */
    int rc = upload_locked(p, 0);
    const double t_up = now_ms();
    if (!rc) rc = choose_variant(p, row0, nrows, col0, ncols, lower);
    const double t_var = now_ms();
    gkm_chunk *chunks = NULL;
    int *owned = NULL;
    if (!rc) {
        gkm_devstate *ds = p->dev;
        const int nchunks = plan_chunks(p, row0, nrows, col0, ncols, lower, ds->ndev, &chunks);
        if (nchunks < 0) rc = 1;
        else if (!(owned = (int *) malloc(sizeof(int) * (size_t) (nchunks + 1)))) { gkm_set_error("out of memory"); rc = 1; }
        if (!rc) {
            gkm_job job;
            memset(&job, 0, sizeof(job));
            job.p = p; job.chunks = chunks; job.owned = owned;
            for (int c = 0; c < nchunks; c++)
                if (gkm_chunk_owner(c, nchunks, p->shard_world) == p->shard_rank) owned[job.nowned++] = c;
            job.row0 = row0; job.col0 = col0; job.ncols = ncols; job.lower = lower;
            job.out = out; job.ld = ld; job.rows = rows; job.hist = hist;
            /* the host threads that scatter finished chunks are shared by the GPUs of the call: each device thread
             * leads a team of its share of them (different chunks, so different 2 MB regions of the destination) */
            job.copy_threads = copy_threads / ds->ndev > 1 ? copy_threads / ds->ndev : 1;
            gkm_devthread dts[GKM_MAX_DEV];
            memset(dts, 0, sizeof(dts));
            for (int i = 0; i < ds->ndev; i++) { dts[i].job = &job; dts[i].slot = i; }
            rc = for_each_gpu(ds, [&](int slot) {
                gkm_team team;
                team_start(&team, (out || rows) ? job.copy_threads : 1);
                const int r = dev_thread_run(&dts[slot], &team);
                team_stop(&team);
                return r;
            });
            p->stats.kernel_ms = 0; p->stats.d2h_bytes = 0; p->stats.entries = 0;
            p->stats.scatter_ms = 0; p->stats.wait_ms = 0;
            p->stats.copy_threads = job.copy_threads * ds->ndev;
            for (int i = 0; i < ds->ndev; i++) {
                if (dts[i].scatter_ms > p->stats.scatter_ms) p->stats.scatter_ms = (float) dts[i].scatter_ms;
                if (dts[i].wait_ms > p->stats.wait_ms) p->stats.wait_ms = (float) dts[i].wait_ms;
                if (dts[i].kernel_ms > p->stats.kernel_ms) p->stats.kernel_ms = dts[i].kernel_ms;
                p->stats.launches += dts[i].launches;
                p->stats.d2h_bytes += dts[i].d2h_bytes;
                p->stats.entries += dts[i].entries;
                if (dts[i].variant) p->stats.kernel_variant = dts[i].variant;
            }
            p->stats.devices = ds->ndev;
            p->stats.shard_rank = p->shard_rank; p->stats.shard_world = p->shard_world;
        }
    }
    free(chunks);
    free(owned);
    p->stats.wall_ms = now_ms() - t0;
    gkm_log(GKM_LOG_DEBUG, "compute: pack+upload %.2f ms, variant+index %.2f ms, chunks %.2f ms (device span %.2f ms)",
            t_up - t0, t_var - t_up, now_ms() - t_var, p->stats.kernel_ms);
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* ------------------------------------------------------------------ */
/* fused decision values (SURVEY.md 8f/f1)                              */
/* ------------------------------------------------------------------ */
/* one GPU's slice of the test rows: out[r] = bias + sum_c alpha[c] K(row0 + r, col0 + c) */
static int decision_slice(gkmb200_problem *p, int slot, int row0, int nrows, int col0, int ncols, const double *alpha, double bias, double *out)
{
    if (nrows <= 0) return 0;
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[slot]];
    double *d_alpha = NULL, *d_dec = NULL;
    int rc = 0;
    do {
        if (cudaMalloc(&d_alpha, sizeof(double) * (size_t) (ncols ? ncols : 1)) != cudaSuccess) { rc = 1; break; }
        if (cudaMalloc(&d_dec, sizeof(double) * (size_t) nrows) != cudaSuccess) { rc = 1; break; }
        if (cudaMemcpyAsync(d_alpha, alpha, sizeof(double) * (size_t) ncols, cudaMemcpyHostToDevice, g->sc) != cudaSuccess) { rc = 1; break; }
        if (cudaMemsetAsync(d_dec, 0, sizeof(double) * (size_t) nrows, g->sc) != cudaSuccess) { rc = 1; break; }
        /* the second compute stream must see alpha and the zeroed accumulator too */
        if (cudaEventRecord(g->join, g->sc) != cudaSuccess || cudaStreamWaitEvent(g->sc2, g->join, 0) != cudaSuccess) { rc = 1; break; }
    } while (0);
    if (rc) gkm_set_error("CUDA: decision-value buffers: %s", cudaGetErrorString(cudaGetLastError()));
    gkm_kparams kp;
    fill_kparams(p, &ds->img[slot], GKM_MODE_RECT, &kp);
    kp.alpha = d_alpha; kp.decision = d_dec;
    kp.col_begin = kp.col_base = col0; kp.col_end = col0 + ncols;
    kp.row_base = row0;
    int launches = 0;
    /* index variant: whole waves of rows per launch, and a bounded cold-bin scratch */
    const int rows_per_launch = (ds->variant == GKM_KERNEL_INDEX) ? 16 * GKM_WAVE_ROWS : 8192;
    for (int r = row0; !rc && r < row0 + nrows; r += rows_per_launch) {
        kp.row_begin = r;
        kp.row_end = (r + rows_per_launch < row0 + nrows) ? r + rows_per_launch : row0 + nrows;
        rc = launch_hist(p, &ds->img[slot], g, kp, (launches++ & 1) ? g->sc2 : g->sc, NULL);
    }
    if (!rc) {
        rc = (cudaStreamSynchronize(g->sc2) != cudaSuccess) ||
             (cudaMemcpyAsync(out, d_dec, sizeof(double) * (size_t) nrows, cudaMemcpyDeviceToHost, g->sc) != cudaSuccess) ||
             (cudaStreamSynchronize(g->sc) != cudaSuccess);
        if (rc) gkm_set_error("CUDA: decision values failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!rc) for (int i = 0; i < nrows; i++) out[i] += bias;
    cudaFree(d_alpha);
    cudaFree(d_dec);
    return rc;
}

/* the test rows are cut into one contiguous slice per selected GPU; every GPU holds all columns (SVs) */
extern "C" int gkm_dev_decision(gkmb200_problem *p, int row0, int nrows, int col0, int ncols,
                                const double *alpha, double bias, double *out)
{
    if (!p || !alpha || !out) { gkm_set_error("null argument"); return 1; }
    if (row0 < 0 || col0 < 0 || nrows < 0 || ncols < 0 || row0 + nrows > p->n || col0 + ncols > p->n) {
        gkm_set_error("block outside the problem");
        return 1;
    }
    pthread_mutex_lock(&g_lock);
    int rc = upload_locked(p, 0);
    if (!rc) rc = choose_variant(p, row0, nrows, col0, ncols, 0);
    if (!rc) {
        const int nd = p->dev->ndev, per = ((nrows + nd - 1) / nd + 7) & ~7;
        rc = for_each_gpu(p->dev, [&](int slot) {
            int b = slot * per, e = b + per;
            if (b > nrows) b = nrows;
            if (e > nrows) e = nrows;
            return decision_slice(p, slot, row0 + b, e - b, col0, ncols, alpha, bias, out + b);
        });
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* ------------------------------------------------------------------ */
/* the consumer: cross-validated C-SVC on the resident matrix (8f/f4)   */
/* ------------------------------------------------------------------ */
/* GPUs of the call that compute chunks of the resident matrix.  The matrix lives on the first selected GPU; the others
 * may help only if they can store into its memory -- peer access over NVLink / NVSwitch, enabled once per process and
 * pair.  All of them or one: on boxes whose GPUs are not peers the owner does the whole pass.  Leaves another device
 * current. */
static int resident_sharers(const gkm_devstate *ds)
{
    static signed char peer_ok[GKM_MAX_DEV][GKM_MAX_DEV]; /* [writer][owner]: 0 not asked yet, 1 yes, -1 no */
    if (ds->ndev < 2) return 1;
    const int owner = ds->dev[0];
    for (int i = 1; i < ds->ndev; i++) {
        const int d = ds->dev[i];
        if (d == owner) return 1;
        if (peer_ok[d][owner] == 0) {
            int can = 0;
            peer_ok[d][owner] = -1;
            if (cudaDeviceCanAccessPeer(&can, d, owner) == cudaSuccess && can && cudaSetDevice(d) == cudaSuccess) {
                const cudaError_t pe = cudaDeviceEnablePeerAccess(owner, 0);
                if (pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled) peer_ok[d][owner] = 1;
            }
            cudaGetLastError();
            gkm_log(GKM_LOG_DEBUG, "GPU %d %s store into the memory of GPU %d", d, peer_ok[d][owner] > 0 ? "may" : "cannot", owner);
        }
        if (peer_ok[d][owner] < 0) return 1;
    }
    return ds->ndev;
}

/* the resident N x full_ld matrix of the first selected GPU (current device must be g's) */
static int ensure_full(gkm_gpu *g, gkm_image *im, int n)
{
    if (im->full) return 0;
    im->full_ld = ((size_t) n + 15) & ~(size_t) 15;
    CK(dev_malloc(g, (void **) &im->full, im->full_ld * (size_t) n * sizeof(double)));
    return 0;
}

/* Queues the chunks of the lower triangle that shard rank/world owns into im->full of the first selected GPU: chunk c
 * runs on GPU c % nshare, on sc or sc2 by that GPU's own count of issued chunks.  Adds the kernels launched and the
 * entries to *kernels / *entries.  With nshare > 1 it leaves another device current. */
static int lower_pass(gkmb200_problem *p, const gkm_chunk *chunks, int nchunks, int nshare, int rank, int world,
                      long long *kernels, long long *entries, int *variant_out)
{
    gkm_devstate *ds = p->dev;
    int issued[GKM_MAX_DEV] = { 0 };
    for (int c = 0; c < nchunks; c++) {
        if (gkm_chunk_owner(c, nchunks, world) != rank) continue;
        const int s = c % nshare;
        gkm_gpu *gs = &g_gpu[ds->dev[s]];
        if (nshare > 1 && cudaSetDevice(ds->dev[s]) != cudaSuccess) { gkm_set_error("CUDA: cannot select device %d", ds->dev[s]); return 1; }
        gkm_kparams kp;
        fill_kparams(p, &ds->img[s], GKM_MODE_LOWER, &kp);
        kp.row_begin = chunks[c].row_begin; kp.row_end = chunks[c].row_end;
        kp.col_begin = chunks[c].col_begin; kp.col_end = chunks[c].col_end;
        kp.out = ds->img[0].full; kp.ld = (long long) ds->img[0].full_ld; /* the owner's block, whichever GPU runs the chunk */
        const long long k_before = gs->nkernels;
        const int rc = launch_hist(p, &ds->img[s], gs, kp, (issued[s]++ & 1) ? gs->sc2 : gs->sc, variant_out);
        *kernels += gs->nkernels - k_before; /* kernels, not chunks: the index variant launches one per column block */
        *entries += chunks[c].entries;
        if (rc) return 1;
    }
    return 0;
}

/* One pass of the lower triangle into im->full on the first selected GPU, then mirrored there: the matrix never leaves
 * the devices.  With several GPUs in the call (one process, GKM_DEVICES) the chunks go round-robin over all of them
 * and every GPU writes its entries straight into the owner's matrix -- the epilogue's streaming stores travel over
 * NVLink while the next rows are being counted, so there is no gather step and no staging copy (SURVEY.md 8f/f4:
 * "NVSwitch allgather of tiles if sharded"; here the tiles are never anywhere else).  Each GPU reads its own replica
 * of the sequence image, the sqnorms and -- index variant -- its own slot tables (choose_variant built them). */
static int resident_symmetric(gkmb200_problem *p)
{
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[0]];
    gkm_image *im = &ds->img[0];
    const int n = p->n;
    if (im->full && im->full_sym) return 0;
    const int nshare = resident_sharers(ds);
    CK(cudaSetDevice(ds->dev[0]));
    if (ensure_full(g, im, n)) return 1;
    gkm_chunk *chunks = NULL;
    const int nchunks = plan_chunks(p, 0, n, 0, n, 1, nshare, &chunks);
    long long kernels = 0, entries = 0;
    int rc = nchunks < 0 || lower_pass(p, chunks, nchunks, nshare, 0, 1, &kernels, &entries, NULL);
    free(chunks);
    /* the stores of the other GPUs have landed once their streams have drained; the owner mirrors the triangle after that */
    for (int s = 1; s < nshare; s++) {
        gkm_gpu *gs = &g_gpu[ds->dev[s]];
        if (cudaSetDevice(ds->dev[s]) != cudaSuccess || cudaStreamSynchronize(gs->sc) != cudaSuccess || cudaStreamSynchronize(gs->sc2) != cudaSuccess) {
            if (!rc) gkm_set_error("CUDA: resident matrix, GPU %d: %s", ds->dev[s], cudaGetErrorString(cudaGetLastError()));
            rc = 1;
        }
    }
    CK(cudaSetDevice(ds->dev[0]));
    if (rc) return 1;
    CK(cudaEventRecord(g->join, g->sc2));
    CK(cudaStreamWaitEvent(g->sc, g->join, 0));
    if (gkm_svm_symmetrize(im->full, (long long) im->full_ld, n, g->sc)) { gkm_set_error("CUDA: symmetrize kernel failed"); return 1; }
    im->full_sym = 1;
    p->stats.launches += kernels + 1;
    p->stats.devices = nshare;
    return 0;
}

/* rows [row0, row0 + nrows) of the resident symmetric matrix, computed on first use: out[(r - row0) * ld + c] = K(r, c)
 * for every c < n, unit diagonal.  nrows = 0 only makes the matrix resident (and waits for it). */
extern "C" int gkmb200_resident_rows(gkmb200_problem *p, int row0, int nrows, double *out, long ld)
{
    if (!p) { gkm_set_error("null problem"); return 1; }
    if (row0 < 0 || nrows < 0 || row0 + nrows > p->n || (nrows > 0 && (!out || ld < p->n))) { gkm_set_error("rows [%d,+%d) outside the matrix (n=%d) or ld < n", row0, nrows, p->n); return 1; }
    pthread_mutex_lock(&g_lock);
    const double t0 = now_ms();
    p->stats.launches = 0;
    int rc = upload_locked(p, 0);
    if (!rc) rc = choose_variant(p, 0, p->n, 0, p->n, 1);
    if (!rc) rc = resident_symmetric(p);
    if (!rc) {
        gkm_devstate *ds = p->dev;
        gkm_gpu *g = &g_gpu[ds->dev[0]];
        const gkm_image *im = &ds->img[0];
        cudaError_t e = cudaSetDevice(ds->dev[0]);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc);
        if (e == cudaSuccess && nrows > 0)
            e = cudaMemcpy2D(out, (size_t) ld * sizeof(double), im->full + (size_t) row0 * im->full_ld, im->full_ld * sizeof(double),
                             (size_t) p->n * sizeof(double), (size_t) nrows, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { gkm_set_error("CUDA: resident matrix read-back: %s", cudaGetErrorString(e)); rc = 1; }
        p->stats.kernel_variant = ds->variant;
        p->stats.wall_ms = now_ms() - t0;
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

extern "C" int gkm_dev_svm_cv(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                              const int *train_idx, const signed char *train_y, const int *test_idx,
                              double C, double eps, int max_iter, double *scores, gkmb200_svm_fit *fits, double *alpha)
{
    if (ntasks < 0 || (ntasks > 0 && (!tasks || !train_idx || !train_y || !test_idx))) { gkm_set_error("null argument"); return 1; }
    if (!(C > 0.0) || !(eps > 0.0)) { gkm_set_error("svm: C and eps must be positive"); return 1; }
    pthread_mutex_lock(&g_lock);
    int rc = 0;
    const double t0 = now_ms();
    if (!kmat) {
        if (!p) { gkm_set_error("svm: neither a matrix nor a problem"); rc = 1; }
        if (!rc && n != p->n) { gkm_set_error("svm: n = %d but the problem holds %d sequences", n, p->n); rc = 1; }
        if (!rc) rc = upload_locked(p, 0);
        if (!rc) rc = choose_variant(p, 0, p->n, 0, p->n, 1);
        if (!rc) rc = resident_symmetric(p);
        if (!rc) {
            gkm_devstate *ds = p->dev;
            gkm_gpu *g = &g_gpu[ds->dev[0]];
            rc = gkm_svm_run(ds->img[0].full, (long long) ds->img[0].full_ld, n, ntasks, tasks, train_idx, train_y, test_idx,
                             C, eps, max_iter, scores, fits, alpha, g->sc);
            p->stats.launches += 3;
            p->stats.wall_ms = now_ms() - t0;
        }
    } else {
        if (n < 2 || ld < n) { gkm_set_error("svm: bad matrix shape"); rc = 1; }
        if (!rc) rc = ensure_selected();
        double *d_K = NULL;
        if (!rc) {
            gkm_gpu *g = &g_gpu[g_sel[0]];
            rc = gpu_prepare(g, g_sel[0], 0, 0);
            if (!rc && dev_malloc(g, (void **) &d_K, sizeof(double) * (size_t) n * (size_t) n) != cudaSuccess) { gkm_set_error("CUDA: svm matrix: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            if (!rc && cudaMemcpy2DAsync(d_K, sizeof(double) * (size_t) n, kmat, sizeof(double) * (size_t) ld, sizeof(double) * (size_t) n, (size_t) n,
                                         cudaMemcpyHostToDevice, g->sc) != cudaSuccess) { gkm_set_error("CUDA: svm matrix upload: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            if (!rc) rc = gkm_svm_run(d_K, (long long) n, n, ntasks, tasks, train_idx, train_y, test_idx, C, eps, max_iter, scores, fits, alpha, g->sc);
            cudaFree(d_K);
        }
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* ------------------------------------------------------------------ */
/* measurement                                                          */
/* ------------------------------------------------------------------ */
extern "C" int gkm_dev_bench_lower(gkmb200_problem *p, int steps, int warmup, int flush_l2, double *ms_each)
{
    if (!p || steps < 1 || !ms_each) { gkm_set_error("bad bench arguments"); return 1; }
    pthread_mutex_lock(&g_lock);
    int rc = upload_locked(p, 0);
    if (!rc) rc = choose_variant(p, 0, p->n, 0, p->n, 1);
    gkm_chunk *chunks = NULL;
    if (!rc) {
        gkm_devstate *ds = p->dev;
        gkm_gpu *g = &g_gpu[ds->dev[0]];
        gkm_image *im = &ds->img[0];
        if (cudaSetDevice(ds->dev[0]) != cudaSuccess || ensure_full(g, im, p->n) ||
            (flush_l2 && !g->d_flush && cudaMalloc(&g->d_flush, GKM_FLUSH_BYTES) != cudaSuccess)) {
            gkm_set_error("CUDA: bench buffers: %s", cudaGetErrorString(cudaGetLastError()));
            rc = 1;
        }
        const int nchunks = rc ? -1 : plan_chunks(p, 0, p->n, 0, p->n, 1, 1, &chunks);
        if (nchunks < 0) rc = 1;
        cudaEvent_t e0 = NULL, e1 = NULL;
        if (!rc) rc = (cudaEventCreate(&e0) != cudaSuccess) || (cudaEventCreate(&e1) != cudaSuccess);
        long long launches = 0, entries = 0;
        int variant = 0;
        im->full_sym = 0; /* the pass writes the lower triangle only: the consumer mirrors it again */
        for (int it = 0; !rc && it < warmup + steps; it++) {
            if (flush_l2) cudaMemsetAsync(g->d_flush, it & 0xff, GKM_FLUSH_BYTES, g->sc);
            cudaEventRecord(e0, g->sc);
            cudaStreamWaitEvent(g->sc2, e0, 0);
            launches = 0; entries = 0;
            rc = lower_pass(p, chunks, nchunks, 1, p->shard_rank, p->shard_world, &launches, &entries, &variant);
            cudaEventRecord(g->join, g->sc2);
            cudaStreamWaitEvent(g->sc, g->join, 0);
            cudaEventRecord(e1, g->sc);
            if (!rc && cudaEventSynchronize(e1) != cudaSuccess) {
                gkm_set_error("CUDA: bench pass failed: %s", cudaGetErrorString(cudaGetLastError()));
                rc = 1;
            }
            float ms = 0.f;
            if (!rc) cudaEventElapsedTime(&ms, e0, e1);
            if (it >= warmup) ms_each[it - warmup] = ms;
        }
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
        p->stats.launches = launches;
        p->stats.entries = entries;
        p->stats.kernel_variant = variant;
        p->stats.devices = 1;
        p->stats.d2h_bytes = 0;
    }
    free(chunks);
    pthread_mutex_unlock(&g_lock);
    return rc;
}

/* ---- issue-rate micro-benchmarks: the denominators of the integer roofline ---- */
template <int OP>
__global__ void __launch_bounds__(256) gkm_mb_kernel(uint32_t *out, int iters, uint32_t seed)
{
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = seed * (uint32_t) (threadIdx.x + 1) + (uint32_t) i * 0x9E3779B9u;
    uint32_t y = seed ^ 0x5bd1e995u, z = seed + (uint32_t) blockIdx.x;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (OP == 0) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                if (OP == 1) asm volatile("shf.r.wrap.b32 %0, %0, %1, 7;" : "+r"(x[i]) : "r"(y));
                if (OP == 2) asm volatile("popc.b32 %0, %0;" : "+r"(x[i]));
                if (OP == 3) asm volatile("add.u32 %0, %0, %1;" : "+r"(x[i]) : "r"(y));
                if (OP == 4) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z));
                if (OP == 5) asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z));
                /* mixes: do the pipes run side by side?  (ops counted: all of them) */
                if (OP == 6) { if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z)); }
                if (OP == 7) { if (i & 3) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("popc.b32 %0, %0;" : "+r"(x[i])); }
                if (OP == 8) { if (i == 0) asm volatile("popc.b32 %0, %0;" : "+r"(x[i]));
                               else if (i < 5) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z)); }
            }
        }
    }
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= x[i];
    if (s == 0x12345u) out[0] = s;
}

/* random 16-byte gathers from a 64 MB (L2-resident) table, four independent loads per thread in flight:
 * the sector rate the "index" variant's slot probes can reach at best */
__global__ void __launch_bounds__(1024, 1) gkm_mb_gather_kernel(const uint4 *__restrict__ tab, uint32_t mask, int iters, uint32_t *out)
{
    uint32_t s = (blockIdx.x * 1024u + threadIdx.x) * 2654435761u + 12345u;
    uint32_t acc = 0;
    for (int i = 0; i < iters; i++) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            s = s * 1664525u + 1013904223u;
            v[u] = __ldg(tab + ((s >> 4) & mask));
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc ^= v[u].x ^ v[u].y ^ v[u].z ^ v[u].w;
    }
    if (acc == 0x9E3779B9u) out[0] = acc;
}

/* shared-memory atomic adds the way the index variant's hit path issues them: each warp instruction has ~`active` of
 * its 32 lanes on (a probe finds a posting in the wanted range for a few lanes only), each on a random column of an
 * 80 KB histogram row; two CTAs of 1024 threads per SM like the hot loop.  Result: atomics per second. */
__global__ void __launch_bounds__(1024, 2) gkm_mb_atoms_kernel(int iters, uint32_t ncols, uint32_t active, unsigned long long *total)
{
    extern __shared__ int32_t mbH[];
    for (uint32_t i = threadIdx.x; i < ncols; i += 1024u) mbH[i] = 0;
    __syncthreads();
    uint32_t s = (blockIdx.x * 1024u + threadIdx.x) * 2654435761u + 12345u;
    uint32_t cnt = 0;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            s ^= s << 13; s ^= s >> 17; s ^= s << 5;
            const uint32_t col = __umulhi(s, ncols);
            const bool on = ((s >> 3) & 31u) < active;
            if (on) atomicAdd(&mbH[col], 1);
            cnt += on;
        }
    }
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xFFFFFFFFu, cnt, o);
    if ((threadIdx.x & 31u) == 0u) atomicAdd(total, (unsigned long long) cnt + (mbH[threadIdx.x % ncols] < 0 ? 1ull : 0ull));
}

/* device time of launch(rep) on g->sc: the best of repetitions 1..3 (repetition 0 warms up) */
template <class F>
static int best_ms(gkm_gpu *g, const F &launch, float *best)
{
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    *best = 1e30f;
    int rc = 0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, g->sc);
        launch(rep);
        cudaEventRecord(e1, g->sc);
        if (cudaEventSynchronize(e1) != cudaSuccess) { gkm_set_error("CUDA: microbench failed: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < *best) *best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

static int microbench_atoms(gkm_gpu *g, int sms, uint32_t active, double *result)
{
    unsigned long long *d = NULL, h = 0; /* one counter per repetition */
    if (cudaMalloc(&d, 4 * sizeof(*d)) != cudaSuccess) { gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    cudaMemsetAsync(d, 0, 4 * sizeof(*d), g->sc);
    const uint32_t ncols = 20000;
    const unsigned smem = ncols * 4;
    const int iters = 4096;
    cudaFuncSetAttribute(gkm_mb_atoms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    float best;
    const int rc = best_ms(g, [&](int rep) { gkm_mb_atoms_kernel<<<2 * sms, 1024, smem, g->sc>>>(iters, ncols, active, d + rep); }, &best);
    if (!rc) cudaMemcpy(&h, d + 3, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (!rc) *result = (double) h / ((double) best * 1e-3) / 1e9;
    return rc;
}

static int microbench_gather(gkm_gpu *g, int sms, double *result)
{
    const size_t slots = (size_t) 1 << 22; /* 4 Mi x 16 B = 64 MB, the size of the L = 11 slot table */
    uint4 *tab = NULL;
    uint32_t *d = NULL;
    if (cudaMalloc(&tab, slots * sizeof(uint4)) != cudaSuccess || cudaMalloc(&d, 64) != cudaSuccess) {
        gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError()));
        cudaFree(tab);
        return 1;
    }
    cudaMemsetAsync(tab, 0x5A, slots * sizeof(uint4), g->sc);
    const int iters = 2048;
    float best;
    const int rc = best_ms(g, [&](int) { gkm_mb_gather_kernel<<<sms, 1024, 0, g->sc>>>(tab, (uint32_t) (slots - 1), iters, d); }, &best);
    cudaFree(tab); cudaFree(d);
    if (!rc) *result = (double) sms * 1024.0 * (double) iters * 4.0 / ((double) best * 1e-3) / 1e9; /* 1e9 gathers (sectors) per second */
    return rc;
}

extern "C" int gkm_dev_microbench(const char *what, double *result)
{
    if (!what || !result) { gkm_set_error("null argument"); return 1; }
    static const struct { const char *name; void (*fn)(uint32_t *, int, uint32_t); } ops[] = {
        { "lop3", gkm_mb_kernel<0> }, { "shf", gkm_mb_kernel<1> }, { "popc", gkm_mb_kernel<2> }, { "iadd3", gkm_mb_kernel<3> },
        { "imad", gkm_mb_kernel<4> }, { "imadhi", gkm_mb_kernel<5> }, { "lop3+imad", gkm_mb_kernel<6> },
        { "lop3+popc", gkm_mb_kernel<7> }, { "lop3+imad+popc", gkm_mb_kernel<8> } };
    pthread_mutex_lock(&g_lock);
    int rc = ensure_selected();
    gkm_gpu *g = rc ? NULL : &g_gpu[g_sel[0]];
    if (!rc) rc = gpu_prepare(g, g_sel[0], 0, 0);
    if (!rc) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->id);
        int op = -1;
        for (int i = 0; i < (int) (sizeof(ops) / sizeof(ops[0])); i++) if (!strcmp(what, ops[i].name)) op = i;
        if (!strcmp(what, "gather16")) rc = microbench_gather(g, sms, result);
        else if (!strcmp(what, "atoms7")) rc = microbench_atoms(g, sms, 7u, result);
        else if (!strcmp(what, "atoms14")) rc = microbench_atoms(g, sms, 14u, result);
        else if (!strcmp(what, "atoms32")) rc = microbench_atoms(g, sms, 32u, result);
        else if (op < 0) { gkm_set_error("unknown microbench %s", what); rc = 1; }
        else {
            uint32_t *d = NULL;
            const int iters = 4096, blocks = sms * 8;
            float best;
            if (cudaMalloc(&d, 64) != cudaSuccess) { gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            else rc = best_ms(g, [&](int rep) { ops[op].fn<<<blocks, 256, 0, g->sc>>>(d, iters, 12345u + rep); }, &best);
            cudaFree(d);
            if (!rc) *result = (double) blocks * 256.0 * (double) iters * 32.0 / ((double) best * 1e-3) / 1e9;
        }
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}
