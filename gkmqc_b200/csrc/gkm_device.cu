/* gkm_device.cu -- device layer of gkmkern_pylib.so: GPU selection, the per-GPU resources and their block pool, and the
 * problem image every selected GPU holds (upload, packing on the device, release).  The other files of the device layer
 * share these through gkm_dev.h. */
#include <time.h>

#include "gkm_dev.h"
#include "gkm_options.h"
#include "gkm_pack.h"

gkm_gpu g_gpu[GKM_MAX_DEV];
int g_sel[GKM_MAX_DEV];
int g_nsel = -1;
pthread_mutex_t g_lock = PTHREAD_MUTEX_INITIALIZER;

/* give the cached blocks of one GPU back to the driver (current device must be g's) */
static void pool_trim(gkm_gpu *g)
{
    for (int i = 0; i < g->npool; i++) cudaFree(g->pool[i].ptr);
    g->npool = 0;
}

/* cudaMalloc that, when the device is out of memory, first returns this library's own cached blocks (up to 32 blocks
 * of up to 512 MB per GPU would otherwise stand between a long-lived host and a 50k x 50k problem) and tries again */
cudaError_t dev_malloc(gkm_gpu *g, void **out, size_t bytes)
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

double now_ms(void)
{
    struct timespec t;
    clock_gettime(CLOCK_MONOTONIC, &t);
    return 1e3 * (double) t.tv_sec + 1e-6 * (double) t.tv_nsec;
}

/* GPU `ordinal` is an sm_100 part (B200) */
static int is_b200(int ordinal)
{
    int major = 0;
    return cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, ordinal) == cudaSuccess && major == 10;
}

extern "C" int gkm_dev_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n && i < GKM_MAX_DEV; i++) ok += is_b200(i);
    return ok;
}

extern "C" int gkmb200_device_count(void) { return gkm_dev_count(); }

extern "C" int gkm_dev_select(const int *ids, int n)
{
    int total = 0;
    if (cudaGetDeviceCount(&total) != cudaSuccess) { cudaGetLastError(); total = 0; }
    if (n < 1 || n > GKM_MAX_DEV) { gkm_set_error("bad device list"); return 1; }
    for (int i = 0; i < n; i++) {
        if (ids[i] < 0 || ids[i] >= total || !is_b200(ids[i])) {
            gkm_set_error("device %d is not a visible sm_100 GPU", ids[i]);
            return 1;
        }
    }
    for (int i = 0; i < n; i++) g_sel[i] = ids[i];
    g_nsel = n;
    return 0;
}

extern "C" int gkmb200_set_devices(const int *ids, int n) { return gkm_dev_select(ids, n); }

int ensure_selected(void)
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
    for (int i = 0; i < total && n < GKM_MAX_DEV; i++) if (is_b200(i)) ids[n++] = i;
    if (n == 0) {
        gkm_set_error("no sm_100 (B200) GPU is visible: gkmkern_pylib.so has no CPU fallback");
        return 1;
    }
    return gkm_dev_select(ids, n);
}

int gpu_prepare(gkm_gpu *g, int id, size_t band_bytes, size_t stage_bytes)
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

/* work queued on `to` from now on waits for what is queued on `from` so far (both compute or copy streams of g) */
int stream_join(gkm_gpu *g, cudaStream_t from, cudaStream_t to)
{
    CK(cudaEventRecord(g->join, from));
    CK(cudaStreamWaitEvent(to, g->join, 0));
    return 0;
}

/* wait until g's compute streams (and its copy stream) have drained; the first error met */
cudaError_t gpu_drain(gkm_gpu *g, int with_copy_stream)
{
    const cudaError_t e1 = cudaStreamSynchronize(g->sc), e2 = cudaStreamSynchronize(g->sc2);
    const cudaError_t e3 = with_copy_stream ? cudaStreamSynchronize(g->sx) : cudaSuccess;
    return e1 != cudaSuccess ? e1 : e2 != cudaSuccess ? e2 : e3;
}


/* ---- upload: packed image to every selected GPU; sqnorm = diagonal of the kernel ---- */
/* device blocks come from / go back to a per-GPU free list (current device must be g's) */
int pool_alloc(gkm_gpu *g, void **out, size_t *got, size_t bytes)
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

void pool_free(gkm_gpu *g, void *ptr, size_t bytes)
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


/* the image as it lies on GPU 0 (tests: the device packer against a model of the image): planes [n][3][W] and, for the
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

/* the index blocks of the last compute call of this problem on its first GPU (0 when another variant ran); per block, up to
 * max of them, 8 values from out[8 k]: {first column, end column, slot format, postings, sum of squared posting-list
 * lengths, builds that ran (bit 2 RANGE + MINB - 1 of gkm_index_rows_kernel), most dynamic shared memory of a launch,
 * launches}.  For tests: which row-kernel builds a call ran. */
extern "C" int gkmb200_problem_index_blocks(const gkmb200_problem *p, long long *out, int max)
{
    if (!p || (!out && max > 0)) { gkm_set_error("null argument"); return -1; }
    int nblk = 0;
    pthread_mutex_lock(&g_lock);
    if (p->dev && p->dev->variant == GKM_KERNEL_INDEX && p->dev->img[0].blk) {
        const gkm_image *im = &p->dev->img[0];
        nblk = im->nblk;
        for (int k = 0; k < nblk && k < max; k++) {
            const gkm_idx_block *b = &im->blk[k];
            long long *o = out + 8 * (size_t) k;
            o[0] = b->cb; o[1] = b->ce; o[2] = b->fmt; o[3] = (long long) b->postings; o[4] = (long long) b->sumsq;
            o[5] = b->inst_mask; o[6] = b->max_smem; o[7] = b->launches;
        }
    }
    pthread_mutex_unlock(&g_lock);
    return nblk;
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
        gpu_drain(g, 1);
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
        if (g->ready) gpu_drain(g, 1);
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

/* ---- packing on the device (SURVEY.md 8f/f2): sequence letters -> the image of 3 ---- */
/* The rule of gkm_pack.h, one CTA per sequence, one warp per 32-position word of the circular string, plane bits by warp
 * ballot.  The input is the sequence TEXT, one byte per base as the FASTA file or the caller spelled it. */
template <bool WEIGHTED>
__global__ void __launch_bounds__(128)
gkm_pack_kernel(const uint8_t *__restrict__ codes, const unsigned long long *__restrict__ off, const int32_t *__restrict__ lens,
                int W, int L, const uint8_t *__restrict__ wtab, uint32_t *__restrict__ planes, uint8_t *__restrict__ wend)
{
    const int i = (int) blockIdx.x;
    const int len = lens[i], centre = (len - L + 1) / 2;
    const uint8_t *c = codes + off[i];
    const int lane = (int) threadIdx.x & 31;
    for (int wi = (int) threadIdx.x >> 5; wi < W; wi += 4) {
        const int j = wi * 32 + lane;
        int s;
        const uint32_t code = gkm_pack_code(c, len, L, j, &s);
        const uint32_t p0 = __ballot_sync(0xFFFFFFFFu, code & 1u), p1 = __ballot_sync(0xFFFFFFFFu, code & 2u);
        const uint32_t pe = __ballot_sync(0xFFFFFFFFu, s >= 0);
        if (lane == 0) {
            uint32_t *pl = planes + (size_t) i * 3 * (size_t) W;
            pl[wi] = p0; pl[W + wi] = p1; pl[2 * W + wi] = pe;
        }
        if (WEIGHTED) wend[(size_t) i * 32 * (size_t) W + (size_t) j] = gkm_pack_weight(wtab, centre, s);
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
int upload_locked(gkmb200_problem *p, int need_host)
{
    if (p->dev && p->packed && p->have_sqnorm) return need_host ? fetch_sqnorm(p) : 0;
    if (ensure_selected()) return 1;
    const double t0 = now_ms();
    gkm_dev_release(p);
    if (gkm_shape_problem(p)) return 1;
    uint8_t wtab[GKM_MAX_BASES + 1];
    if (p->weighted) gkm_posweight_table(p->param.kernel_type, p->param.M, p->param.H, wtab);
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
        /* one byte per base goes up (3 MB at 10k x 300 bp, against 8.3 MB for the packed image of a weighted problem) and
         * the GPU packs: codes | offsets | weight table in one block */
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
        /* sqnorm: Kraw(a,a) by the same kernel in diagonal mode */
        gkm_kparams kp;
        fill_kparams(p, im, GKM_MODE_DIAG, &kp);
        kp.sqnorm_out = im->sqnorm;
        const int launches = launch_diag_rows(p, im, g, 0, p->n, kp);
        if (launches < 0) return 1;
        p->stats.launches += launches;
        if (stream_join(g, g->sc, g->sc2)) return 1; /* the second compute stream starts behind sqnorm too */
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

