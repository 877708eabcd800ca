/* gkm_resident.cu -- the resident kernel matrix: one pass of the lower triangle that stays on the GPU, the cross-validated
 * C-SVC that consumes it (SURVEY.md 8f/f4), and the timing of that pass (bench.py). */
#include "gkm_dev.h"
#include "gkm_svm.h"

#define GKM_FLUSH_BYTES ((size_t) 256 << 20) /* > 126 MB L2 */

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
        gkm_kparams kp = chunk_kparams(p, &ds->img[s], &chunks[c], GKM_MODE_LOWER);
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
        if (cudaSetDevice(ds->dev[s]) != cudaSuccess || gpu_drain(gs, 0) != cudaSuccess) {
            if (!rc) gkm_set_error("CUDA: resident matrix, GPU %d: %s", ds->dev[s], cudaGetErrorString(cudaGetLastError()));
            rc = 1;
        }
    }
    CK(cudaSetDevice(ds->dev[0]));
    if (rc) return 1;
    if (stream_join(g, g->sc2, g->sc)) return 1;
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

static int svm_cv(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                  const int *train_idx, const signed char *train_y, const int *test_idx, double C, double eps, int max_iter,
                  int shrinking, double *scores, gkmb200_svm_fit *fits, double *alpha, gkmb200_svm_shrink_stats *stats)
{
    if (ntasks < 0 || (ntasks > 0 && (!tasks || !train_idx || !train_y || !test_idx))) { gkm_set_error("null argument"); return 1; }
    if (!(C > 0.0) || !(eps > 0.0)) { gkm_set_error("svm: C and eps must be positive"); return 1; }
    if (shrinking != 0 && shrinking != 1) { gkm_set_error("svm: shrinking must be 0 or 1, not %d", shrinking); return 1; }
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
                             C, eps, max_iter, shrinking, scores, fits, alpha, stats, g->sc);
            p->stats.launches += 3;
            p->stats.wall_ms = now_ms() - t0;
        }
    } else {
        if (n < 2 || ld < n) { gkm_set_error("svm: bad matrix shape"); rc = 1; }
        if (!rc) rc = ensure_selected();
        if (!rc) {
            gkm_gpu *g = &g_gpu[g_sel[0]];
            gkm_dbuf<double> d_K(g);
            rc = gpu_prepare(g, g_sel[0], 0, 0);
            if (!rc && d_K.alloc((size_t) n * (size_t) n) != cudaSuccess) { gkm_set_error("CUDA: svm matrix: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            if (!rc && cudaMemcpy2DAsync(d_K, sizeof(double) * (size_t) n, kmat, sizeof(double) * (size_t) ld, sizeof(double) * (size_t) n, (size_t) n,
                                         cudaMemcpyHostToDevice, g->sc) != cudaSuccess) { gkm_set_error("CUDA: svm matrix upload: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            if (!rc) rc = gkm_svm_run(d_K, (long long) n, n, ntasks, tasks, train_idx, train_y, test_idx, C, eps, max_iter, shrinking,
                                      scores, fits, alpha, stats, g->sc);
        }
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}

extern "C" int gkm_dev_svm_cv(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                              const int *train_idx, const signed char *train_y, const int *test_idx,
                              double C, double eps, int max_iter, double *scores, gkmb200_svm_fit *fits, double *alpha)
{
    return svm_cv(p, kmat, ld, n, ntasks, tasks, train_idx, train_y, test_idx, C, eps, max_iter, 0, scores, fits, alpha, NULL);
}

extern "C" int gkmb200_svm_cv_ex(gkmb200_problem *p, const double *kmat, long ld, int n, int ntasks, const gkmb200_svm_task *tasks,
                                 const int *train_idx, const signed char *train_y, const int *test_idx, const gkmb200_svm_options *opt,
                                 double *scores, gkmb200_svm_fit *fits, double *alpha, gkmb200_svm_shrink_stats *stats)
{
    if (!opt) { gkm_set_error("null argument"); return 1; }
    return svm_cv(p, kmat, ld, n, ntasks, tasks, train_idx, train_y, test_idx, opt->C, opt->eps, opt->max_iter, opt->shrinking,
                  scores, fits, alpha, stats);
}

/* ---- measurement ---- */
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
            (flush_l2 && !g->d_flush && dev_malloc(g, &g->d_flush, GKM_FLUSH_BYTES) != cudaSuccess)) {
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
            stream_join(g, g->sc2, g->sc);
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

