/* gkm_compute.cu -- blocks of the kernel matrix into caller memory, and the fused decision values.
 * Stands where the reference has its pthread row scheduler and row loop
 * (gkmkern_pylib.c:70-90,169-216 -> libgkm.c:1156): thread t there takes rows
 * t, t+T, ...; here one host thread per GPU takes whole chunks of row tiles, the
 * GPU computes chunk i+1 while chunk i is copied D2H (second stream, pinned
 * staging) and scattered into the caller's rows by `copy_threads` host threads.
 * The caller's matrix is neither pinned nor contiguous (numpy rows with a
 * 120 000-byte stride, gkmsvm.py:75-77), hence the bounce buffer.
 * There is no collective: every chunk depends only on the replicated sequence image.
 */
#include <sched.h>
#include <semaphore.h>
#include <unistd.h>

#include "gkm_dev.h"
#include "gkm_options.h"

#define GKM_WAVE_ROWS 148 /* rows of one wave of the index variant's row kernel: one CTA per row and SM */

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
    gkm_kparams kp = chunk_kparams(job->p, im, c, job->lower ? GKM_MODE_LOWER : GKM_MODE_RECT);
    kp.row_base = c->row_begin;
    kp.col_base = c->col_begin;
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
    gkm_dbuf<int32_t> d_hist(g);
    int32_t *h_hist = NULL;
    if (job->hist) {
        CK(d_hist.alloc((maxhist ? maxhist : 4) / 4));
        h_hist = (int32_t *) malloc(maxhist ? maxhist : 4);
        if (!h_hist) { gkm_set_error("out of memory"); return 1; }
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
int plan_chunks(const gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower, int nshare, gkm_chunk **out)
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

/* ---- fused decision values (SURVEY.md 8f/f1) ---- */
/* one GPU's slice of the test rows: out[r] = bias + sum_c alpha[c] K(row0 + r, col0 + c) */
static int decision_slice(gkmb200_problem *p, int slot, int row0, int nrows, int col0, int ncols, const double *alpha, double bias, double *out)
{
    if (nrows <= 0) return 0;
    gkm_devstate *ds = p->dev;
    gkm_gpu *g = &g_gpu[ds->dev[slot]];
    gkm_dbuf<double> d_alpha(g), d_dec(g);
    cudaError_t e = d_alpha.alloc((size_t) (ncols ? ncols : 1));
    if (e == cudaSuccess) e = d_dec.alloc((size_t) nrows);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_alpha, alpha, sizeof(double) * (size_t) ncols, cudaMemcpyHostToDevice, g->sc);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_dec, 0, sizeof(double) * (size_t) nrows, g->sc);
    /* the second compute stream must see alpha and the zeroed accumulator too */
    int rc = e != cudaSuccess || stream_join(g, g->sc, g->sc2);
    if (rc) gkm_set_error("CUDA: decision-value buffers: %s", cudaGetErrorString(cudaGetLastError()));
    gkm_kparams kp;
    fill_kparams(p, &ds->img[slot], GKM_MODE_RECT, &kp);
    kp.alpha = d_alpha; kp.decision = d_dec;
    kp.col_begin = kp.col_base = col0; kp.col_end = col0 + ncols;
    kp.row_base = row0;
    const long long k_before = g->nkernels;
    int launches = 0;
    /* index variant: whole waves of rows per launch, and a bounded cold-bin scratch */
    const int rows_per_launch = (ds->variant == GKM_KERNEL_INDEX) ? 16 * GKM_WAVE_ROWS : 8192;
    for (int r = row0; !rc && r < row0 + nrows; r += rows_per_launch) {
        kp.row_begin = r;
        kp.row_end = (r + rows_per_launch < row0 + nrows) ? r + rows_per_launch : row0 + nrows;
        rc = launch_hist(p, &ds->img[slot], g, kp, (launches++ & 1) ? g->sc2 : g->sc, NULL);
    }
    /* kernels, not row blocks: the index variant launches one per column block; the GPUs of a call add side by side */
    __atomic_fetch_add(&p->stats.launches, g->nkernels - k_before, __ATOMIC_RELAXED);
    if (!rc) {
        rc = (cudaStreamSynchronize(g->sc2) != cudaSuccess) ||
             (cudaMemcpyAsync(out, d_dec, sizeof(double) * (size_t) nrows, cudaMemcpyDeviceToHost, g->sc) != cudaSuccess) ||
             (cudaStreamSynchronize(g->sc) != cudaSuccess);
        if (rc) gkm_set_error("CUDA: decision values failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!rc) for (int i = 0; i < nrows; i++) out[i] += bias;
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
    p->stats.launches = 0;
    int rc = upload_locked(p, 0);
    if (!rc) rc = choose_variant(p, row0, nrows, col0, ncols, 0);
    if (!rc) p->stats.kernel_variant = p->dev->variant;
    if (!rc) rc = for_each_gpu_share(p->dev, nrows, 8, [&](int slot, long long b, long long e) {
        return decision_slice(p, slot, row0 + (int) b, (int) (e - b), col0, ncols, alpha, bias, out + b);
    });
    pthread_mutex_unlock(&g_lock);
    return rc;
}

