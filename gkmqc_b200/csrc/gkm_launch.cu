/* gkm_launch.cu -- which kernel variant serves a call and one launch of a histogram kernel: the bit-sliced kernels
 * (one object per L, gkm_diag_inst.cu), the lmer and mma kernels, and the index variant's row kernel over the column
 * blocks this file cuts and builds. */
#include "gkm_dev.h"
#include "gkm_options.h"
#include "gkm_lmer_kernel.cuh"

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

/* ---- one launch of a histogram kernel over the block described by kp ---- */
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
        gkm_idx_launch ran;
        if (gkm_idx_rows(&kp, &ra, p->weighted, st, &ran)) return 1;
        g->nkernels++;
        if (im == &p->dev->img[0] && ran.minb) { /* what gkmb200_problem_index_blocks reports */
            gkm_idx_block *bw = const_cast<gkm_idx_block *>(b);
            bw->inst_mask |= 1 << (2 * ran.range + ran.minb - 1);
            if (ran.smem > bw->max_smem) bw->max_smem = ran.smem;
            bw->launches++;
        }
    }
    return 0;
}

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

int launch_hist(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, gkm_kparams kp, cudaStream_t st, int *variant_out)
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
        if (st == g->sc && stream_join(g, g->sc, g->sc2)) return 1; /* the other compute stream sees the copy too */
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

void fill_kparams(const gkmb200_problem *p, const gkm_image *im, int mode, gkm_kparams *kp)
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

/* the rows and columns of one chunk; the caller says where the entries go */
gkm_kparams chunk_kparams(const gkmb200_problem *p, const gkm_image *im, const gkm_chunk *c, int mode)
{
    gkm_kparams kp;
    fill_kparams(p, im, mode, &kp);
    kp.row_begin = c->row_begin; kp.row_end = c->row_end;
    kp.col_begin = c->col_begin; kp.col_end = c->col_end;
    return kp;
}

/* kp (GKM_MODE_DIAG) over the diagonal entries of the rows [r0, r1) on g->sc, kp.hist (if set) from row r0; returns the number of
 * launches, or -1.  The bit-sliced kernel covers the diagonal with one column of CTAs, 8 rows each: one launch for up to
 * 131 070 rows (grid.y <= 65 535 row tiles of at least 2 rows; it was 10 launches of 32 x 128 CTAs at 10k, 1.8 ms of
 * device time); other variants take blocks of 1024 rows. */
int launch_diag_rows(const gkmb200_problem *p, const gkm_image *im, gkm_gpu *g, int r0, int r1, gkm_kparams kp)
{
    int32_t *H = kp.hist;
    const int step = (pick_variant(p, GKM_MODE_DIAG) == GKM_KERNEL_DIAG) ? 131070 : 1024;
    for (int r = r0; r < r1; r += step) {
        kp.row_begin = kp.col_begin = kp.row_base = kp.col_base = r;
        kp.row_end = kp.col_end = (r + step < r1) ? r + step : r1;
        if (H) kp.hist = H + (size_t) (r - r0) * (size_t) p->nbins;
        if (launch_hist(p, im, g, kp, g->sc, NULL)) return -1;
    }
    return (r1 - r0 + step - 1) / step;
}
/* ---- "index" variant: per-GPU mask list, per-image column-block indexes ---- */
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

void release_index(gkm_gpu *g, gkm_image *im)
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
    if (g->d_deltas) { gpu_drain(g, 0); pool_free(g, g->d_deltas, g->deltas_bytes); g->d_deltas = NULL; }
    if (pool_alloc(g, (void **) &g->d_deltas, &g->deltas_bytes, (size_t) nd * 4)) { free(h); return 1; }
    cudaError_t e = cudaMemcpyAsync(g->d_deltas, h, (size_t) nd * 4, cudaMemcpyHostToDevice, g->sc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc); /* h is pageable and freed below */
    free(h);
    if (e != cudaSuccess) { gkm_set_error("CUDA: mask upload: %s", cudaGetErrorString(e)); return 1; }
    g->delta_L = L; g->delta_d = d; g->ndelta = (int) nd; g->ncold = (int) gkm_idx_cold_count(L, d);
    return 0;
}

/* The key fields of *a for the columns [cb, ce) of im but offs and scratch: the posting offsets of the columns into *offs
 * (malloc'd) and the sort's scratch bytes into *sbytes.  Returns 0; 1 out of memory; 2 when the columns hold more
 * postings than a key can number (a->P tells how many, the caller words the error). */
int column_keys_prepare(const gkmb200_problem *p, const gkm_image *im, int cb, int ce, gkm_idx_build_args *a, uint32_t **offs, size_t *sbytes)
{
    const int L = p->param.L;
    if (!(*offs = (uint32_t *) malloc((size_t) (ce - cb) * 4))) { gkm_set_error("out of memory"); return 1; }
    size_t P = 0;
    for (int i = 0; i < ce - cb; i++) { (*offs)[i] = (uint32_t) P; P += 2 * (size_t) (p->len[cb + i] - L + 1); }
    a->planes = im->planes; a->lens = im->lens; a->wend = p->weighted ? im->wend : NULL;
    a->W = p->Wmax; a->L = L; a->cb = cb; a->ce = ce; a->P = P;
    if (P > 0x7FFFFFF0u) { free(*offs); *offs = NULL; return 2; }
    *sbytes = gkm_idx_scratch_bytes(P, L, &a->cub_bytes);
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
        gpu_drain(g, 0);
        release_index(g, im);
    }
    if (!im->blk) {
        const int cap = index_block_cap(p);
        if (cap <= 0) { gkm_set_error("index variant: sequences too long for shared memory"); return 1; }
        int cols = 0;
        const int nblk = gkm_plan_index_blocks(col_end - col_begin, cap, greedy, &cols);
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
        gkm_idx_build_args a;
        uint32_t *offs = NULL;
        size_t sbytes = 0;
        const int kr = column_keys_prepare(p, im, b->cb, b->ce, &a, &offs, &sbytes);
        if (kr == 2) gkm_set_error("index variant: column block too large");
        if (kr) return 1;
        const size_t P = a.P;
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
            a.offs = (const uint32_t *) d_offs; a.scratch = scratch;
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
        b->postings = P;
        b->skew = (double) b->sumsq / (double) (P ? P : 1);
        gkm_log(GKM_LOG_DEBUG, "index block %d: %zu postings, sum len^2 / postings = %.2f", k, P, b->skew);
        b->built = 1;
        __atomic_fetch_add(&p->stats.launches, 5, __ATOMIC_RELAXED); /* the GPUs of a call build their indexes side by side */
    }
    return 0;
}

/* which kernel variant serves a block of rows x cols; for the index also makes sure that the
 * indexes exist on every GPU.  Called under g_lock after upload_locked. */
int choose_variant(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower)
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
        int blocks = 0, cols = 0;
        if (ok) {
            blocks = gkm_plan_index_blocks(ncols, cap, greedy, &cols);
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
            if (greedy) { /* rows of block k probe k + 1 blocks; all blocks but the last hold cols columns */
                double s = 0.0;
                for (int k = 0; k < blocks; k++) s += (double) (k + 1) * (double) ((k + 1) * cols <= ncols ? cols : ncols - k * cols);
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
                return ensure_index(p, g, &ds->img[slot], col0, col0 + ncols, greedy, gopt >= 0) || stream_join(g, g->sc, g->sc2);
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
    for (int k = 0; k < ds->img[0].nblk; k++) { /* the launch record starts over with every compute call */
        gkm_idx_block *b = &ds->img[0].blk[k];
        b->inst_mask = 0; b->max_smem = 0; b->launches = 0;
    }
    return 0;
}
