/* gkm_mma_kernel.cuh -- sm_100a kernel "mma": candidate (b) of the north star, round-2 build.
 *
 * One-hot L-mer GEMM on the 5th-generation tensor cores: every L-mer becomes a row of K = 64 bytes (byte 4t + code(t) = 1
 * for t < L, zero padding behind 4L), so that
 *     D[i][j] = sum_k A[i][k] B[j][k] = number of MATCHING positions of query L-mer i and target L-mer j;
 * mismatches = L - D.  `tcgen05.mma.cta_group::1.kind::i8` (M = 128, N = 256, two K = 32 steps, int32 accumulators in
 * TMEM), fused epilogue: the L-mer x L-mer product never reaches HBM.
 *
 * Round 1 ran MMA -> wait -> epilogue strictly one after the other, one query per CTA, operands fetched with plain
 * loads (tensor pipe 15 % active).  This build is a warp-specialised pipeline:
 *
 *   TMA          the 2-bit plane rows of the CTA's QA queries and TB targets arrive in shared memory by
 *                cp.async.bulk.tensor.2d (one elected thread, mbarrier complete_tx) from a 16-byte-pitched copy of the
 *                problem image
 *   A operand    the L-mers of up to 4 queries STACKED (rows of consecutive queries follow each other, so 4 x 290 rows
 *                fill 10 tiles of 128 instead of 4 x 3), built once per CTA in the K-major no-swizzle core-matrix layout
 *   builders     2 warps expand the target L-mers of the next N tile into a 2-stage ring of B operands
 *   MMA warp     one elected thread issues the two K = 32 MMAs of tile (A[mt], B[stage]) into one of TWO 256-column
 *                accumulators and commits to its mbarrier; a commit per B stage hands the stage back to the builders
 *   epilogue     16 warps (TMEM lane quarter x column group of 64) read an accumulator with one
 *                tcgen05.ld.32x32b.x32.pack::16b (two 16-bit columns per register), hand it back -- the MMA of tile n + 1
 *                runs under the epilogue of tile n -- reject groups of 16 registers by an OR tree on the hit bit that
 *                the operands' bias sets (a max tree at L = 16), and bin the rest
 *
 * It exists for the measured comparison with the bit-sliced kernel (DESIGN.md 4.3): every accumulator -- one per L-mer
 * PAIR -- has to leave TMEM and meet at least half a CUDA-core instruction.  Selected with GKM_KERNEL=mma.
 */
#ifndef GKM_MMA_KERNEL_CUH_INCLUDED
#define GKM_MMA_KERNEL_CUH_INCLUDED

#include <cuda.h> /* CUtensorMap */

#include "gkm_diag_kernel.cuh" /* gkm_emit_entry */

#define GKM_MMA_EPI 16           /* epilogue warps: TMEM lane quarter (w & 3) x column group (w >> 2) */
#define GKM_MMA_CW (GKM_MMA_N / (GKM_MMA_EPI / 4))   /* accumulator columns per epilogue warp */
#define GKM_MMA_NV (GKM_MMA_CW / 2)                  /* registers of one epilogue thread per tile: two columns each */
#define GKM_MMA_HSETS (GKM_MMA_EPI / 4)              /* histogram sets: one per column group */
#define GKM_MMA_THREADS ((GKM_MMA_EPI + 4) * 32)     /* epilogue warps, then MMA, TMA, two builder warps */
#define GKM_MMA_M 128
#define GKM_MMA_N 256
#define GKM_MMA_TB 8             /* targets per CTA */
#define GKM_MMA_QA 4             /* queries per CTA, at most */
#define GKM_MMA_ROWS_CAP 2176    /* stacked query L-mers per CTA (17 tiles of 128: 136 KB of A operand) */
#define GKM_MMA_BUILDERS 64
#define GKM_MMA_TMA_BOX 256      /* elements of one TMA box along a plane row, at most */

struct gkm_mma_args {
    int QA;        /* queries per CTA for this launch: min(4, ROWS_CAP / longest query) */
    int P;         /* words per row of the padded image (3 W rounded up to a multiple of 4: 16-byte pitch) */
    int box;       /* words per TMA box (P split into equal boxes of at most 256) */
    int nbox;      /* boxes per row */
};

__host__ __device__ inline int gkm_mma_stage_words(const gkm_mma_args &m) { return m.box * m.nbox; }

__host__ __device__ inline unsigned gkm_mma_smem_bytes(int rows_cap_tiles, int stage_words, int nbins, int weighted)
{
    unsigned o = 1024;                                               /* barriers, TMEM slot, lengths, tile table */
    o += (unsigned) rows_cap_tiles * GKM_MMA_M * 64u;                /* A operand: the stacked query L-mers */
    o += 2u * GKM_MMA_N * 64u;                                       /* B operand ring */
    o += (unsigned) (GKM_MMA_QA + GKM_MMA_TB) * (unsigned) stage_words * 4u;   /* plane rows as TMA delivers them */
    o += (unsigned) rows_cap_tiles * GKM_MMA_M;                      /* query of every stacked row */
    o += (unsigned) GKM_MMA_HSETS * GKM_MMA_QA * GKM_MMA_TB * (unsigned) nbins * 4u;   /* histograms, one set per column group */
    if (weighted) o += (unsigned) rows_cap_tiles * GKM_MMA_M + 8u * GKM_MMA_N;
    return (o + 127u) & ~127u;
}

__device__ __forceinline__ uint32_t gkm_smem_u32(const void *p) { return (uint32_t) __cvta_generic_to_shared(p); }

/* K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
 * core matrix = 8 rows x 16 bytes, rows 16 bytes apart; LBO = distance of the two 16-byte K chunks,
 * SBO = distance of consecutive 8-row groups, both in 16-byte units; version 1 (Blackwell). */
__device__ __forceinline__ uint64_t gkm_umma_desc(uint32_t saddr, uint32_t lbo16, uint32_t sbo16)
{
    return (uint64_t) ((saddr >> 4) & 0x3FFFu) | ((uint64_t) (lbo16 & 0x3FFFu) << 16) |
           ((uint64_t) (sbo16 & 0x3FFFu) << 32) | ((uint64_t) 1 << 46);
}

/* one operand row (64 bytes = 16 words, word t = one-hot byte of base t) as 4 chunks of 16 bytes:
 * chunk kc of row r lives at base + kc*rows*16 + r*16 */
/* `spare` goes into word L, the first K bytes behind the L-mer (zero for L = 16 and for rows of padding): the bias
 * factors of gkm_mma_bias */
__device__ __forceinline__ void gkm_mma_store_row(unsigned char *base, int rows, int r, uint32_t p0, uint32_t p1, int L, bool valid, uint32_t spare)
{
#pragma unroll
    for (int kc = 0; kc < 4; kc++) {
        uint32_t w[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int t = 4 * kc + u;
            const uint32_t code = ((p0 >> t) & 1u) | (((p1 >> t) & 1u) << 1);
            w[u] = !valid ? 0u : (t < L) ? (1u << (8u * code)) : (t == L) ? spare : 0u;
        }
        *reinterpret_cast<uint4 *>(base + (size_t) kc * rows * 16 + (size_t) r * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

__device__ __forceinline__ void gkm_lmer_planes(const uint32_t *pl, int W, int o, int L, uint32_t &p0, uint32_t &p1)
{
    const int wi = o >> 5, sh = o & 31;
    const uint32_t mask = (L >= 32) ? 0xFFFFFFFFu : ((1u << L) - 1u);
    const uint32_t n0 = (wi + 1 < W) ? pl[wi + 1] : 0u, n1 = (wi + 1 < W) ? pl[W + wi + 1] : 0u;
    p0 = __funnelshift_r(pl[wi], n0, sh) & mask;
    p1 = __funnelshift_r(pl[W + wi], n1, sh) & mask;
}

/* The threshold test rides on the MMA.  K = 64 bytes hold 4 L <= 60 one-hot bytes; two of the spare ones carry factors
 * whose product sum is 2^15 - thr (255 * 128 + (128 - thr) * 1, thr = L - d matches needed for a hit), so that every
 * accumulator of two real L-mers comes out of TMEM as matches + 2^15 - thr: bit 15 is set exactly for the hits.  The
 * epilogue then rejects 16 accumulators with an OR tree (LOP3, 0.5 instructions per accumulator at full ALU rate) instead of
 * the 3-input max tree of the first build, which ncu showed to be the bound (VIMNMX3 issues at a fraction of the ALU
 * rate: 344 of 463 ms at 4 000 sequences).  L = 16 has no spare byte and keeps the max tree. */
__device__ __forceinline__ uint32_t gkm_mma_bias_a(int L, int thr) { return (L <= 15) ? (255u | ((uint32_t) (128 - thr) << 8)) : 0u; }
__device__ __forceinline__ uint32_t gkm_mma_bias_b(int L) { return (L <= 15) ? (128u | (1u << 8)) : 0u; }

/* ---- mbarrier helpers.  A wait never hangs the device: a lost arrival is a hard error (__trap). ---- */
__device__ __forceinline__ void gkm_mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(gkm_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void gkm_mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(gkm_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void gkm_mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(gkm_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gkm_mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done = 0, spins = 0;
    while (!done) {
        if (++spins > (1u << 24)) __trap();
        asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                     : "=r"(done) : "r"(gkm_smem_u32(bar)), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void gkm_umma_commit(uint64_t *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(gkm_smem_u32(bar)) : "memory");
}
/* one box of a plane row: words [x, x + box) of image row y -> shared memory, completion counted in bytes on `bar` */
__device__ __forceinline__ void gkm_tma_row(const CUtensorMap *map, uint64_t *bar, void *dst, int x, int y)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 :: "r"(gkm_smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(gkm_smem_u32(bar)), "r"(x), "r"(y) : "memory");
}

/* barrier block at the head of shared memory */
struct gkm_mma_bars {
    uint64_t planes;        /* TMA: plane rows have landed */
    uint64_t b_full[2];     /* builders -> MMA: B stage holds the next N tile */
    uint64_t b_empty[2];    /* MMA (commit) -> builders: the MMAs that read the stage are done */
    uint64_t acc_full[2];   /* MMA (commit) -> epilogue: accumulator is complete */
    uint64_t acc_empty[2];  /* epilogue -> MMA: accumulator has been read */
    uint32_t tmem_slot;
    int lenA[GKM_MMA_QA], rowoff[GKM_MMA_QA + 1], lenB[GKM_MMA_TB], tile0[GKM_MMA_TB + 1]; /* first N tile of every target */
};

template <bool WEIGHTED>
__global__ void __launch_bounds__(GKM_MMA_THREADS, 1)
gkm_mma_kernel(const __grid_constant__ gkm_kparams p, const __grid_constant__ gkm_mma_args ma, const __grid_constant__ CUtensorMap tmap)
{
    extern __shared__ __align__(128) unsigned char smem_mma[];
    const int W = p.W, L = p.L, d = p.d, NBN = p.nbins, QA = ma.QA;
    const int SW = gkm_mma_stage_words(ma);
    gkm_mma_bars *bars = reinterpret_cast<gkm_mma_bars *>(smem_mma);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int a0 = p.row_begin + (int) blockIdx.y * QA;
    const int col0 = p.col_begin + (int) blockIdx.x * GKM_MMA_TB;
    if (a0 >= p.row_end) return;
    const int nA = min(QA, p.row_end - a0), nB = min(GKM_MMA_TB, p.col_end - col0);
    if (p.mode == GKM_MODE_LOWER && col0 >= a0 + nA - 1) return; /* no column of the group lies below any of its rows */

    /* ---- set-up: barriers, TMEM (both accumulators), the plane rows by TMA ---- */
    if (tid == 0) {
        gkm_mbar_init(&bars->planes, 1);
        for (int s = 0; s < 2; s++) {
            gkm_mbar_init(&bars->b_full[s], GKM_MMA_BUILDERS / 32);
            gkm_mbar_init(&bars->b_empty[s], 1);
            gkm_mbar_init(&bars->acc_full[s], 1);
            gkm_mbar_init(&bars->acc_empty[s], GKM_MMA_EPI);
        }
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == GKM_MMA_EPI) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(gkm_smem_u32(&bars->tmem_slot)), "n"(2 * GKM_MMA_N));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid < GKM_MMA_QA) bars->lenA[tid] = (tid < nA) ? p.lens[a0 + tid] : 0;
    if (tid >= 32 && tid < 32 + GKM_MMA_TB) bars->lenB[tid - 32] = (tid - 32 < nB) ? p.lens[col0 + tid - 32] : 0;
    __syncthreads();

    /* carve shared memory (the A operand sized for this CTA's own rows) */
    int R = 0;
    for (int q = 0; q < GKM_MMA_QA; q++) R += (bars->lenA[q] > 0) ? bars->lenA[q] - L + 1 : 0;
    const int MT = (R + GKM_MMA_M - 1) / GKM_MMA_M;
    unsigned char *sAop = smem_mma + 1024;
    unsigned char *sBop = sAop + (size_t) MT * GKM_MMA_M * 64;
    uint32_t *sPl = reinterpret_cast<uint32_t *>(sBop + 2 * GKM_MMA_N * 64);       /* [QA + TB][SW] */
    uint8_t *sRowQ = reinterpret_cast<uint8_t *>(sPl + (size_t) (GKM_MMA_QA + GKM_MMA_TB) * SW);
    int32_t *sH = reinterpret_cast<int32_t *>(sRowQ + (size_t) MT * GKM_MMA_M);     /* MT*128 is a multiple of 4 */
    uint8_t *sWa = reinterpret_cast<uint8_t *>(sH + GKM_MMA_HSETS * GKM_MMA_QA * GKM_MMA_TB * NBN);
    /* weights of the target L-mers of N tile t live in slot t & 7: the epilogue of tile t still reads them while the
     * builders fill B stages for later tiles (a stage is free as soon as the MMAs have read it, an accumulator as soon
     * as it is in registers; with one M tile per N tile the compares of tile t can lag four tiles behind the builders) */
    uint8_t *sWb = sWa + (WEIGHTED ? MT * GKM_MMA_M : 0);                          /* [8][256] */

    if (warp == GKM_MMA_EPI + 1 && lane == 0) {
        gkm_mbar_expect_tx(&bars->planes, (uint32_t) (nA + nB) * (uint32_t) SW * 4u);
        for (int q = 0; q < nA; q++)
            for (int b = 0; b < ma.nbox; b++) gkm_tma_row(&tmap, &bars->planes, sPl + (size_t) q * SW + (size_t) b * ma.box, b * ma.box, a0 + q);
        for (int t = 0; t < nB; t++)
            for (int b = 0; b < ma.nbox; b++) gkm_tma_row(&tmap, &bars->planes, sPl + (size_t) (GKM_MMA_QA + t) * SW + (size_t) b * ma.box, b * ma.box, col0 + t);
    }
    if (tid == 0) {
        int off = 0, t0 = 0;
        for (int q = 0; q < GKM_MMA_QA; q++) { bars->rowoff[q] = off; off += (bars->lenA[q] > 0) ? bars->lenA[q] - L + 1 : 0; }
        bars->rowoff[GKM_MMA_QA] = off;
        for (int b = 0; b < GKM_MMA_TB; b++) {
            bars->tile0[b] = t0;
            const int nk = (bars->lenB[b] > 0) ? bars->lenB[b] - L + 1 : 0;
            t0 += (2 * nk + GKM_MMA_N - 1) / GKM_MMA_N;
        }
        bars->tile0[GKM_MMA_TB] = t0;
    }
    for (int i = tid; i < GKM_MMA_HSETS * GKM_MMA_QA * GKM_MMA_TB * NBN; i += GKM_MMA_THREADS) sH[i] = 0;
    __syncthreads();
    gkm_mbar_wait(&bars->planes, 0); /* everyone reads the plane rows */

    /* A operand: the forward-strand L-mers of the CTA's queries, stacked */
    for (int i = tid; i < MT * GKM_MMA_M; i += GKM_MMA_THREADS) {
        int q = 0;
        while (q + 1 < GKM_MMA_QA && i >= bars->rowoff[q + 1]) q++;
        const bool valid = i < R;
        const int li = i - bars->rowoff[q];
        uint32_t p0 = 0, p1 = 0;
        if (valid) gkm_lmer_planes(sPl + (size_t) q * SW, W, li, L, p0, p1);
        const int mt = i / GKM_MMA_M, r = i - mt * GKM_MMA_M;
        gkm_mma_store_row(sAop + (size_t) mt * GKM_MMA_M * 64, GKM_MMA_M, r, p0, p1, L, valid, gkm_mma_bias_a(L, L - d));
        sRowQ[i] = valid ? (uint8_t) q : (uint8_t) 0xFF;
        if (WEIGHTED) sWa[i] = valid ? p.wend[(size_t) (a0 + q) * 32 * W + li + L - 1] : 0;
    }
    asm volatile("fence.proxy.async.shared::cta;"); /* generic-proxy stores -> visible to the tensor core */
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem_base = bars->tmem_slot;
    const int NTILES = bars->tile0[GKM_MMA_TB];

    if (warp >= GKM_MMA_EPI + 2) {
        /* ---- builders: target L-mers jj = 256 nt .. +255 over both strands (jj >= nkB: reverse complement) ---- */
        const int bt = tid - (GKM_MMA_EPI + 2) * 32;
        for (int t = 0, b_l = 0; t < NTILES; t++) {
            while (t >= bars->tile0[b_l + 1]) b_l++;
            const int nt = t - bars->tile0[b_l], s = t & 1;
            const int lenB = bars->lenB[b_l], nkB = lenB - L + 1;
            gkm_mbar_wait(&bars->b_empty[s], ((uint32_t) (t >> 1) & 1u) ^ 1u);
            const uint32_t *plb = sPl + (size_t) (GKM_MMA_QA + b_l) * SW;
            for (int r = bt; r < GKM_MMA_N; r += GKM_MMA_BUILDERS) {
                const int jj = GKM_MMA_N * nt + r;
                const bool valid = jj < 2 * nkB;
                const int strand = (jj >= nkB) ? 1 : 0;
                const int o = strand * lenB + (jj - strand * nkB);
                uint32_t p0 = 0, p1 = 0;
                if (valid) gkm_lmer_planes(plb, W, o, L, p0, p1);
                gkm_mma_store_row(sBop + (size_t) s * GKM_MMA_N * 64, GKM_MMA_N, r, p0, p1, L, valid, gkm_mma_bias_b(L));
                if (WEIGHTED) sWb[(t & 7) * GKM_MMA_N + r] = valid ? p.wend[(size_t) (col0 + b_l) * 32 * W + o + L - 1] : 0;
            }
            asm volatile("fence.proxy.async.shared::cta;");
            __syncwarp();
            if (lane == 0) gkm_mbar_arrive(&bars->b_full[s]);
        }
    } else if (warp == GKM_MMA_EPI) {
        /* ---- MMA issuer ---- */
        if (lane == 0) {
            /* instruction descriptor (cute::UMMA::InstrDescriptor): D = S32 (2 << 4), A = B = unsigned 8 bit (0),
             * both K-major, N >> 3 at bit 17, M >> 4 at bit 24 */
            const uint32_t idesc = (2u << 4) | ((uint32_t) (GKM_MMA_N >> 3) << 17) | ((uint32_t) (GKM_MMA_M >> 4) << 24);
            int j = 0;
            for (int t = 0; t < NTILES; t++) {
                const int s = t & 1;
                gkm_mbar_wait(&bars->b_full[s], (uint32_t) (t >> 1) & 1u);
                for (int mt = 0; mt < MT; mt++, j++) {
                    const int buf = j & 1;
                    gkm_mbar_wait(&bars->acc_empty[buf], ((uint32_t) (j >> 1) & 1u) ^ 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;");
#pragma unroll
                    for (int ks = 0; ks < 2; ks++) { /* K = 64 bytes = two K = 32 instructions = chunks (2ks, 2ks+1) */
                        const uint64_t adesc = gkm_umma_desc(gkm_smem_u32(sAop + (size_t) mt * GKM_MMA_M * 64 + (size_t) ks * 2 * GKM_MMA_M * 16), GKM_MMA_M, 8);
                        const uint64_t bdesc = gkm_umma_desc(gkm_smem_u32(sBop + (size_t) s * GKM_MMA_N * 64 + (size_t) ks * 2 * GKM_MMA_N * 16), GKM_MMA_N, 8);
                        const uint32_t acc = ks ? 1u : 0u;
                        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                                     "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
                                     :: "r"(tmem_base + (uint32_t) buf * GKM_MMA_N), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u) : "memory");
                    }
                    gkm_umma_commit(&bars->acc_full[buf]);
                }
                gkm_umma_commit(&bars->b_empty[s]); /* arrives once every MMA that read this stage has completed */
            }
        }
        __syncwarp();
    } else if (warp < GKM_MMA_EPI) {
        /* ---- epilogue: thread = one stacked query L-mer (TMEM lane), 64 target L-mers in one load of 32 registers ---- */
        const int thr = L - d; /* matches needed for a hit; the launcher guarantees thr >= 1 */
        const int lane_base = 32 * (warp & 3), col_half = (warp >> 2) * GKM_MMA_CW;
        int j = 0;
        for (int t = 0, b_l = 0; t < NTILES; t++) {
            while (t >= bars->tile0[b_l + 1]) b_l++;
            for (int mt = 0; mt < MT; mt++, j++) {
                const int buf = j & 1;
                const int i = mt * GKM_MMA_M + lane_base + lane;
                gkm_mbar_wait(&bars->acc_full[buf], (uint32_t) (j >> 1) & 1u);
                asm volatile("tcgen05.fence::after_thread_sync;");
                /* one load brings all 64 columns of this warp's group, two adjacent columns per register, before the first
                 * is looked at (four load -> wait -> compare rounds exposed the TMEM latency four times per tile) */
                static_assert(GKM_MMA_NV == 32, "one tcgen05.ld .x32 per tile");
                uint32_t v[GKM_MMA_NV];
                const uint32_t taddr = tmem_base + ((uint32_t) lane_base << 16) + (uint32_t) (buf * GKM_MMA_N + col_half);
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "
                             "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                             "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                               "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                               "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                               "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                             : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                /* the accumulator is in registers: hand it back to the MMA warp before the compares */
                asm volatile("tcgen05.fence::before_thread_sync;");
                __syncwarp();
                if (lane == 0) gkm_mbar_arrive(&bars->acc_empty[buf]);
                /* what a hit costs is paid only by a hit: the row's query, weight and histogram are looked up here.  The
                 * warps of one column group share a histogram set. */
                auto hit = [&](int col, int matches) {
                    const int q = sRowQ[i];
                    int32_t *Hq = sH + ((((warp >> 2) * GKM_MMA_QA) + (q & 3)) * GKM_MMA_TB + b_l) * NBN;
                    atomicAdd(Hq + (L - matches), WEIGHTED ? (int) sWa[i] * (int) sWb[(t & 7) * GKM_MMA_N + col_half + col] : 1);
                };
                /* cheap reject of 16 registers at a time, then the exact bins.  Rows and columns of padding are all-zero
                 * operand rows: accumulator 0, never a hit. */
                if (L <= 15) {
                    /* accumulator = matches + 2^15 - thr (gkm_mma_bias_*): bit 15 marks the hits, an OR tree finds them.
                     * A hit is rare per accumulator (0.12 % at L = 11, d = 3) but not per WARP: one of the 32 lanes has one
                     * in a fifth of the groups, and every lane then walks the slow path.  So the slow path is a second look
                     * at the five partial ORs of the tree (three registers each) and only then at single accumulators. */
                    constexpr uint32_t HB = 0x80008000u;
                    auto look = [&](int r) {
                        const uint32_t x = v[r];
                        if (x & 0x8000u) hit(2 * r, (int) (x & 0x7FFFu) + thr);
                        if (x & 0x80000000u) hit(2 * r + 1, (int) ((x >> 16) & 0x7FFFu) + thr);
                    };
#pragma unroll
                    for (int g = 0; g < GKM_MMA_NV; g += 16) {
                        uint32_t tr[5];
#pragma unroll
                        for (int k = 0; k < 5; k++) tr[k] = v[g + 3 * k] | v[g + 3 * k + 1] | v[g + 3 * k + 2];
                        const uint32_t o = (tr[0] | tr[1] | tr[2]) | (tr[3] | tr[4] | v[g + 15]);
                        if (o & HB) {
#pragma unroll
                            for (int k = 0; k < 5; k++)
                                if (tr[k] & HB) {
#pragma unroll
                                    for (int u = 0; u < 3; u++) look(g + 3 * k + u);
                                }
                            look(g + 15);
                        }
                    }
                } else {
                    /* L = 16: no spare K byte for the bias; 3-input max tree (VIMNMX3) on the plain match counts */
#pragma unroll
                    for (int g = 0; g < GKM_MMA_NV; g += 16) {
                        int mx = 0;
#pragma unroll
                        for (int u = 0; u < 16; u++) {
                            const uint32_t x = v[g + u];
                            mx = max(mx, max((int) (x & 0xFFFFu), (int) (x >> 16)));
                        }
                        if (mx >= thr) {
#pragma unroll
                            for (int u = 0; u < 16; u++) {
                                const uint32_t x = v[g + u];
                                if ((int) (x & 0xFFFFu) >= thr) hit(2 * (g + u), (int) (x & 0xFFFFu));
                                if ((int) (x >> 16) >= thr) hit(2 * (g + u) + 1, (int) (x >> 16));
                            }
                        }
                    }
                }
            }
        }
    }
    __syncthreads();
    if (tid < GKM_MMA_QA * GKM_MMA_TB) {
        const int q = tid / GKM_MMA_TB, b_l = tid - q * GKM_MMA_TB;
        const int a_g = a0 + q, b_g = col0 + b_l;
        const bool skip = q >= nA || b_l >= nB || (p.mode == GKM_MODE_LOWER && b_g >= a_g);
        int32_t *h0 = sH + (q * GKM_MMA_TB + b_l) * NBN;
        for (int w = 1; w < GKM_MMA_HSETS; w++)
            for (int m = 0; m < NBN; m++) h0[m] += sH[((w * GKM_MMA_QA + q) * GKM_MMA_TB + b_l) * NBN + m];
        if (!skip) gkm_emit_entry(p, a_g, b_g, h0);
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == GKM_MMA_EPI) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "n"(2 * GKM_MMA_N));
}

#endif /* GKM_MMA_KERNEL_CUH_INCLUDED */
