/* gkm_diag_kernel.cuh -- sm_100a kernel "diag": bit-sliced diagonals (see gkm_bitslice.h).
 *
 * Replaces kmertree_dfs + gkmkernel_kernelfunc_batch_single + the normalisation of
 * gkmkernel_kernelfunc_batch_all (libgkm.c:315-387, :553-589, :1156-1185) for a
 * TA x TB tile of (query, target) sequence pairs per CTA.
 *
 * CTA = 256 threads.  Shared memory holds, for the tile,
 *   sAp   [TA/2][32WA] gkm_apos2   records of query PAIRS (one broadcast LDS.128 per step)
 *   sAx   [TA/2][32WA] gkm_aaux2   validity / weight words of the pairs (read by the edge chunks
 *                                   and by the weighted kernel types only)
 *   sS    [TB][3][W]   target bit planes of the circular both-strand string + valid-window-end plane
 *   sW    [TB][32W+32] bytes       target weights by window end + wrap-around copy (weighted types)
 *   sTask [<= TB*W]                lane tasks (target, block of 32 diagonals)
 *   sH    [TA][TB][NB] int32       the tile's histograms
 * A warp takes (query pair, group of 32 tasks) combos round-robin; every lane runs
 * gkm_diag_lane over the two queries, then adds its 2*NB counters into sH with shared
 * atomics (a few per ~10^4 instructions).  The epilogue turns each histogram into
 * the normalised double exactly like the reference does: ascending-m sum from 0.0,
 * one division by sqnorm_a*sqnorm_b, no FMA contraction (libgkm.c:576-582,:1169-1179).
 * Nothing but the 8-byte results (or raw histograms when asked) reaches HBM.
 */
#ifndef GKM_DIAG_KERNEL_CUH_INCLUDED
#define GKM_DIAG_KERNEL_CUH_INCLUDED

#include "gkm_bitslice.h"
#include "gkm_kparams.h"

#define GKM_DIAG_THREADS 256

struct gkm_diag_layout_t {
    unsigned offA, offX, offS, offZ, offW, offTask, offH, offLenA, offLenB, offPre, total;
};

/* W = words per target plane (both strands), WA = 32-position chunks of the longest query, TA even */
__host__ __device__ inline gkm_diag_layout_t gkm_diag_layout(int W, int WA, int TA, int TB, int NB, int weighted)
{
    gkm_diag_layout_t l;
    const unsigned npair = (unsigned) (TA + 1) / 2u;
    unsigned o = 0;
    l.offA = o;    o += npair * 32u * (unsigned) WA * 16u;
    l.offX = o;    o += npair * 32u * (unsigned) WA * 16u;
    l.offS = o;    o += (unsigned) TB * 3u * (unsigned) W * 4u;
    l.offZ = o;    o += (unsigned) W * 4u;
    l.offW = o;    o += weighted ? (unsigned) TB * (32u * (unsigned) W + 32u) : 0u; /* + wrap-around copy of 32 bytes */
    l.offTask = o; o += (unsigned) TB * (unsigned) W * 4u;
    l.offH = o;    o += 2u * npair * (unsigned) TB * (unsigned) NB * 4u;
    l.offLenA = o; o += 2u * npair * 4u;
    l.offLenB = o; o += (unsigned) TB * 4u;
    l.offPre = o;  o += ((unsigned) TB + 1u) * 4u;
    l.total = (o + 15u) & ~15u;
    return l;
}

/* histogram -> kernel value; shared by all kernel variants */
__device__ __forceinline__ double gkm_kraw(const gkm_kparams &p, const int32_t *H)
{
    double sum = 0.0;
    for (int m = 0; m < p.nbins; m++) sum = __dadd_rn(sum, __dmul_rn(p.w[m], (double) H[m]));
    return sum;
}

__device__ __forceinline__ void gkm_emit_entry(const gkm_kparams &p, int a_g, int b_g, const int32_t *H)
{
    if (p.hist) {
        int32_t *dst = p.hist + ((size_t) (a_g - p.row_base) * (size_t) p.hist_cols + (size_t) (b_g - p.col_base)) * (size_t) p.nbins;
        for (int m = 0; m < p.nbins; m++) dst[m] = H[m];
    }
    const double kraw = gkm_kraw(p, H);
    if (p.mode == GKM_MODE_DIAG) {
        if (p.sqnorm_out) p.sqnorm_out[a_g] = __dsqrt_rn(kraw);
        return;
    }
    if (!p.out && !p.decision) return;
    double v = __ddiv_rn(kraw, __dmul_rn(p.sqnorm[a_g], p.sqnorm[b_g]));
    if (p.kernel_type == 3 || p.kernel_type == 5) v = exp(__dmul_rn(p.gamma, __dadd_rn(v, -1.0)));
    if (p.out) p.out[(size_t) (a_g - p.row_base) * (size_t) p.ld + (size_t) (b_g - p.col_base)] = v;
    if (p.decision) atomicAdd(p.decision + (a_g - p.row_base), p.alpha[b_g - p.col_base] * v);
}

template <int L, int NB, bool WEIGHTED, bool D4>
__global__ void __launch_bounds__(GKM_DIAG_THREADS)
gkm_diag_kernel(const __grid_constant__ gkm_kparams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int W = p.W, WA = p.WA, TA = p.TA, TB = p.TB;
    const int NPAIR = (TA + 1) >> 1;
    const gkm_diag_layout_t lay = gkm_diag_layout(W, WA, TA, TB, NB, WEIGHTED ? 1 : 0);
    gkm_apos2 *sAp = reinterpret_cast<gkm_apos2 *>(smem + lay.offA);
    gkm_aaux2 *sAx = reinterpret_cast<gkm_aaux2 *>(smem + lay.offX);
    uint32_t *sS = reinterpret_cast<uint32_t *>(smem + lay.offS);
    uint32_t *sZ = reinterpret_cast<uint32_t *>(smem + lay.offZ);
    uint8_t *sW = smem + lay.offW;
    uint32_t *sTask = reinterpret_cast<uint32_t *>(smem + lay.offTask);
    int32_t *sH = reinterpret_cast<int32_t *>(smem + lay.offH);
    int *sLenA = reinterpret_cast<int *>(smem + lay.offLenA);
    int *sLenB = reinterpret_cast<int *>(smem + lay.offLenB);
    int *sPre = reinterpret_cast<int *>(smem + lay.offPre);

    const int tid = threadIdx.x;
    const int row0 = p.row_begin + (int) blockIdx.y * TA;
    /* sqnorm (GKM_MODE_DIAG) launches ONE column of CTAs: each takes the column tile that holds its rows' diagonal
     * (TB is a multiple of TA, so a row tile never straddles two column tiles) */
    const int col0 = (p.mode == GKM_MODE_DIAG && gridDim.x == 1) ? p.col_begin + ((row0 - p.col_begin) / TB) * TB
                                                                 : p.col_begin + (int) blockIdx.x * TB;
    const int row_last = min(row0 + TA, p.row_end) - 1;
    const int col_last = min(col0 + TB, p.col_end) - 1;
    if (p.mode == GKM_MODE_LOWER && col0 > row_last) return;           /* tile entirely above the diagonal */
    if (p.mode == GKM_MODE_DIAG && (col0 > row_last || col_last < row0)) return;

    /* ---- stage the tile ---- */
    if (tid < 2 * NPAIR) sLenA[tid] = (tid < TA && row0 + tid < p.row_end) ? p.lens[row0 + tid] : 0;
    if (tid < TB) sLenB[tid] = (col0 + tid < p.col_end) ? p.lens[col0 + tid] : 0;
    for (int i = tid; i < W; i += GKM_DIAG_THREADS) sZ[i] = 0u;
    for (int i = tid; i < 2 * NPAIR * TB * NB; i += GKM_DIAG_THREADS) sH[i] = 0;
    for (int i = tid; i < TB * 3 * W; i += GKM_DIAG_THREADS) {
        const int b = i / (3 * W);
        sS[i] = (col0 + b < p.col_end) ? p.planes[(size_t) (col0 + b) * 3 * W + (i - b * 3 * W)] : 0u;
    }
    if (WEIGHTED) {
        const int wordsPerB = 8 * W; /* 32W bytes */
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.wend);
        uint32_t *dst = reinterpret_cast<uint32_t *>(sW);
        for (int i = tid; i < TB * wordsPerB; i += GKM_DIAG_THREADS) {
            const int b = i / wordsPerB;
            dst[b * (wordsPerB + 8) + (i - b * wordsPerB)] =
                (col0 + b < p.col_end) ? src[(size_t) (col0 + b) * wordsPerB + (i - b * wordsPerB)] : 0u;
        }
    }
    __syncthreads();
    if (WEIGHTED) {
        /* wrap-around copy: bytes [P_b, P_b + 32) repeat bytes [0, 32) of target b */
        uint32_t *dst = reinterpret_cast<uint32_t *>(sW);
        for (int i = tid; i < TB * 8; i += GKM_DIAG_THREADS) {
            const int b = i >> 3, k = i & 7;
            const int pw = ((2 * sLenB[b] + 31) >> 5) * 8; /* P_b / 4 words */
            dst[b * (8 * W + 8) + pw + k] = dst[b * (8 * W + 8) + k];
        }
    }
    /* query records, two queries interleaved: the forward strand is the first len bits of the circular string */
    for (int i = tid; i < 2 * NPAIR * 32 * WA; i += GKM_DIAG_THREADS) {
        const int a = i / (32 * WA), e = i - a * 32 * WA;
        const int pi = a >> 1, qi = a & 1;
        uint32_t a0 = 0u, a1 = 0u, va = 0u, wa = 1u;
        if (e < sLenA[a]) {
            const uint32_t *pl = p.planes + (size_t) (row0 + a) * 3 * W;
            a0 = ((pl[e >> 5] >> (e & 31)) & 1u) ? 0xFFFFFFFFu : 0u;
            a1 = ((pl[W + (e >> 5)] >> (e & 31)) & 1u) ? 0xFFFFFFFFu : 0u;
            va = (e >= L - 1) ? 0xFFFFFFFFu : 0u;
            if (WEIGHTED) wa = p.wend[(size_t) (row0 + a) * 32 * W + e];
        }
        gkm_apos2 *rp = sAp + (size_t) pi * 32 * WA + e;
        gkm_aaux2 *rx = sAx + (size_t) pi * 32 * WA + e;
        rp->a0[qi] = a0; rp->a1[qi] = a1;
        rx->va[qi] = va; rx->wa[qi] = wa;
    }
    /* lane tasks: target b contributes ceil(2*len_b/32) blocks of 32 diagonals */
    if (tid == 0) {
        int acc = 0;
        for (int b = 0; b < TB; b++) { sPre[b] = acc; acc += (2 * sLenB[b] + 31) >> 5; }
        sPre[TB] = acc;
    }
    __syncthreads();
    const int ntasks = sPre[TB];
    for (int t = tid; t < ntasks; t += GKM_DIAG_THREADS) {
        int b = 0;
        while (sPre[b + 1] <= t) b++;
        sTask[t] = ((uint32_t) b << 16) | (uint32_t) (t - sPre[b]);
    }
    __syncthreads();

    /* ---- main loop: (query pair, task group) combos ---- */
    const int lane = tid & 31, warp = tid >> 5;
    const int ngroups = (ntasks + 31) >> 5;
    const int ncombos = NPAIR * ngroups;
    for (int combo = warp; combo < ncombos; combo += GKM_DIAG_THREADS / 32) {
        const int pi = combo / ngroups, g = combo - pi * ngroups;
        const int a0_g = row0 + 2 * pi;
        const int len0 = sLenA[2 * pi], len1 = sLenA[2 * pi + 1];
        if (len0 == 0) break;                                     /* past the last row of the block */
        const int a_hi = (len1 > 0) ? a0_g + 1 : a0_g;            /* largest valid row of the pair */
        const int t = 32 * g + lane;
        bool active = t < ntasks;
        const uint32_t task = active ? sTask[t] : 0u;
        const int b_l = (int) (task >> 16), q = (int) (task & 0xFFFFu);
        const int b_g = col0 + b_l;
        if (p.mode == GKM_MODE_LOWER) active = active && (b_g < a_hi);
        if (p.mode == GKM_MODE_DIAG) active = active && (b_g == a0_g || (len1 > 0 && b_g == a0_g + 1));
        if (!__any_sync(0xFFFFFFFFu, active)) continue;

        const uint32_t *C0 = sS + (b_l * 3 + 0) * W;
        const uint32_t *C1 = sS + (b_l * 3 + 1) * W;
        const uint32_t *E = active ? (sS + (b_l * 3 + 2) * W) : sZ;
        const int Wc = active ? ((2 * sLenB[b_l] + 31) >> 5) : 1;
        const uint8_t *wendp = WEIGHTED ? (sW + (size_t) b_l * (32 * W + 32)) : nullptr;

        int32_t acc0[NB], acc1[NB];
#pragma unroll
        for (int m = 0; m < NB; m++) { acc0[m] = 0; acc1[m] = 0; }
        gkm_diag_lane<L, NB, WEIGHTED, D4>(sAp + (size_t) pi * 32 * WA, sAx + (size_t) pi * 32 * WA, len0, len1,
                                           C0, C1, E, Wc, active ? q : 0, wendp, acc0, acc1);
        if (active) {
            int32_t *h0 = sH + ((2 * pi) * TB + b_l) * NB;
            int32_t *h1 = sH + ((2 * pi + 1) * TB + b_l) * NB;
#pragma unroll
            for (int m = 0; m < NB; m++) {
                if (acc0[m]) atomicAdd(h0 + m, acc0[m]);
                if (acc1[m]) atomicAdd(h1 + m, acc1[m]);
            }
        }
    }
    __syncthreads();

    /* ---- epilogue: histogram -> normalised double ---- */
    for (int i = tid; i < TA * TB; i += GKM_DIAG_THREADS) {
        const int a_l = i / TB, b_l = i - a_l * TB;
        const int a_g = row0 + a_l, b_g = col0 + b_l;
        if (a_g >= p.row_end || b_g >= p.col_end) continue;
        if (p.mode == GKM_MODE_LOWER && b_g >= a_g) continue;
        if (p.mode == GKM_MODE_DIAG && b_g != a_g) continue;
        gkm_emit_entry(p, a_g, b_g, sH + (a_l * TB + b_l) * NB);
    }
}

#endif /* GKM_DIAG_KERNEL_CUH_INCLUDED */
