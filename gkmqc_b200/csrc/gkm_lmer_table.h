/* gkm_lmer_table.h -- the arithmetic of the L-mer weight table: a linear gkm-SVM model folded into one weight per L-mer.
 *
 * For the kernel types that are linear in the gkm feature space (0, 1, 2, 4; not the RBF types 3, 5):
 *
 *   f(r) = bias + sum_c alpha_c Kraw(r, c) / (|r| |c|)
 *        = bias + (1 / |r|) sum_{x forward L-mer of r} wt_r(x) T[code(x)]
 *   T[u]   = sum_{m = 0..d} w[m] A_m[u],      A_m[u] = sum_{v : ham(u, v) = m} S[v]
 *   S[v]   = sum_c beta_c sum_{y L-mer of either strand of c, code(y) = v} wt_c(y),   beta_c = alpha_c / |c|
 *
 * The sm_100a kernels (gkm_lmer_table.cu) and the CPU emulator (tests/emu/lmer_table_emu.cc) include this header
 * verbatim, and tests/lmer_table_model.py restates it in numpy: every operation order is fixed here, all of it in
 * round-to-nearest fp64 without FMA, so the three agree bit for bit.
 *
 * Codes are those of gkm_idx_code (gkm_index.h): base t of the window lives in code bits gkm_idx_base_bit(t, L, 0)
 * (its low bit) and gkm_idx_base_bit(t, L, 1) (its high bit), the rule of the index variant's substitution masks.
 */
#ifndef GKM_LMER_TABLE_H_INCLUDED
#define GKM_LMER_TABLE_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#include "gkm_index.h"

/* A (d + 1 planes) and T: (d + 2) 4^L doubles per GPU may not exceed this.  At the cap L = 16 is always refused and
 * L = 15 above d = 0. */
#define GKM_LT_MAX_BYTES ((unsigned long long) 16 << 30)
/* columns one table may fold: the column field of the index keys (code << 32 | column << 8 | weight) has 24 bits */
#define GKM_LT_MAX_COLS (1 << 24)

#if defined(__CUDACC__)
#define GKM_LT_HD __host__ __device__ __forceinline__
#else
#define GKM_LT_HD static inline
#endif
#if defined(__CUDA_ARCH__)
#define GKM_LT_ADD(a, b) __dadd_rn((a), (b))
#define GKM_LT_MUL(a, b) __dmul_rn((a), (b))
#define GKM_LT_DIV(a, b) __ddiv_rn((a), (b))
#else
/* host code is compiled with -ffp-contract=off: one rounding per operation, as on the device */
#define GKM_LT_ADD(a, b) ((a) + (b))
#define GKM_LT_MUL(a, b) ((a) * (b))
#define GKM_LT_DIV(a, b) ((a) / (b))
#endif

/* (d + 2) 4^L doubles: the planes A_0..A_d and T */
GKM_LT_HD unsigned long long gkm_lt_bytes(int L, int d) { return (unsigned long long) (d + 2) << (2 * L + 3); }

/* ---- S ---- */
/* beta_c = alpha_c / |c|, once per column */
GKM_LT_HD double gkm_lt_beta(double alpha, double norm) { return GKM_LT_DIV(alpha, norm); }
/* S[v] starts at 0 and takes s <- s + beta_c * wt for every posting of code v, in the order the stable sort by code leaves
 * them: by column, and inside a column in key-generation order (forward strand, then reverse complement, by window end) */
GKM_LT_HD double gkm_lt_s_add(double s, double beta, uint32_t wt) { return GKM_LT_ADD(s, GKM_LT_MUL(beta, (double) wt)); }

/* ---- the transform: A_0 = S, A_m = 0 for m > 0; then one step per base t = 0 .. L-1 ---- */
/* the codes of group g (0 <= g < 4^(L-1)) for base t: the four codes that differ only in base t, b[v] with value v there */
GKM_LT_HD void gkm_lt_group(uint32_t g, int t, int L, uint32_t b[4])
{
    const int lo = gkm_idx_base_bit(t, L, 0), hi = gkm_idx_base_bit(t, L, 1); /* lo < hi */
    uint32_t c = ((g >> lo) << (lo + 1)) | (g & ((1u << lo) - 1u));            /* a zero at bit lo */
    c = ((c >> hi) << (hi + 1)) | (c & ((1u << hi) - 1u));                      /* and at bit hi */
    for (int v = 0; v < 4; v++) b[v] = c | ((uint32_t) (v & 1) << lo) | ((uint32_t) (v >> 1) << hi);
}

/* one group's step: for m = d down to 1, A_m[b] <- A_m[b] + ((A_{m-1}[b1] + A_{m-1}[b2]) + A_{m-1}[b3]), b1 < b2 < b3 the
 * other three values of the base; every right-hand side is read before this step writes (A is [d + 1][n], n = 4^L) */
GKM_LT_HD void gkm_lt_step(double *A, size_t n, int d, const uint32_t b[4])
{
    double lo[4], cur[4];
    for (int v = 0; v < 4; v++) cur[v] = A[(size_t) d * n + b[v]];
    for (int m = d; m >= 1; m--) {
        for (int v = 0; v < 4; v++) lo[v] = A[(size_t) (m - 1) * n + b[v]];
        for (int v = 0; v < 4; v++) {
            const int v1 = v == 0 ? 1 : 0, v2 = v <= 1 ? 2 : 1, v3 = v <= 2 ? 3 : 2;
            A[(size_t) m * n + b[v]] = GKM_LT_ADD(cur[v], GKM_LT_ADD(GKM_LT_ADD(lo[v1], lo[v2]), lo[v3]));
        }
        for (int v = 0; v < 4; v++) cur[v] = lo[v];
    }
}

/* ---- combine: T[u] = sum_m w[m] A_m[u], m ascending from 0 ---- */
GKM_LT_HD double gkm_lt_combine(const double *A, size_t n, int d, const double *w, uint32_t u)
{
    double t = 0.0;
    for (int m = 0; m <= d; m++) t = GKM_LT_ADD(t, GKM_LT_MUL(w[m], A[(size_t) m * n + u]));
    return t;
}

/* ---- export: lexicographic index (A, C, G, T = 0..3, first base most significant) -> code ---- */
GKM_LT_HD uint32_t gkm_lt_lex_code(uint32_t lex, int L)
{
    uint32_t c = 0;
    for (int t = 0; t < L; t++) {
        const uint32_t v = (lex >> (2 * (L - 1 - t))) & 3u;
        c |= ((v & 1u) << gkm_idx_base_bit(t, L, 0)) | ((v >> 1) << gkm_idx_base_bit(t, L, 1));
    }
    return c;
}

/* ---- the score of a row: s starts at 0 and takes s <- s + wt * T[code] for its forward windows by ascending end
 * position; then one division by |r|.  The bias is added to that quotient, as for the decision values. ---- */
GKM_LT_HD double gkm_lt_row_add(double s, uint32_t wt, double t) { return GKM_LT_ADD(s, GKM_LT_MUL((double) wt, t)); }
GKM_LT_HD double gkm_lt_row_end(double s, double norm) { return GKM_LT_DIV(s, norm); }

#endif /* GKM_LMER_TABLE_H_INCLUDED */
