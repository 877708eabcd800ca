/* gkm_lmer_subst.h -- the arithmetic of single-base substitutions scored through the L-mer table (DESIGN.md 4.6).
 *
 * The score of a row r (gkm_lmer_table.h) is (sum_{x forward window of r} wt(x) T[code(x)]) / |r| with
 *   |r| = sqrt(sum_m w[m] H_m(r, r)),   H_m(r, r) = sum_{x fwd} sum_{y fwd or rc} wt(x) wt(y) [ham(x, y) = m].
 * Replacing base p of r by v changes only the forward windows Cx that cover p and the reverse-complement windows that
 * cover rc position len - 1 - p; C = both sets.  Weights do not change.  Every value here equals, bit for bit, what the
 * upload and gkm_lt_score_kernel compute for the materialised mutant:
 *
 *   dH.  The pairs whose Hamming distance can change are (x in Cx, any y) and (x not in Cx, y in C).  The rc window s is
 *        the reverse complement of forward window n - 1 - s with the same weight, and ham(x, rc y) = ham(rc x, y), so the
 *        second set contributes what (x in Cx, y not in C) does.  Hence dH = 2 A + B with
 *          A = sum_{x in Cx, y not in C} (new - old),   B = sum_{x in Cx, y in C} (new - old).
 *        In A only bit t = p - i of the mismatch mask of x = window i moves: ham' = popc(mask & ~bit t) + [v != y_t].
 *        So A needs, per site, old[m] (v-independent) and Q_v[m] = 2 sum_{y_t = v} wt wt [popc(mask & ~bit t) = m]:
 *          A_v[m] = Q_v[m] + (P[m - 1] - Q_v[m - 1]) - old[m],   P = Q_0 + Q_1 + Q_2 + Q_3.
 *        In B both windows moved (the window itself, overlapping windows, palindromes): both are rebuilt, ham' recomputed.
 *        A pair with popc(mask) > d + 1 has ham and ham' above d and is skipped.  All sums are 32-bit two's complement,
 *        so H' = H + dH is the upload's 32-bit histogram even where M = 255 wraps it.
 *   norm sqrt(sum_m w[m] H'_m), m ascending from 0.0, one rounding per operation: gkm_kraw and __dsqrt_rn.
 *   num  gkm_lt_score_kernel's sum by ascending window: the row's own prefix sum up to the first window of Cx, then the
 *        new terms of Cx (one table read each), then the row's later terms (wt, T[code]) one by one.
 *
 * Windows are those of the packed image's circular string (gkm_seq.c): forward window i starts at bit i, rc window s at
 * bit len + s; bit t of a plane window is base t of the window (the code bits gkm_idx_base_bit names).  The sm_100a
 * kernel (gkm_lmer_table.cu) and the CPU emulator (tests/emu/lmer_subst_emu.cc) include this header verbatim.
 */
#ifndef GKM_LMER_SUBST_H_INCLUDED
#define GKM_LMER_SUBST_H_INCLUDED

#include <stdint.h>

#include "gkm_lmer_table.h"

#if defined(__CUDA_ARCH__)
#define GKM_LS_SQRT(a) __dsqrt_rn(a)
#define GKM_LS_POPC(a) __popc(a)
#define GKM_LS_LDG(a) __ldg(a)
#else
#include <math.h>
#define GKM_LS_SQRT(a) sqrt(a) /* correctly rounded (IEEE 754) */
#define GKM_LS_POPC(a) __builtin_popcount(a)
#define GKM_LS_LDG(a) (*(a))
#endif

/* histogram bins per site: old, Q_0..Q_3 and B_0..B_3 (new part of B per base), each d + 1 <= 17 bins */
#define GKM_LS_NB 17
#define GKM_LS_OLD 0
#define GKM_LS_Q(v) (1 + (v))
#define GKM_LS_B(v) (5 + (v))
#define GKM_LS_ACC (9 * GKM_LS_NB)

/* the changed windows of a substitution at p of a row of len bases, n = len - L + 1 windows per strand: forward windows
 * i in [*flo, *fhi] (offset p - i) and rc windows s in [*rlo, *rhi] (offset len - 1 - p - s, base v ^ 3) */
GKM_LT_HD void gkm_ls_changed(int p, int len, int L, int *flo, int *fhi, int *rlo, int *rhi)
{
    const int n = len - L + 1, q = len - 1 - p;
    *flo = p - L + 1 > 0 ? p - L + 1 : 0;
    *fhi = p < n - 1 ? p : n - 1;
    *rlo = q - L + 1 > 0 ? q - L + 1 : 0;
    *rhi = q < n - 1 ? q : n - 1;
}

/* base t of a window given as two planes */
GKM_LT_HD uint32_t gkm_ls_base(uint32_t x0, uint32_t x1, int t) { return ((x0 >> t) & 1u) | (((x1 >> t) & 1u) << 1); }

/* the window with base t replaced by v */
GKM_LT_HD void gkm_ls_put(uint32_t *x0, uint32_t *x1, int t, uint32_t v)
{
    *x0 = (*x0 & ~(1u << t)) | ((v & 1u) << t);
    *x1 = (*x1 & ~(1u << t)) | ((v >> 1) << t);
}

GKM_LT_HD int gkm_ls_ham(uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1) { return GKM_LS_POPC((x0 ^ y0) | (x1 ^ y1)); }

/* part A, one pair: x = changed forward window (base t moves), y unchanged, ww = wt(x) wt(y).  add(&acc[bin], value):
 * shared atomics on the device, += in the emulator; acc holds GKM_LS_ACC counters */
template <class ADD>
GKM_LT_HD void gkm_ls_pair_a(uint32_t x0, uint32_t x1, uint32_t y0, uint32_t y1, int t, int d, uint32_t ww, const ADD &add, uint32_t *acc)
{
    const uint32_t mask = (x0 ^ y0) | (x1 ^ y1);
    const int h = GKM_LS_POPC(mask);
    if (h > d + 1) return;
    if (h <= d) add(acc + GKM_LS_OLD * GKM_LS_NB + h, 2u * ww);
    const int h0 = h - (int) ((mask >> t) & 1u);
    if (h0 <= d) add(acc + GKM_LS_Q(gkm_ls_base(y0, y1, t)) * GKM_LS_NB + h0, 2u * ww);
}

/* part B, one pair: x = changed forward window (base tx becomes v), y changed too (base ty becomes vy(v): v forward,
 * v ^ 3 reverse complement) */
template <class ADD>
GKM_LT_HD void gkm_ls_pair_b(uint32_t x0, uint32_t x1, int tx, uint32_t y0, uint32_t y1, int ty, uint32_t yflip, int d,
                             uint32_t ww, const ADD &add, uint32_t *acc)
{
    const int h = gkm_ls_ham(x0, x1, y0, y1);
    if (h <= d) add(acc + GKM_LS_OLD * GKM_LS_NB + h, ww);
    for (uint32_t v = 0; v < 4; v++) {
        uint32_t a0 = x0, a1 = x1, b0 = y0, b1 = y1;
        gkm_ls_put(&a0, &a1, tx, v);
        gkm_ls_put(&b0, &b1, ty, v ^ yflip);
        const int hv = gkm_ls_ham(a0, a1, b0, b1);
        if (hv <= d) add(acc + GKM_LS_B(v) * GKM_LS_NB + hv, ww);
    }
}

/* H'_m = H_m + dH_m for base v, m = 0..d (32-bit wrap-around) */
GKM_LT_HD int32_t gkm_ls_hist(const int32_t *H, const uint32_t *acc, uint32_t v, int m)
{
    const uint32_t *q = acc + GKM_LS_Q(v) * GKM_LS_NB;
    uint32_t a = q[m] - acc[GKM_LS_OLD * GKM_LS_NB + m] + acc[GKM_LS_B(v) * GKM_LS_NB + m];
    if (m > 0) a += (acc[GKM_LS_Q(0) * GKM_LS_NB + m - 1] + acc[GKM_LS_Q(1) * GKM_LS_NB + m - 1] + acc[GKM_LS_Q(2) * GKM_LS_NB + m - 1] +
                     acc[GKM_LS_Q(3) * GKM_LS_NB + m - 1]) - q[m - 1];
    return (int32_t) ((uint32_t) H[m] + a);
}

/* |mutant| = sqrt(sum_m w[m] H'_m) in gkm_kraw's order */
GKM_LT_HD double gkm_ls_norm(const int32_t *H, const uint32_t *acc, uint32_t v, int d, const double *w)
{
    double s = 0.0;
    for (int m = 0; m <= d; m++) s = GKM_LT_ADD(s, GKM_LT_MUL(w[m], (double) gkm_ls_hist(H, acc, v, m)));
    return GKM_LS_SQRT(s);
}

/* ---- one site over a row staged as 2n plane windows X0, X1 (forward windows 0..n-1, then rc windows n..2n-1) and their
 * weights WT, the work split over nl lanes (lane = 0..nl-1; the emulator runs nl = 1) ---- */
GKM_LT_HD int gkm_ls_in_c(int k, int n, int flo, int fhi, int rlo, int rhi)
{
    return (k >= flo && k <= fhi) || (k >= n + rlo && k <= n + rhi);
}

/* A: every changed forward window against every unchanged window of either strand */
template <class ADD>
GKM_LT_HD void gkm_ls_site_a(int lane, int nl, const uint32_t *X0, const uint32_t *X1, const uint8_t *WT, int n, int p,
                             int flo, int fhi, int rlo, int rhi, int d, const ADD &add, uint32_t *acc)
{
    for (int k = lane; k < 2 * n; k += nl) {
        if (gkm_ls_in_c(k, n, flo, fhi, rlo, rhi)) continue;
        const uint32_t y0 = X0[k], y1 = X1[k], wy = WT[k];
        for (int i = flo; i <= fhi; i++) gkm_ls_pair_a(X0[i], X1[i], y0, y1, p - i, d, (uint32_t) WT[i] * wy, add, acc);
    }
}

/* the b-th changed window, b < nf + nr: forward window flo + b (base p - i, as is) or rc window rlo + b - nf (base at rc
 * position len - 1 - p, complemented) */
GKM_LT_HD void gkm_ls_partner(int b, int nf, int n, int len, int p, int flo, int rlo, int *k, int *t, uint32_t *flip)
{
    if (b < nf) { *k = flo + b; *t = p - *k; *flip = 0u; }
    else { const int s = rlo + b - nf; *k = n + s; *t = len - 1 - p - s; *flip = 3u; }
}

/* B: every changed forward window against every changed window */
template <class ADD>
GKM_LT_HD void gkm_ls_site_b(int lane, int nl, const uint32_t *X0, const uint32_t *X1, const uint8_t *WT, int n, int len,
                             int p, int flo, int fhi, int rlo, int rhi, int d, const ADD &add, uint32_t *acc)
{
    const int nf = fhi - flo + 1, nc = nf + rhi - rlo + 1;
    for (int j = lane; j < nf * nc; j += nl) {
        const int i = flo + j / nc;
        int k, t;
        uint32_t flip;
        gkm_ls_partner(j % nc, nf, n, len, p, flo, rlo, &k, &t, &flip);
        gkm_ls_pair_b(X0[i], X1[i], p - i, X0[k], X1[k], t, flip, d, (uint32_t) WT[i] * WT[k], add, acc);
    }
}

/* the numerator of base v: PRE[i] = the row's sum of its first i terms, TX[i] = T[code of window i]; T is read for the
 * changed windows only */
GKM_LT_HD double gkm_ls_num(const double *T, const double *PRE, const double *TX, const uint32_t *X0, const uint32_t *X1,
                            const uint8_t *WT, int n, int L, int p, int flo, int fhi, uint32_t v)
{
    double s = PRE[flo];
    for (int i = flo; i <= fhi; i++) {
        uint32_t x0 = X0[i], x1 = X1[i];
        gkm_ls_put(&x0, &x1, p - i, v);
        s = gkm_lt_row_add(s, WT[i], GKM_LS_LDG(T + gkm_idx_code(x0, x1, L)));
    }
    for (int i = fhi + 1; i < n; i++) s = gkm_lt_row_add(s, WT[i], TX[i]);
    return s;
}

#endif /* GKM_LMER_SUBST_H_INCLUDED */
