/* tests/emu/lmer_subst_emu.cc -- CPU emulator of the substitution kernel (gkm_lmer_subst.h / gkm_lt_subst_kernel).
 *
 * TEST INFRASTRUCTURE, not a fallback: nothing in the product links it.  It stages each row of the product's own packed
 * image (gkm_seq.c) as the kernel does and runs the header's site functions with one lane.  The self histograms H(r, r)
 * are an input: the device takes them from the upload's diagonal launch.
 */
#include <stdint.h>
#include <vector>

#include "../../gkmqc_b200/csrc/gkm_internal.h"
#include "../../gkmqc_b200/csrc/gkm_lmer_subst.h"

/* idx_window (gkm_index_dev.h) */
static uint32_t window(const uint32_t *pl, int W, int lo, uint32_t mask)
{
    const int w = lo >> 5, s = lo & 31;
    const uint64_t x = pl[w] | ((uint64_t) ((w + 1 < W) ? pl[w + 1] : 0u) << 32);
    return (uint32_t) (x >> s) & mask;
}

struct emu_add {
    void operator()(uint32_t *a, uint32_t v) const { *a += v; }
};

extern "C" {

/* out[4 i + v] = bias + the score of row[i] with base pos[i] replaced by v, through T (code order); H = [n][d + 1] self
 * histograms of the rows; Hout = NULL or [nsites][4][d + 1]: the mutants' histograms H' */
int gkm_emu_lmer_subst(gkmb200_problem *p, const double *T, const int32_t *H, long long nsites, const int *row, const int *pos,
                       double bias, double *out, int32_t *Hout)
{
    if (gkm_pack_problem(p)) return 1;
    const int L = p->param.L, d = p->param.d, W = p->Wmax;
    const uint32_t mask = (1u << L) - 1u;
    std::vector<uint32_t> X0, X1, acc(GKM_LS_ACC);
    std::vector<uint8_t> WT;
    std::vector<double> PRE, TX;
    int staged = -1;
    for (long long i = 0; i < nsites; i++) {
        const int r = row[i], len = p->len[r], n = len - L + 1;
        if (r != staged) {                                                                  /* the CTA's staging */
            const uint32_t *pl = p->planes + (size_t) r * 3 * W;
            X0.assign(2 * n, 0u); X1.assign(2 * n, 0u); WT.assign(2 * n, 1u); TX.assign(n, 0.0); PRE.assign(n + 1, 0.0);
            for (int k = 0; k < 2 * n; k++) {
                const int lo = k < n ? k : len + k - n;
                X0[k] = window(pl, W, lo, mask);
                X1[k] = window(pl + W, W, lo, mask);
                if (p->weighted) WT[k] = p->wend[(size_t) r * 32 * W + lo + L - 1];
                if (k < n) TX[k] = T[gkm_idx_code(X0[k], X1[k], L)];
            }
            double s = 0.0;
            for (int k = 0; k < n; k++) { s = gkm_lt_row_add(s, WT[k], TX[k]); PRE[k + 1] = s; }
            staged = r;
        }
        const int q = pos[i];
        int flo, fhi, rlo, rhi;
        gkm_ls_changed(q, len, L, &flo, &fhi, &rlo, &rhi);
        for (auto &a : acc) a = 0u;
        gkm_ls_site_a(0, 1, X0.data(), X1.data(), WT.data(), n, q, flo, fhi, rlo, rhi, d, emu_add(), acc.data());
        gkm_ls_site_b(0, 1, X0.data(), X1.data(), WT.data(), n, len, q, flo, fhi, rlo, rhi, d, emu_add(), acc.data());
        const int32_t *Hr = H + (size_t) r * (size_t) (d + 1);
        for (uint32_t v = 0; v < 4; v++) {
            if (Hout)
                for (int m = 0; m <= d; m++) Hout[((size_t) i * 4 + v) * (size_t) (d + 1) + m] = gkm_ls_hist(Hr, acc.data(), v, m);
            const double norm = gkm_ls_norm(Hr, acc.data(), v, d, p->w);
            const double num = gkm_ls_num(T, PRE.data(), TX.data(), X0.data(), X1.data(), WT.data(), n, L, q, flo, fhi, v);
            out[4 * i + v] = gkm_lt_row_end(num, norm) + bias;
        }
    }
    return 0;
}

} /* extern "C" */
