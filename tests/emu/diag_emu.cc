/* tests/emu/diag_emu.cc -- CPU lane emulator for the bit-sliced diagonal kernel.
 *
 * TEST INFRASTRUCTURE: runs gkm_bitslice.h (the exact arithmetic the sm_100a kernel
 * executes per lane) serially on the host, over the packed image produced by the
 * product's own packer (gkm_seq.c), so that packing, circular indexing, the running
 * bit-sliced counters, query pairing and the binning can be checked against the
 * oracle in the CPU-only test tier.  It is not a fallback: nothing in the product
 * links it.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../../gkmqc_b200/csrc/gkm_internal.h"
#include "../../gkmqc_b200/csrc/gkm_bitslice.h"

/* the device layer is absent in the emulator build */
extern "C" {
void gkm_dev_release(gkmb200_problem *) {}
}

/* records of the query pair (a0, a1); a1 < 0 = dummy second query */
static void build_records(const gkmb200_problem *p, int L, int a0, int a1,
                          std::vector<gkm_apos2> &apos, std::vector<gkm_aaux2> &aaux, int len[2])
{
    const int W = p->Wmax;
    const int ids[2] = { a0, a1 };
    len[0] = p->len[a0];
    len[1] = a1 >= 0 ? p->len[a1] : 0;
    const int lmax = len[0] > len[1] ? len[0] : len[1];
    const int n = 32 * ((lmax + 31) / 32);
    apos.assign((size_t) n, gkm_apos2());
    aaux.assign((size_t) n, gkm_aaux2());
    for (int q = 0; q < 2; q++) {
        const uint32_t *pa = ids[q] >= 0 ? p->planes + (size_t) ids[q] * 3 * W : NULL;
        const uint8_t *wea = (p->weighted && ids[q] >= 0) ? p->wend + (size_t) ids[q] * 32 * W : NULL;
        for (int e = 0; e < n; e++) {
            const bool in = e < len[q];
            apos[(size_t) e].a0[q] = (in && ((pa[0 * W + (e >> 5)] >> (e & 31)) & 1u)) ? ~0u : 0u;
            apos[(size_t) e].a1[q] = (in && ((pa[1 * W + (e >> 5)] >> (e & 31)) & 1u)) ? ~0u : 0u;
            aaux[(size_t) e].va[q] = (in && e >= L - 1) ? ~0u : 0u;
            aaux[(size_t) e].wa[q] = (in && wea) ? wea[e] : 1u;
        }
    }
}

template <int L, int NB, bool WEIGHTED, bool D4>
static void emu_pair(const gkmb200_problem *p, int a0, int a1, int b, int32_t *H0, int32_t *H1)
{
    const int W = p->Wmax;
    std::vector<gkm_apos2> apos;
    std::vector<gkm_aaux2> aaux;
    int len[2];
    build_records(p, L, a0, a1, apos, aaux, len);
    const int Wc = (2 * p->len[b] + 31) / 32;
    int32_t acc0[NB], acc1[NB];
    for (int m = 0; m < NB; m++) acc0[m] = acc1[m] = 0;
    const uint32_t *pb = p->planes + (size_t) b * 3 * W;
    std::vector<uint8_t> wext; /* target weights with the wrap-around copy of 32 bytes the kernel keeps in smem */
    const uint8_t *we = NULL;
    if (p->weighted) {
        const uint8_t *src = p->wend + (size_t) b * 32 * W;
        wext.assign(src, src + 32 * Wc);
        wext.insert(wext.end(), src, src + 32);
        we = wext.data();
    }
    for (int q = 0; q < Wc; q++)
        gkm_diag_lane<L, NB, WEIGHTED, D4>(apos.data(), aaux.data(), len[0], len[1], pb, pb + W, pb + 2 * W, Wc, q, we, acc0, acc1);
    for (int m = 0; m <= p->param.d; m++) { H0[m] = acc0[m]; if (H1) H1[m] = acc1[m]; }
}

/* the instance the kernel launcher picks for the problem (gkm_diag_nb, gkm_diag_instance) */
template <int L, int NB, bool WEIGHTED>
static int emu_run(const gkmb200_problem *p, int a0, int a1, int b, int32_t *H0, int32_t *H1)
{
    gkm_diag_instance<NB, WEIGHTED>(p->param.d, [&](auto d4) { emu_pair<L, NB, WEIGHTED, decltype(d4)::value>(p, a0, a1, b, H0, H1); });
    return 0;
}

template <int L>
static int emu_dispatch(const gkmb200_problem *p, int a0, int a1, int b, int32_t *H0, int32_t *H1)
{
    const int nb = gkm_diag_nb(p->param.d);
    if (nb == 4) return p->weighted ? emu_run<L, 4, true>(p, a0, a1, b, H0, H1) : emu_run<L, 4, false>(p, a0, a1, b, H0, H1);
    if (nb == 8) return p->weighted ? emu_run<L, 8, true>(p, a0, a1, b, H0, H1) : emu_run<L, 8, false>(p, a0, a1, b, H0, H1);
    return p->weighted ? emu_run<L, 16, true>(p, a0, a1, b, H0, H1) : emu_run<L, 16, false>(p, a0, a1, b, H0, H1);
}

/* histograms of the query pair (a0, a1) against target b; a1 < 0: single query */
extern "C" int gkm_emu_hist_pair(gkmb200_problem *p, int a0, int a1, int b, int32_t *H0, int32_t *H1)
{
    if (gkm_pack_problem(p)) return 1;
    switch (p->param.L) {
#define CASE(x) case x: return emu_dispatch<x>(p, a0, a1, b, H0, H1);
        CASE(2) CASE(3) CASE(4) CASE(5) CASE(6) CASE(7) CASE(8) CASE(9)
        CASE(10) CASE(11) CASE(12) CASE(13) CASE(14) CASE(15) CASE(16)
#undef CASE
        default: return 1;
    }
}

extern "C" int gkm_emu_hist(gkmb200_problem *p, int a, int b, int32_t *H)
{
    return gkm_emu_hist_pair(p, a, -1, b, H, NULL);
}

/* all pairs j <= a of the problem, queries taken two at a time like the kernel does:
 * H[(a*n + j)*(d+1) + m] */
extern "C" int gkm_emu_hist_lower(gkmb200_problem *p, int32_t *H)
{
    const int n = p->n, nb = p->param.d + 1;
    int32_t scratch[16];
    for (int a = 0; a < n; a += 2) {
        const int a1 = (a + 1 < n) ? a + 1 : -1;
        const int top = (a1 >= 0) ? a1 : a;
        for (int b = 0; b <= top; b++) {
            int32_t *h0 = (b <= a) ? H + ((size_t) a * n + b) * nb : scratch;
            int32_t *h1 = (a1 >= 0) ? H + ((size_t) a1 * n + b) * nb : NULL;
            if (gkm_emu_hist_pair(p, a, a1, b, h0, h1)) return 1;
        }
    }
    return 0;
}
