/* tests/emu/index_emu.cc -- CPU emulator of the "index" kernel variant (gkm_index.h / gkm_index.cu).
 *
 * TEST INFRASTRUCTURE, not a fallback: nothing in the product links it.  It runs on the host, over the product's own
 * packed image (gkm_seq.c), the steps of the sm_100a code.  The kernel's own code, shared verbatim:
 *   the slot format of a block         gkm_idx_block_fmt()          (gkm_index_host.c, as ensure_index calls it)
 *   overflow demand of a run           gkm_idx_ovf_need()           (gkm_index_slot.h, as gkm_idx_runs_kernel)
 *   placement of a posting             gkm_idx_place()              (gkm_index_slot.h, as gkm_idx_fill_kernel)
 *   decoding of a slot / overflow unit gkm_idx_slot(), gkm_idx_unit(), gkm_idx_unit_folded()
 *                                                                   (gkm_index_slot.h, as gkm_index_rows_kernel)
 *   the L-mer code and the mask list   gkm_idx_code(), gkm_idx_deltas()
 * Emulation: the key generation (gkm_idx_keys_kernel), a stable sort by code in place of the CUB radix sort, the
 * exclusive sum of the demands (the device's overflow layout), one serial loop over the postings in place of the
 * fill kernel's threads, and serial probes in place of the row kernel's warps and queues, counting into the histogram
 * instead of shared memory.  The slot table is a hash map (4^L slots do not fit a test box at L = 14); a slot that was
 * never written reads as all ones, as the device's table after its memset.
 */
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <unordered_map>
#include <vector>

#include "../../gkmqc_b200/csrc/gkm_internal.h"
#include "../../gkmqc_b200/csrc/gkm_index_slot.h"
#include "../../gkmqc_b200/csrc/gkm_options.h"

struct emu_slot { uint32_t v[4] = { ~0u, ~0u, ~0u, ~0u }; };

/* the fill kernel's stores, one thread after the other */
struct emu_store {
    static void st(uint32_t *p, uint32_t v) { *p = v; }
    static void st(uint16_t *p, uint16_t v) { memcpy(p, &v, sizeof v); } /* halves of 32-bit words */
    static void and_(uint32_t *p, uint32_t v) { *p &= v; }
};

static uint32_t window(const uint32_t *pl, int W, int lo, uint32_t mask)
{
    const int w = lo >> 5, s = lo & 31;
    const uint64_t x = pl[w] | ((uint64_t) ((w + 1 < W) ? pl[w + 1] : 0u) << 32);
    return (uint32_t) (x >> s) & mask;
}

struct emu_index {
    int fmt;
    std::unordered_map<uint32_t, emu_slot> tab;
    std::vector<uint32_t> ovf;
};

template <int FMT>
static void fill(const std::vector<uint64_t> &keys, emu_index &ix)
{
    const size_t P = keys.size();
    std::vector<uint32_t> runlen(P, 0), ofs(P);
    for (size_t i = 0, e; i < P; i = e) {
        for (e = i + 1; e < P && (keys[e] >> 32) == (keys[i] >> 32); e++) {}
        runlen[i] = (uint32_t) (e - i);
    }
    uint32_t total = 0;
    for (size_t i = 0; i < P; i++) { ofs[i] = total; total += gkm_idx_ovf_need(FMT, runlen[i]); }
    /* the device does not clear the overflow array: an entry the placement misses reads as a posting of column 0 */
    ix.ovf.assign(gkm_idx_unit_word(FMT, total), gkm_idx_posting(0, 1));
    for (size_t i = 0, lb = 0; i < P; i++) {
        if (runlen[i]) lb = i;
        gkm_idx_place<FMT, emu_store>((uint32_t) (i - lb), runlen[lb], ofs[lb], (uint32_t) (keys[i] >> 8) & GKM_IDX_COL_MASK,
                                      (uint32_t) keys[i] & 0xFFu, ix.tab[(uint32_t) (keys[i] >> 32)].v, ix.ovf.data());
    }
}

/* index over the columns [cb, ce) */
static void build_index(const gkmb200_problem *p, int cb, int ce, emu_index &ix)
{
    const int L = p->param.L, W = p->Wmax;
    const uint32_t mask = (1u << L) - 1u;
    std::vector<uint64_t> keys;
    for (int g = cb; g < ce; g++) {
        const int len = p->len[g];
        const uint32_t *pl = p->planes + (size_t) g * 3 * W;
        for (int j = 0; j < 2 * len; j++) {
            const int rel = j < len ? j : j - len;
            if (rel < L - 1) continue;
            const uint32_t code = gkm_idx_code(window(pl, W, j - L + 1, mask), window(pl + W, W, j - L + 1, mask), L);
            const uint32_t wt = p->weighted ? p->wend[(size_t) g * 32 * W + j] : 1u;
            keys.push_back(((uint64_t) code << 32) | ((uint64_t) (uint32_t) (g - cb) << 8) | wt);
        }
    }
    std::stable_sort(keys.begin(), keys.end(), [](uint64_t a, uint64_t b) { return (a >> 32) < (b >> 32); });
    ix.fmt = gkm_idx_block_fmt(p->weighted, p->param.M, ce - cb, keys.size(), gkm_opt_index_wide());
    if (ix.fmt == GKM_IDX_FMT_C16) fill<GKM_IDX_FMT_C16>(keys, ix);
    else if (ix.fmt == GKM_IDX_FMT_W20) fill<GKM_IDX_FMT_W20>(keys, ix);
    else fill<GKM_IDX_FMT_P32>(keys, ix);
}

/* H[(b - blo) * nbins + m] += ... for row a against the indexed columns [blo, bhi) (relative) */
template <int FMT, bool WEIGHTED>
static void probe_row(const gkmb200_problem *p, const emu_index &ix, const std::vector<uint32_t> &deltas, int a,
                      uint32_t blo, uint32_t bhi, int32_t *H)
{
    const int L = p->param.L, W = p->Wmax, nb = p->nbins;
    const uint32_t mask = (1u << L) - 1u;
    const uint32_t *pl = p->planes + (size_t) a * 3 * W;
    const int nq = p->len[a] - L + 1;
    const emu_slot empty;
    for (int i = 0; i < nq; i++) {
        const uint32_t x = gkm_idx_code(window(pl, W, i, mask), window(pl + W, W, i, mask), L);
        const int w = WEIGHTED ? p->wend[(size_t) a * 32 * W + i + L - 1] : 1;
        for (uint32_t dl : deltas) {
            const int m = (int) (dl >> 28);
            const auto hit = [&](uint32_t b, int v) { H[(size_t) b * nb + m] += v; };
            const auto it = ix.tab.find(x ^ (dl & 0x0FFFFFFFu));
            const uint32_t *s = it == ix.tab.end() ? empty.v : it->second.v;
            const uint32_t o = gkm_idx_slot<FMT, WEIGHTED, true>(s[0], s[1], s[2], s[3], blo, bhi, w, hit);
            if (o == ~0u) continue;
            const uint32_t *q = ix.ovf.data() + gkm_idx_unit_word(FMT, o & ~GKM_IDX_LONG);
            if (o & GKM_IDX_LONG) { /* idx_walk_long: the units behind the header, one per lane */
                for (uint32_t u = 1; u <= q[0]; u++)
                    if (!gkm_idx_unit_folded<FMT, WEIGHTED, true>(q[4 * u], q[4 * u + 1], q[4 * u + 2], q[4 * u + 3], blo, bhi, w, hit)) break;
            } else {
                while (gkm_idx_unit<FMT, WEIGHTED, true>(q[0], q[1], q[2], q[3], blo, bhi, w, hit)) q += 4;
            }
        }
    }
}

static void probe(const gkmb200_problem *p, const emu_index &ix, const std::vector<uint32_t> &deltas, int a,
                  uint32_t blo, uint32_t bhi, int32_t *H)
{
    if (ix.fmt == GKM_IDX_FMT_C16) probe_row<GKM_IDX_FMT_C16, false>(p, ix, deltas, a, blo, bhi, H);
    else if (ix.fmt == GKM_IDX_FMT_W20) probe_row<GKM_IDX_FMT_W20, true>(p, ix, deltas, a, blo, bhi, H);
    else if (p->weighted) probe_row<GKM_IDX_FMT_P32, true>(p, ix, deltas, a, blo, bhi, H);
    else probe_row<GKM_IDX_FMT_P32, false>(p, ix, deltas, a, blo, bhi, H);
}

extern "C" {

/* how much work the emulation of a problem is: masks x query L-mers */
long long gkm_emu_index_cost(gkmb200_problem *p)
{
    long long nq = 0;
    for (int i = 0; i < p->n; i++) nq += p->len[i] - p->param.L + 1;
    return nq * gkm_idx_delta_count(p->param.L, p->param.d);
}

/* H[(a * n + b) * nbins + m] for b <= a (the diagonal included), the columns cut into blocks of
 * `block_cols` like the product cuts them when a histogram row does not fit shared memory */
int gkm_emu_index_hist_lower(gkmb200_problem *p, int block_cols, int32_t *H)
{
    if (!gkm_idx_supported(p->param.L, p->param.d, p->nbins)) return 2;
    if (gkm_pack_problem(p)) return 1;
    const int n = p->n, nb = p->nbins;
    const long long nd = gkm_idx_delta_count(p->param.L, p->param.d);
    std::vector<uint32_t> deltas((size_t) nd);
    if (gkm_idx_deltas(p->param.L, p->param.d, deltas.data(), nd) != nd) return 1;
    if (block_cols < 1) block_cols = n;
    for (int cb = 0; cb < n; cb += block_cols) {
        const int ce = cb + block_cols < n ? cb + block_cols : n;
        emu_index ix;
        build_index(p, cb, ce, ix);
        for (int a = cb; a < n; a++) {
            const uint32_t bhi = (uint32_t) ((a + 1 < ce ? a + 1 : ce) - cb); /* columns <= a */
            probe(p, ix, deltas, a, 0u, bhi, H + ((size_t) a * n + cb) * nb);
        }
    }
    return 0;
}

/* one rectangular block with a lower column bound inside the index block (the RANGE path of the kernel) */
int gkm_emu_index_hist_rect(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int32_t *H)
{
    if (!gkm_idx_supported(p->param.L, p->param.d, p->nbins)) return 2;
    if (gkm_pack_problem(p)) return 1;
    const int nb = p->nbins;
    const long long nd = gkm_idx_delta_count(p->param.L, p->param.d);
    std::vector<uint32_t> deltas((size_t) nd);
    if (gkm_idx_deltas(p->param.L, p->param.d, deltas.data(), nd) != nd) return 1;
    emu_index ix;
    build_index(p, 0, p->n, ix); /* the whole problem is one block; only [col0, col0 + ncols) is wanted */
    for (int r = 0; r < nrows; r++)
        probe(p, ix, deltas, row0 + r, (uint32_t) col0, (uint32_t) (col0 + ncols), H + (size_t) r * ncols * nb);
    return 0;
}

}
