/* gkm_index_host.c -- host logic of the "index" kernel variant (gkm_index.h): the list of
 * XOR masks a query L-mer is probed with, applicability, the slot format of a column block,
 * and the cost model behind kernel = auto.  Pure C, no CUDA: covered by the CPU test tier. */
#include <math.h>

#include "gkm_index.h"

static long long binom(int n, int k)
{
    if (k < 0 || k > n) return 0;
    long long r = 1;
    for (int i = 1; i <= k; i++) r = r * (n - k + i) / i;
    return r;
}

long long gkm_idx_delta_count(int L, int d)
{
    if (L < 1 || d < 0) return 0;
    if (d > L) d = L;
    long long total = 0, p3 = 1;
    for (int m = 0; m <= d; m++) {
        total += binom(L, m) * p3;
        if (total > 0x7FFFFFFFLL) return 0;
        p3 *= 3;
    }
    return total;
}

/* mask of a substitution by XOR value v (1..3) at base t (gkm_idx_code layout) */
static uint32_t sub_mask(int t, int v, int L)
{
    return ((uint32_t) (v & 1) << gkm_idx_base_bit(t, L, 0)) | ((uint32_t) (v >> 1) << gkm_idx_base_bit(t, L, 1));
}

struct emit_ctx {
    uint32_t *out;
    long long n, cap;
    int L, d, lb;
    int m_lo, m_hi; /* only masks with m_lo <= m <= m_hi are emitted in this pass */
};

/* every combination of the low bases with at most `budget` substitutions, in ascending address order */
static void emit_low(struct emit_ctx *c, uint32_t du, int mu, int budget)
{
    const int nlow = 1 << (2 * c->lb);
    for (int low = 0; low < nlow; low++) {
        int ml = 0;
        for (int t = 0; t < c->lb; t++) ml += ((low >> (2 * t)) & 3) != 0;
        if (ml > budget || mu + ml < c->m_lo || mu + ml > c->m_hi) continue;
        if (c->n < c->cap) c->out[c->n] = (du | (uint32_t) low) | ((uint32_t) (mu + ml) << 28);
        c->n++;
    }
}

/* all masks over the upper bases lb..L-1 with exactly `left` more substitutions */
static void rec_upper(struct emit_ctx *c, int first, int left, uint32_t du, int mu)
{
    if (left == 0) { emit_low(c, du, mu, c->d - mu); return; }
    for (int t = first; t <= c->L - left; t++)
        for (int v = 1; v <= 3; v++) rec_upper(c, t + 1, left - 1, du | sub_mask(t, v, c->L), mu);
}

long long gkm_idx_deltas(int L, int d, uint32_t *out, long long cap)
{
    if (L < 1 || L > GKM_IDX_MAX_L || d < 0 || d > 15 || !out) return -1;
    if (d > L) d = L;
    struct emit_ctx c;
    c.out = out; c.n = 0; c.cap = cap; c.L = L; c.d = d; c.lb = gkm_idx_lowb(L);
    /* the masks of the cold bins (m <= d - 2) first, then the others; inside each part the fewest upper
     * substitutions first: those leave the largest groups of low-base variants */
    c.m_lo = 0; c.m_hi = d - GKM_IDX_HOT_BINS;
    if (c.m_hi >= 0)
        for (int mu = 0; mu <= c.m_hi && mu <= L - c.lb; mu++) rec_upper(&c, c.lb, mu, 0u, mu);
    c.m_lo = c.m_hi + 1; c.m_hi = d;
    if (c.m_lo < 0) c.m_lo = 0;
    for (int mu = 0; mu <= d && mu <= L - c.lb; mu++) rec_upper(&c, c.lb, mu, 0u, mu);
    return (c.n <= cap) ? c.n : -1;
}

long long gkm_idx_cold_count(int L, int d)
{
    return d >= GKM_IDX_HOT_BINS ? gkm_idx_delta_count(L, d - GKM_IDX_HOT_BINS) : 0;
}

int gkm_idx_supported(int L, int d, int nbins)
{
    if (L < 2 || L > GKM_IDX_MAX_L) return 0;
    if (d < 0 || d > 15 || nbins != d + 1) return 0;
    const long long nd = gkm_idx_delta_count(L, d);
    return nd > 0 && nd <= (64LL << 20); /* the mask list itself must stay small (256 MB) */
}

int gkm_idx_block_fmt(int weighted, int M, int ncols, size_t postings, int wide)
{
    if (wide) return GKM_IDX_FMT_P32;
    if (!weighted) return ncols <= GKM_IDX_C16_MAX_COLS ? GKM_IDX_FMT_C16 : GKM_IDX_FMT_P32;
    /* the overflow offsets must fit as well: worst case 4/3 overflow entries per posting + padding */
    if (ncols <= GKM_IDX_W20_MAX_COLS && M <= GKM_IDX_W20_MAX_WEIGHT && (4 * postings) / 3 + 64 < 4 * (size_t) GKM_IDX_W20_MAX_UNITS)
        return GKM_IDX_FMT_W20;
    return GKM_IDX_FMT_P32;
}

/* Device-time estimates, fitted to round-1 measurements on one B200 (DESIGN.md 4.4; 300 bp):
 *   L = 11, d = 3: 10 000 rows x 1 block 41.0 ms, 14 144 x 1 block 72.2 ms, 28 288 x 2 blocks 228 ms (compact slots)
 *   -> probes 8.7e11 /s + postings in range 4.1e11 /s, and never faster than the sector rate of the slot probes:
 *      4e11 /s while the table sits in L2 (<= 64 MB), 1.8e11 /s up to 256 MB (L = 12), 0.9e11 /s beyond (L >= 13);
 *      checked against the 15 (L, d) of BASELINE configs[2] at 20 000 sequences (profiles/r1_config3_sweep_20k_index.*);
 *   weighted types (compact 20-bit postings, two loads in flight): 0.86 of that;  build ~1 ms per column block + 0.3 ms + the table memset;
 *   diag  2.94e13 L-mer pairs /s (d <= 3), 2.06e13 (d = 4: 1.6 s per 20k pass in profiles/r1_v9_config3_sweep_20k_auto.log), ~1.2e13 (d <= 7), ~6e12 above; weighted types 0.6 of that. */
double gkm_idx_cost_ms(int L, int d, int weighted, long long rows, double mean_query_lmers, double col_blocks, long long entries,
                       double mean_pairs_per_entry)
{
    const double nd = (double) gkm_idx_delta_count(L, d);
    const double slots = pow(4.0, (double) L);
    const double slot_bytes = weighted ? 16.0 : 8.0;
    const double tab_mb = slots * slot_bytes / 1048576.0;
    const double scale = weighted ? 0.86 : 1.0;
    const double probes = (double) rows * mean_query_lmers * nd * col_blocks;
    const double hits = (double) entries * mean_pairs_per_entry * nd / slots; /* random sequences: P(distance <= d) = nd / 4^L */
    /* postings found per probe: with several per probe the lanes of a warp share their shared atomics and overflow walks
     * (fuller warps), and the hit side runs up to 1.7x faster (round 2: L = 10, d = 4 at 20k, 3.7 hits per probe, 7.4e11
     * hits/s -- the flat round-1 rate sent that problem to the bit-sliced kernel, 1515 against 1089 ms) */
    const double hpp = probes > 0.0 ? hits / probes : 0.0;
    const double hit_rate = 4.1e11 * (hpp <= 1.0 ? 1.0 : hpp >= 3.0 ? 1.7 : 1.0 + 0.35 * (hpp - 1.0));
    double t = probes / (8.7e11 * scale) + hits / (hit_rate * scale);
    const double floor_t = probes / ((tab_mb <= 64.0 ? 4.0e11 : tab_mb <= 256.0 ? 1.8e11 : 0.9e11) * scale);
    if (t < floor_t) t = floor_t;
    return 1e3 * t + 1.0 * col_blocks + 0.3 + slots * slot_bytes / 3e12 * 1e3;
}

double gkm_diag_cost_ms(int d, int weighted, long long entries, double mean_pairs_per_entry)
{
    double rate = (d <= 3) ? 2.94e13 : (d == 4) ? 2.06e13 : (d <= 7) ? 1.2e13 : 6e12;
    if (weighted) rate *= 0.6;
    return 1e3 * (double) entries * mean_pairs_per_entry / rate;
}
