/* gkm_index.h -- kernel variant "index": inverted L-mer index + neighbour enumeration.
 *
 * Candidate (c) next to the north star's (a) bit-sliced XOR/POPC and (b) tcgen05 one-hot
 * GEMM.  It replaces the same reference code as they do -- kmertree_dfs +
 * gkmkernel_kernelfunc_batch_single (libgkm.c:315-387,:553-589) -- and, like the
 * reference's k-mer tree, avoids touching L-mer pairs that are more than d mismatches
 * apart, but by a different construction that suits the GPU:
 *
 *   target side   every L-mer of both strands of the columns [cb, ce) is a POSTING
 *                 (column - cb, positional weight); postings are sorted by (L-mer,
 *                 column) and laid out in a direct-addressed table of 4^L sixteen-byte
 *                 slots {posting 0, 1, 2, posting 3 | overflow pointer}.  The table
 *                 (67 MB at L = 11) stays in the 126 MB L2.
 *   query side    for every forward L-mer x of row a and every XOR mask `delta` with at
 *                 most d non-zero 2-bit fields (sum_m C(L,m) 3^m of them: 4984 at L=11,
 *                 d=3) the slot of y = x ^ delta is fetched; each posting (b, wt) found
 *                 there is one L-mer pair at Hamming distance m = weight(delta), added as
 *                 wt_a * wt_b to the row histogram H[m][b]: bins d and d-1 (99 % of the hits
 *                 on random sequences) in shared memory, the rarer ones in an L2-resident
 *                 scratch row, so that a block holds twice as many columns.
 *
 * Work per entry is ~290 slot probes + ~200 shared atomics instead of 168 200 pair
 * evaluations; the bound is the L1/LSU sector rate of the random slot probes, not the
 * integer pipe (DESIGN.md 4.4).  Counting is exact, so the integer histograms are the
 * same ones the reference's DFS produces.
 *
 * This header holds what host C, the CPU tests and the CUDA code share: the L-mer code,
 * the posting / slot encoding and the delta list.
 */
#ifndef GKM_INDEX_H_INCLUDED
#define GKM_INDEX_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GKM_IDX_MAX_L 14              /* 4^14 slots = 4 GiB; beyond that the variant is refused */
#define GKM_IDX_EMPTY 0xFFFFFFFFu     /* no posting here / end of an overflow list */
#define GKM_IDX_PTR 0x80000000u       /* slot.w: bits 0..30 = offset of postings 3.. in the overflow array */
#define GKM_IDX_COL_BITS 23
#define GKM_IDX_COL_MASK 0x007FFFFFu  /* posting = column | weight << 23, bit 31 clear */
#define GKM_IDX_MAX_COLS 0x007FFFFEu
/* compact slots of the unit-weight kernel types (0..3): 8 bytes = four 16-bit columns {c0, c1, c2, c3}, 0xFFFF = none;
 * five or more postings: {c0, c1, 0x80000000 | offset of columns 2.. in the overflow array (16-bit entries, lists
 * aligned to 16 bytes and padded with 0xFFFF)}.  Columns stay below 0x8000, so bit 31 of the second word set and its
 * upper half not 0xFFFF means "pointer".  Half the table (33.5 MB at L = 11) and 4 slots per 32-byte sector. */
#define GKM_IDX_FMT_P32 0             /* 16-byte slots of 32-bit postings (column | weight << 23) */
#define GKM_IDX_FMT_C16 1
#define GKM_IDX_C16_NONE 0xFFFFu
#define GKM_IDX_C16_MAX_COLS 0x7FFF
/* compact slots of the weighted kernel types (4, 5): 8 bytes = three 20-bit postings (column : 14 | weight : 6) + 4 flag
 * bits; four or more postings: two inline + pointer to 32-bit postings (the P32 entry format) in the overflow array.
 * Needs weights <= 63 (M <= 63; gkmQC's default is 50), <= 16 352 columns per block and < 2^22 overflow units;
 * otherwise the 16-byte slots are used.  Same table size and sector density as C16.  The three formats are written
 * out in gkm_index_slot.h. */
#define GKM_IDX_FMT_W20 2
#define GKM_IDX_W20_COL_BITS 14
#define GKM_IDX_W20_COL_MASK 0x3FFFu
#define GKM_IDX_W20_MAX_COLS 16352
#define GKM_IDX_W20_MAX_WEIGHT 63
#define GKM_IDX_W20_MAX_UNITS (1u << 22)
/* long lists (repeats, homopolymers): an overflow list of GKM_IDX_LONG_UNITS or more 16-byte units is not walked by
 * the lane that met it (one dependent load per unit: a 20 000-posting poly-A list cost that lane ~1 ms, and every
 * third random row meets it) but by its whole warp, a unit per lane.  Such a list starts with a 16-byte header
 * {number of units, 0, 0, 0} and its slot pointer carries GKM_IDX_LONG (lists are 16-byte aligned, so the low
 * bits of the offset are free). */
#define GKM_IDX_LONG 1u
#define GKM_IDX_LONG_UNITS 8u
#define GKM_IDX_HOT_BINS 2            /* bins d and d-1 (99 % of the hits) live in shared memory, the others in L2 */

#if defined(__CUDACC__)
#define GKM_IDX_HD __host__ __device__ __forceinline__
#else
#define GKM_IDX_HD static inline
#endif

/* table address of an L-mer given its two L-bit plane windows (bit t = base t of the window).
 * The first GKM_IDX_LOWB bases occupy the lowest bits, two bits each, so that the L-mers that differ
 * only there share one 128-byte line of the table (16 slots; the four that differ only in base 0
 * share a 32-byte sector); the other bases stay planar. */
#define GKM_IDX_LOWB 2
GKM_IDX_HD int gkm_idx_lowb(int L) { return L < GKM_IDX_LOWB ? L : GKM_IDX_LOWB; }
GKM_IDX_HD uint32_t gkm_idx_code(uint32_t p0, uint32_t p1, int L)
{
    const int lb = gkm_idx_lowb(L);
    uint32_t c = ((p0 >> lb) << (2 * lb)) | ((p1 >> lb) << (L + lb));
    for (int t = 0; t < lb; t++) c |= (((p0 >> t) & 1u) | (((p1 >> t) & 1u) << 1)) << (2 * t);
    return c;
}

/* the code bit that holds bit `hi` (0: the p0 bit, 1: the p1 bit) of base t of the window, in the layout above */
GKM_IDX_HD int gkm_idx_base_bit(int t, int L, int hi)
{
    const int lb = gkm_idx_lowb(L);
    return t < lb ? 2 * t + hi : (hi ? L : lb) + t;
}

GKM_IDX_HD uint32_t gkm_idx_posting(uint32_t col, uint32_t wt) { return col | (wt << GKM_IDX_COL_BITS); }

/* number of XOR masks with at most d substituted bases: sum_{m<=d} C(L,m) 3^m (0 if it overflows 2^31) */
long long gkm_idx_delta_count(int L, int d);

/* the masks, in probe order: out[i] = mask | m << 28.  The masks of the cold bins (m <= d - 2,
 * gkm_idx_cold_count of them) come first; inside each part masks that differ only in the low bases are
 * adjacent (adjacent lanes -> one line of the table), largest groups first.
 * Returns the number written (= gkm_idx_delta_count), or -1. */
long long gkm_idx_deltas(int L, int d, uint32_t *out, long long cap);
long long gkm_idx_cold_count(int L, int d);

/* is the variant applicable at all (table and masks representable)? */
int gkm_idx_supported(int L, int d, int nbins);

/* the slot format of a column block of ncols columns and `postings` postings: C16 for unit weights, W20 for weights
 * where the weights (M), the columns and the overflow units fit, P32 otherwise and whenever `wide` is set */
int gkm_idx_block_fmt(int weighted, int M, int ncols, size_t postings, int wide);

/* rough cost model used by kernel = auto (DESIGN.md 4.4): estimated device milliseconds */
double gkm_idx_cost_ms(int L, int d, int weighted, long long rows, double mean_query_lmers, double col_blocks, long long entries,
                       double mean_pairs_per_entry);
double gkm_diag_cost_ms(int d, int weighted, long long entries, double mean_pairs_per_entry);

#ifdef __cplusplus
}
#endif

#endif /* GKM_INDEX_H_INCLUDED */
