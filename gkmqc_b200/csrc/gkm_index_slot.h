/* gkm_index_slot.h -- the three slot formats of the "index" variant (gkm_index.h), shared verbatim by the sm_100a
 * build and row kernels (gkm_index.cu) and by the CPU emulator in tests/emu (index_emu.cc), so that the encoder and
 * the decoders the device runs are checked against the oracle on a machine without a GPU.  C++ templates: it cannot
 * sit in the C header.
 *
 *   P32  16-byte slots {posting 0, 1, 2, posting 3 | pointer} of 32-bit postings column | weight << 23.
 *   C16  8-byte slots {c0 | c1 << 16, c2 | c3 << 16} of 16-bit columns (unit weights), 0xFFFF = none; five or more
 *        postings: {c0 | c1 << 16, pointer}, columns 2.. in the overflow array as 16-bit entries.
 *   W20  8-byte slots of three 20-bit postings (column : 14 | weight : 6): x = p0 | p1 << 20, y = p1 >> 12 | p2 << 8 |
 *        flags << 28.  Four or more postings: p0 and p1 inline, y bit 31 set, y bits 9..30 = offset of postings 2.. in
 *        the overflow array in 16-byte units (32-bit postings of the P32 format: the walks are shared), y bit 8 =
 *        GKM_IDX_LONG.  A column field of all ones (0x3FFF: blocks hold at most 16 352 columns) fails the range test;
 *        an empty slot is all ones and is told from a pointer by its first column.
 * A pointer is GKM_IDX_PTR | offset in overflow entries | GKM_IDX_LONG for a long list.  Overflow lists are 16-byte
 * aligned and padded with at least one end marker up to a whole 16-byte unit; long lists start with a header unit
 * {units, 0, 0, 0}.  An end marker, like an empty slot, has an all-ones column, which fails every range test.
 *
 * Writes go through a store policy ST: ST::st(p, v) stores a 16- or 32-bit word, ST::and_(p, v) ANDs into a 32-bit
 * word (a W20 slot is shared by the threads of up to three postings).  The table starts as all ones.  Reads call
 * hit(i, v) for every posting in the wanted columns [blo, bhi), i = column - blo (RANGE) or column (!RANGE); the
 * callback decides where the count goes.
 */
#ifndef GKM_INDEX_SLOT_H_INCLUDED
#define GKM_INDEX_SLOT_H_INCLUDED

#include "gkm_index.h"

/* entries of one 16-byte overflow unit: 16-bit columns (C16) or 32-bit postings (P32, W20) */
GKM_IDX_HD uint32_t gkm_idx_unit_entries(int fmt) { return fmt == GKM_IDX_FMT_C16 ? 8u : 4u; }

/* the 32-bit word where the overflow unit that starts at entry ofs begins */
GKM_IDX_HD uint32_t gkm_idx_unit_word(int fmt, uint32_t ofs) { return fmt == GKM_IDX_FMT_C16 ? ofs >> 1 : ofs; }

/* overflow units of a run of len postings, end marker included, header unit not: P32 keeps postings 3.. of a run
 * of five or more, C16 columns 2.. of five or more, W20 postings 2.. of four or more */
GKM_IDX_HD uint32_t gkm_idx_ovf_units(int fmt, uint32_t len)
{
    if (fmt == GKM_IDX_FMT_C16) return len >= 5 ? (len - 2u + 8u) >> 3 : 0u;
    if (fmt == GKM_IDX_FMT_W20) return len >= 4 ? (len - 2u + 4u) >> 2 : 0u;
    return len >= 5 ? (len - 3u + 4u) >> 2 : 0u;
}

/* overflow entries a run of len postings needs, the header unit of a long list included */
GKM_IDX_HD uint32_t gkm_idx_ovf_need(int fmt, uint32_t len)
{
    const uint32_t units = gkm_idx_ovf_units(fmt, len);
    return gkm_idx_unit_entries(fmt) * (units + (units >= GKM_IDX_LONG_UNITS ? 1u : 0u));
}

/* Posting r of a run of len postings (columns ascending) whose overflow list starts at entry ofs (the exclusive sum of
 * gkm_idx_ovf_need over the runs before it): writes it into the slot (its 32-bit words) or the overflow array ovf.  The
 * head of the run (r == 0) also writes the pointer, the header unit of a long list and the end markers. */
template <int FMT, class ST>
GKM_IDX_HD void gkm_idx_place(uint32_t r, uint32_t len, uint32_t ofs, uint32_t col, uint32_t wt, uint32_t *slot, uint32_t *ovf)
{
    constexpr bool C16 = FMT == GKM_IDX_FMT_C16, W20 = FMT == GKM_IDX_FMT_W20;
    constexpr uint32_t K = FMT == GKM_IDX_FMT_P32 ? 3u : 2u; /* postings kept inline by a list that overflows */
    uint16_t *o16 = reinterpret_cast<uint16_t *>(ovf);
    const uint32_t units = gkm_idx_ovf_units(FMT, len);
    const bool lng = units >= GKM_IDX_LONG_UNITS;
    const uint32_t data = ofs + (lng ? gkm_idx_unit_entries(FMT) : 0u); /* behind the header unit */
    if (C16) col &= GKM_IDX_C16_MAX_COLS;
    if (W20) col &= GKM_IDX_W20_COL_MASK;
    const uint32_t p20 = col | (wt << GKM_IDX_W20_COL_BITS);
    if (units && r >= K) {
        if constexpr (C16) ST::st(o16 + data + r - K, (uint16_t) col);
        else ST::st(ovf + data + r - K, gkm_idx_posting(col, wt));
    } else if constexpr (C16) {
        ST::st(reinterpret_cast<uint16_t *>(slot) + r, (uint16_t) col);
    } else if constexpr (W20) {
        if (r == 0) {
            ST::and_(slot, p20 | ~0xFFFFFu);
            if (!units) ST::and_(slot + 1, ~GKM_IDX_PTR);
        } else if (r == 1) {
            ST::and_(slot, (p20 << 20) | 0xFFFFFu);
            ST::and_(slot + 1, (p20 >> 12) | ~0xFFu);
        } else {
            ST::and_(slot + 1, (p20 << 8) | ~(0xFFFFFu << 8));
        }
    } else {
        ST::st(slot + r, gkm_idx_posting(col, wt));
    }
    if (r != 0 || !units) return;
    if constexpr (W20) ST::and_(slot + 1, GKM_IDX_PTR | ((ofs >> 2) << 9) | (lng ? (GKM_IDX_LONG << 8) : 0u) | 0xFFu);
    else ST::st(slot + (C16 ? 1 : 3), GKM_IDX_PTR | ofs | (lng ? GKM_IDX_LONG : 0u));
    if (lng) {
        uint32_t *h = ovf + gkm_idx_unit_word(FMT, ofs);
        ST::st(h, units); ST::st(h + 1, 0u); ST::st(h + 2, 0u); ST::st(h + 3, 0u);
    }
    for (uint32_t t = len - K; t < gkm_idx_unit_entries(FMT) * units; t++) { /* lists are read 16 bytes at a time */
        if constexpr (C16) ST::st(o16 + data + t, (uint16_t) GKM_IDX_C16_NONE);
        else ST::st(ovf + data + t, GKM_IDX_EMPTY);
    }
}

/* One column against the wanted range [blo, bhi).  (ptxas turns a predicated red.shared back into a branch around
 * ATOMS, so this is plain C++.) */
template <bool RANGE, class HIT>
GKM_IDX_HD void gkm_idx_hit(uint32_t b, uint32_t blo, uint32_t bhi, int v, const HIT &hit)
{
    bool ok = b < bhi;
    if (RANGE) ok = ok && b >= blo;
    if (ok) hit(RANGE ? b - blo : b, v);
}

/* one 32-bit posting, its weight times the query's w */
template <bool WEIGHTED, bool RANGE, class HIT>
GKM_IDX_HD void gkm_idx_hit32(uint32_t e, uint32_t blo, uint32_t bhi, int w, const HIT &hit)
{
    gkm_idx_hit<RANGE>(e & GKM_IDX_COL_MASK, blo, bhi, WEIGHTED ? w * (int) (e >> GKM_IDX_COL_BITS) : 1, hit);
}

/* The inline postings of the slot {s0, s1, s2, s3} (8-byte slots: s0, s1).  Returns the offset of the overflow list
 * that still has to be walked (| GKM_IDX_LONG), or ~0u.  Lists are sorted by column, so a list whose last inline
 * posting is behind the range needs no walk. */
template <int FMT, bool WEIGHTED, bool RANGE, class HIT>
GKM_IDX_HD uint32_t gkm_idx_slot(uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t blo, uint32_t bhi, int w, const HIT &hit)
{
    if constexpr (FMT == GKM_IDX_FMT_C16) {
        const uint32_t c1 = s0 >> 16, c3 = s1 >> 16;
        gkm_idx_hit<RANGE>(s0 & 0xFFFFu, blo, bhi, 1, hit);
        gkm_idx_hit<RANGE>(c1, blo, bhi, 1, hit);
        if (!(s1 & GKM_IDX_PTR) || c3 == GKM_IDX_C16_NONE) {
            gkm_idx_hit<RANGE>(s1 & 0xFFFFu, blo, bhi, 1, hit);
            gkm_idx_hit<RANGE>(c3, blo, bhi, 1, hit);
            return ~0u;
        }
        return (c1 < bhi) ? (s1 & ~GKM_IDX_PTR) : ~0u;
    } else if constexpr (FMT == GKM_IDX_FMT_W20) {
        const uint32_t p0 = s0 & 0xFFFFFu, p1 = (s0 >> 20) | ((s1 & 0xFFu) << 12);
        const uint32_t c0 = p0 & GKM_IDX_W20_COL_MASK, c1 = p1 & GKM_IDX_W20_COL_MASK;
        gkm_idx_hit<RANGE>(c0, blo, bhi, w * (int) (p0 >> GKM_IDX_W20_COL_BITS), hit);
        gkm_idx_hit<RANGE>(c1, blo, bhi, w * (int) (p1 >> GKM_IDX_W20_COL_BITS), hit);
        if (!(s1 & GKM_IDX_PTR) || c0 == GKM_IDX_W20_COL_MASK) {
            const uint32_t p2 = (s1 >> 8) & 0xFFFFFu;
            gkm_idx_hit<RANGE>(p2 & GKM_IDX_W20_COL_MASK, blo, bhi, w * (int) (p2 >> GKM_IDX_W20_COL_BITS), hit);
            return ~0u;
        }
        return (c1 < bhi) ? ((((s1 >> 9) & 0x3FFFFFu) << 2) | ((s1 >> 8) & GKM_IDX_LONG)) : ~0u;
    } else {
        gkm_idx_hit32<WEIGHTED, RANGE>(s0, blo, bhi, w, hit);
        gkm_idx_hit32<WEIGHTED, RANGE>(s1, blo, bhi, w, hit);
        gkm_idx_hit32<WEIGHTED, RANGE>(s2, blo, bhi, w, hit);
        if (!(s3 & GKM_IDX_PTR)) { gkm_idx_hit32<WEIGHTED, RANGE>(s3, blo, bhi, w, hit); return ~0u; }
        return (s3 != GKM_IDX_EMPTY && (s2 & GKM_IDX_COL_MASK) < bhi) ? (s3 & ~GKM_IDX_PTR) : ~0u;
    }
}

/* The hits of one 16-byte overflow unit {u0, u1, u2, u3}: eight 16-bit columns (C16) or four 32-bit postings (P32, and
 * the overflow of W20).  Returns false where the list ends: its last column is behind the range (an end marker is). */
template <int FMT, bool WEIGHTED, bool RANGE, class HIT>
GKM_IDX_HD bool gkm_idx_unit(uint32_t u0, uint32_t u1, uint32_t u2, uint32_t u3, uint32_t blo, uint32_t bhi, int w, const HIT &hit)
{
    if constexpr (FMT == GKM_IDX_FMT_C16) {
        gkm_idx_hit<RANGE>(u0 & 0xFFFFu, blo, bhi, 1, hit); gkm_idx_hit<RANGE>(u0 >> 16, blo, bhi, 1, hit);
        gkm_idx_hit<RANGE>(u1 & 0xFFFFu, blo, bhi, 1, hit); gkm_idx_hit<RANGE>(u1 >> 16, blo, bhi, 1, hit);
        gkm_idx_hit<RANGE>(u2 & 0xFFFFu, blo, bhi, 1, hit); gkm_idx_hit<RANGE>(u2 >> 16, blo, bhi, 1, hit);
        gkm_idx_hit<RANGE>(u3 & 0xFFFFu, blo, bhi, 1, hit); gkm_idx_hit<RANGE>(u3 >> 16, blo, bhi, 1, hit);
        return (u3 >> 16) < bhi;
    } else {
        gkm_idx_hit32<WEIGHTED, RANGE>(u0, blo, bhi, w, hit);
        gkm_idx_hit32<WEIGHTED, RANGE>(u1, blo, bhi, w, hit);
        gkm_idx_hit32<WEIGHTED, RANGE>(u2, blo, bhi, w, hit);
        gkm_idx_hit32<WEIGHTED, RANGE>(u3, blo, bhi, w, hit);
        return (u3 & GKM_IDX_COL_MASK) < bhi;
    }
}

/* The same unit of a long list, whose lanes walk a unit each: equal columns are adjacent in a list (a column with a
 * repeat owns a run of postings), so the runs inside the unit are folded into one hit each and a homopolymer costs
 * one atomic per unit instead of eight on one address.  Returns false where nothing in this unit or behind it is
 * wanted (its first column is behind the range). */
template <int FMT, bool WEIGHTED, bool RANGE, class HIT>
GKM_IDX_HD bool gkm_idx_unit_folded(uint32_t u0, uint32_t u1, uint32_t u2, uint32_t u3, uint32_t blo, uint32_t bhi, int w, const HIT &hit)
{
    if constexpr (FMT == GKM_IDX_FMT_C16) {
        uint32_t cur = u0 & 0xFFFFu;
        if (cur >= bhi) return false;
        int cnt = 1;
        const uint32_t c[7] = { u0 >> 16, u1 & 0xFFFFu, u1 >> 16, u2 & 0xFFFFu, u2 >> 16, u3 & 0xFFFFu, u3 >> 16 };
#pragma unroll
        for (int t = 0; t < 7; t++) {
            if (c[t] == cur) cnt++;
            else { gkm_idx_hit<RANGE>(cur, blo, bhi, cnt, hit); cur = c[t]; cnt = 1; }
        }
        gkm_idx_hit<RANGE>(cur, blo, bhi, cnt, hit);
    } else {
        uint32_t cur = u0 & GKM_IDX_COL_MASK;
        if (cur >= bhi) return false;
        int acc = WEIGHTED ? w * (int) (u0 >> GKM_IDX_COL_BITS) : 1;
        const uint32_t e[3] = { u1, u2, u3 };
#pragma unroll
        for (int t = 0; t < 3; t++) {
            const uint32_t col = e[t] & GKM_IDX_COL_MASK;
            const int val = WEIGHTED ? w * (int) (e[t] >> GKM_IDX_COL_BITS) : 1;
            if (col == cur) acc += val;
            else { gkm_idx_hit<RANGE>(cur, blo, bhi, acc, hit); cur = col; acc = val; }
        }
        gkm_idx_hit<RANGE>(cur, blo, bhi, acc, hit);
    }
    return true;
}

#endif /* GKM_INDEX_SLOT_H_INCLUDED */
