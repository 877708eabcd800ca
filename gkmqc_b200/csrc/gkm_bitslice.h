/* gkm_bitslice.h -- the bit-sliced "diagonal" formulation of the truncated
 * mismatch histogram, shared verbatim by the sm_100a kernel (gkm_diag_kernel.cuh)
 * and by the CPU lane emulator in tests/emu (which exists so that this arithmetic
 * can be checked against the oracle on a machine without a GPU).
 *
 * Replaces, by a different algorithm, what the reference computes with its k-mer
 * tree DFS (libgkm.c:315-387) and, for the diagonal, with an XOR + byte-table
 * loop (libgkm.c:738-751):  H_m(a,b) = sum over L-mer pairs at Hamming distance
 * m <= d of wt_a * wt_b.
 *
 * Formulation.  The target b is laid out as ONE circular string C of P = 32*Wc
 * positions: forward strand at [0,len), reverse complement at [len,2len), zero
 * padding after it.  Fix query a and a diagonal delta and let
 *     mm_delta[e] = [ a[e] != C[(e + delta) mod P] ]            (one bit)
 * The L-mer pair (window of a ENDING at e, window of C ending at j = e + delta)
 * has Hamming distance  cnt[e] = sum_{t<L} mm_delta[e - t].  One 32-bit word holds
 * 32 consecutive diagonals delta = 32q .. 32q+31 (one word per lane) and the kernel
 * walks e = 0, 1, 2, ...  The count is kept as a bit-sliced RUNNING counter
 * (plane i = bit i of 32 independent counters):
 *     cnt[e] = cnt[e-1] + mm[e] - mm[e-L]
 * i.e. one conditional +-1 per step: x = mm[e] ^ mm[e-L] says "changes",
 * mm[e-L] says "down"; a ripple of  p_i ^= c ; c &= (p_i ^ down)  costs two LOP3
 * per plane -- 8 for L <= 15 -- against a 16-word register ring of past mm words.
 * No shifts are needed for the sum because it slides ACROSS successive words.
 *
 * Each lane serves TWO queries at once: the three sliding bit windows of the
 * target (two code planes and the validity plane E) are extracted once per step
 * with funnel shifts and used for both.
 *
 * Validity: windows that run off either strand, straddle the strand junction or
 * the wrap, or end before position L-1 are removed by AND-ing the hit word with
 *   E[j]   target side bit plane: 1 iff j is a valid window end of either strand
 *   Va[e]  query side, warp-uniform word: all-ones iff L-1 <= e < len_a (only the
 *          first and the last chunks of a query can contain invalid ends, so only
 *          those run the body variant that pays for the AND),
 * so garbage in padding bits can never be counted.
 *
 * Pipe balance (sm_100, measured, DESIGN.md): LOP3/SHF/IADD3 issue at 64
 * lanes/clk/SM on the ALU pipe, IMAD at 64 on the FMA pipe, POPC at 16 on the XU
 * pipe.  The counter is LOP3-only, so the ALU pipe is the bound; the XU pipe comes
 * second.  The unweighted NB = 4 kernel therefore takes its two rarest bins (count
 * <= 1) off the straight-line path (no POPC for them; a loop entered for ~1 % of the
 * warp steps), and so does the unweighted NB = 8 kernel for d = 4 (D4, counts <= 2).
 */
#ifndef GKM_BITSLICE_H_INCLUDED
#define GKM_BITSLICE_H_INCLUDED

#include <stdint.h>
#include <type_traits>

#if defined(__CUDACC__)
#define GKM_HD __host__ __device__ __forceinline__
#define GKM_HDM __host__ __device__ __forceinline__
#else
#define GKM_HD static inline
#define GKM_HDM inline
#endif

/* The instance of the lane code that serves a problem with d mismatches: NB = gkm_diag_nb(d) bins; one instance per
 * (L, NB, WEIGHTED), and for the unweighted NB = 8 problems with d = 4 (the top of the BASELINE sweep) a second one with
 * D4 set.  gkm_diag_instance<NB, WEIGHTED>(d, f) calls f(std::bool_constant<D4>()).  The kernel launcher
 * (gkm_diag_inst.cu) and the CPU emulator both choose through these, so the emulator runs what the device runs. */
constexpr int gkm_diag_nb(int d) { return d < 4 ? 4 : d < 8 ? 8 : 16; }

template <int NB, bool WEIGHTED, class F>
auto gkm_diag_instance(int d, F f)
{
    if constexpr (NB == 8 && !WEIGHTED)
        if (d == 4) return f(std::true_type());
    return f(std::false_type());
}

/* query-side records of a PAIR of queries for one position e (two 16-byte broadcast loads) */
struct alignas(16) gkm_apos2 {
    uint32_t a0[2]; /* [q]: all-ones iff low  bit of base code a_q[e] is 1 */
    uint32_t a1[2]; /* [q]: all-ones iff high bit of base code a_q[e] is 1 */
};
struct alignas(16) gkm_aaux2 {
    uint32_t va[2]; /* [q]: all-ones iff a window of query q may end at e  */
    uint32_t wa[2]; /* [q]: positional weight of the window ending at e    */
};

/* bits [s, s+32) of the 64-bit value hi:lo, 0 <= s < 32 */
GKM_HD uint32_t gkm_funnel(uint32_t lo, uint32_t hi, int s)
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, (uint32_t) s);
#else
    return s ? ((lo >> s) | (hi << (32 - s))) : lo;
#endif
}

GKM_HD int gkm_popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

GKM_HD int gkm_ffs0(uint32_t x) /* index of lowest set bit, x != 0 */
{
#if defined(__CUDA_ARCH__)
    return __ffs((int) x) - 1;
#else
    return __builtin_ctz(x);
#endif
}

constexpr int gkm_nplanes(int maxv) { return maxv >= 16 ? 5 : maxv >= 8 ? 4 : maxv >= 4 ? 3 : maxv >= 2 ? 2 : 1; }

template <int NB> struct gkm_log2nb;
template <> struct gkm_log2nb<4> { static constexpr int v = 2; };
template <> struct gkm_log2nb<8> { static constexpr int v = 3; };
template <> struct gkm_log2nb<16> { static constexpr int v = 4; };

/* ---- per-lane, per-query sliding state ---- */
/* INV = index of a plane that is stored COMPLEMENTED (-1: none).  The rare-bin test needs
 * hit & ~p1; with plane 1 kept inverted that is a plain AND and every other use absorbs the
 * complement into its LOP3 truth table for free. */
template <int L, int INV = -1>
struct gkm_win_state {
    static constexpr int NP = gkm_nplanes(L);
    static constexpr int INVP = INV;
    uint32_t m[16];  /* ring of the last 16 mismatch words */
    uint32_t p[NP];  /* bit-sliced count of mismatches in the current L-window */
    GKM_HDM void clear()
    {
#pragma unroll
        for (int i = 0; i < 16; i++) m[i] = 0u;
#pragma unroll
        for (int i = 0; i < NP; i++) p[i] = (i == INV) ? 0xFFFFFFFFu : 0u;
    }
    GKM_HDM uint32_t plane(int i) const { return i < NP ? (i == INV ? ~p[i] : p[i]) : 0u; }
};

/* push mismatch word `mm` of step S (compile-time ring slot): cnt += mm - mm[e-L] */
template <int L, int INV, int S>
GKM_HD void gkm_win_push(gkm_win_state<L, INV> &st, uint32_t mm)
{
    constexpr int NP = gkm_win_state<L, INV>::NP;
    const uint32_t down = st.m[(S - L) & 15]; /* the position leaving the window (read before the slot is reused) */
    st.m[S & 15] = mm;
    uint32_t c = mm ^ down;                   /* lanes whose count changes */
#pragma unroll
    for (int i = 0; i < NP; i++) {
        const uint32_t t = st.p[i];
        st.p[i] = t ^ c;                      /* same for a complemented plane: ~(x ^ c) = ~x ^ c */
        if (i + 1 < NP) c &= ((i == INV ? ~t : t) ^ down); /* carry when counting up, borrow when counting down */
    }
}

/* bit lanes whose count is < NB, restricted to `valid` */
template <int L, int INV, int LB>
GKM_HD uint32_t gkm_hit_word(const gkm_win_state<L, INV> &st, uint32_t valid)
{
    uint32_t high = 0u;
#pragma unroll
    for (int i = LB; i < gkm_win_state<L, INV>::NP; i++) high |= st.plane(i);
    return valid & ~high;
}

/* mask of bit lanes (within hit) whose count equals V */
template <int L, int INV, int LB, int V>
GKM_HD uint32_t gkm_bin_mask(const gkm_win_state<L, INV> &st, uint32_t hit)
{
    uint32_t r = hit;
#pragma unroll
    for (int i = 0; i < LB; i++) r &= ((V >> i) & 1) ? st.plane(i) : ~st.plane(i);
    return r;
}

template <int L, int INV, int LB, int V0, int V1>
GKM_HD void gkm_bins_popc(const gkm_win_state<L, INV> &st, uint32_t hit, int32_t *acc)
{
    if constexpr (V0 < V1) {
        if constexpr (V0 <= L) acc[V0] += gkm_popc(gkm_bin_mask<L, INV, LB, V0>(st, hit));
        gkm_bins_popc<L, INV, LB, V0 + 1, V1>(st, hit, acc);
    }
}

/* weighted bins: rare path, one (e, j) pair per set bit of `hit` */
template <int L, int INV, int LB>
GKM_HD void gkm_bins_weighted(const gkm_win_state<L, INV> &st, uint32_t hit, uint32_t wa, const uint8_t *wend,
                              int jbase, int P, int32_t *acc)
{
    /* `wend` carries a wrap-around copy of its first 32 bytes behind position P-1, so that
     * jbase + bit (< P + 32) needs no modulo */
    (void) P;
    constexpr int NB = 1 << LB;
    const uint8_t *wj = wend + jbase;
    while (hit) {
        const int bit = gkm_ffs0(hit);
        hit &= hit - 1u;
        int v = 0;
#pragma unroll
        for (int i = 0; i < LB; i++) v |= (int) ((st.plane(i) >> bit) & 1u) << i;
        const int w = (int) wa * (int) wj[bit];
#pragma unroll
        for (int b = 0; b < NB; b++) acc[b] += (v == b) ? w : 0;
    }
}

/* binning of one query at one step */
template <int L, int INV, int NB, bool WEIGHTED, bool D4>
GKM_HD void gkm_bins(const gkm_win_state<L, INV> &st, uint32_t hit, uint32_t wa, const uint8_t *wend,
                     int jbase, int P, int32_t *acc)
{
    constexpr int LB = gkm_log2nb<NB>::v;
    if constexpr (WEIGHTED) {
        gkm_bins_weighted<L, INV, LB>(st, hit, wa, wend, jbase, P, acc);
    } else if constexpr (NB == 4) {
        gkm_bins_popc<L, INV, LB, 2, 4>(st, hit, acc);        /* counts 2 and 3: ~99 % of all hits */
        uint32_t rare = hit & ~st.plane(1);                   /* counts 0 and 1 (plane 1 is stored inverted) */
        if (rare) {
            /* a loop, so that the compiler keeps this off the straight-line path (a real branch,
             * not predication): entered for ~1 % of the warp steps on random sequences */
            do {
                const uint32_t low = rare & (0u - rare);
                rare ^= low;
                if (st.plane(0) & low) acc[1] += 1; else acc[0] += 1;
            } while (rare);
        }
    } else if constexpr (NB == 8 && D4) {
        /* d = 4 known at compile time: counts 5..7 are not wanted at all, 4 and 3 hold ~99 % of the
         * wanted hits, 0..2 take the rare path.  2 POPC per step instead of 8. */
        const uint32_t p0 = st.plane(0), p1 = st.plane(1), p2 = st.plane(2);
        const uint32_t b4 = hit & p2 & ~(p1 | p0);
        const uint32_t low = hit & ~p2;
        const uint32_t b3 = low & p1 & p0;
        uint32_t rare = low & ~(p1 & p0);
        acc[4] += gkm_popc(b4);
        acc[3] += gkm_popc(b3);
        if (rare) {
            do {
                const uint32_t lowbit = rare & (0u - rare);
                rare ^= lowbit;
                if (p1 & lowbit) acc[2] += 1; else if (p0 & lowbit) acc[1] += 1; else acc[0] += 1;
            } while (rare);
        }
    } else {
        gkm_bins_popc<L, INV, LB, 0, NB>(st, hit, acc);
    }
}

/* steps S0..S1-1 of one half chunk (16 positions) for the query pair */
template <int L, int INV, int NB, bool WEIGHTED, bool D4, bool USE_VA, int S0, int S1>
GKM_HD void gkm_diag_steps(gkm_win_state<L, INV> &st0, gkm_win_state<L, INV> &st1,
                           const gkm_apos2 *ap, const gkm_aaux2 *ax,
                           uint32_t lo0, uint32_t hi0, uint32_t lo1, uint32_t hi1, uint32_t loE, uint32_t hiE,
                           const uint8_t *wend, int jbase, int P, int32_t *acc0, int32_t *acc1)
{
    if constexpr (S0 < S1) {
        constexpr int LB = gkm_log2nb<NB>::v;
        const gkm_apos2 a = ap[S0];
        const uint32_t s0 = gkm_funnel(lo0, hi0, S0);
        const uint32_t s1 = gkm_funnel(lo1, hi1, S0);
        const uint32_t ev = gkm_funnel(loE, hiE, S0);
        gkm_win_push<L, INV, S0>(st0, (s0 ^ a.a0[0]) | (s1 ^ a.a1[0]));
        gkm_win_push<L, INV, S0>(st1, (s0 ^ a.a0[1]) | (s1 ^ a.a1[1]));
        uint32_t v0 = ev, v1 = ev, w0 = 1u, w1 = 1u;
        if constexpr (USE_VA || WEIGHTED) {
            const gkm_aaux2 x = ax[S0];
            if constexpr (USE_VA) { v0 &= x.va[0]; v1 &= x.va[1]; }
            w0 = x.wa[0]; w1 = x.wa[1];
        }
        const uint32_t h0 = gkm_hit_word<L, INV, LB>(st0, v0), h1 = gkm_hit_word<L, INV, LB>(st1, v1);
        if (!WEIGHTED || (h0 | h1) != 0u) { /* weighted: ONE divergent region per step for both queries */
            gkm_bins<L, INV, NB, WEIGHTED, D4>(st0, h0, w0, wend, jbase + S0, P, acc0);
            gkm_bins<L, INV, NB, WEIGHTED, D4>(st1, h1, w1, wend, jbase + S0, P, acc1);
        }
        gkm_diag_steps<L, INV, NB, WEIGHTED, D4, USE_VA, S0 + 1, S1>(st0, st1, ap, ax, lo0, hi0, lo1, hi1, loE, hiE,
                                                                 wend, jbase, P, acc0, acc1);
    }
}

/* One lane = one block of 32 diagonals q of one target against a PAIR of queries.
 *   apos/aaux  records of the pair, 32*ceil(max(len0,len1)/32) of each (va = 0 beyond a query's end;
 *              a query of length 0 is a dummy)
 *   C0,C1,E    target bit planes (both strands, circular) and valid-window-end plane, Wc words each
 *   wend       WEIGHTED: target weights by window end position, 32*Wc bytes
 *   acc0/acc1  NB counters per query, added to
 *   D4         unweighted NB = 8 only: d = 4, counts above 4 are not wanted (gkm_diag_instance)        */
template <int L, int NB, bool WEIGHTED, bool D4>
GKM_HD void gkm_diag_lane(const gkm_apos2 *apos, const gkm_aaux2 *aaux, int len0, int len1,
                          const uint32_t *C0, const uint32_t *C1, const uint32_t *E, int Wc, int q,
                          const uint8_t *wend, int32_t *acc0, int32_t *acc1)
{
    constexpr int INV = (!WEIGHTED && NB == 4) ? 1 : -1; /* the rare-bin test of the unweighted NB = 4 kernel wants ~p1 */
    gkm_win_state<L, INV> st0, st1;
    st0.clear();
    st1.clear();
    const int lmax = len0 > len1 ? len0 : len1;
    const int lmin = (len0 > 0 && len1 > 0) ? (len0 < len1 ? len0 : len1) : 0; /* a dummy needs va everywhere */
    const int P = 32 * Wc;
    int k = q;                                   /* word holding stream bits [32(q+c), 32(q+c)+32) */
    int k1 = (k + 1 == Wc) ? 0 : k + 1;
    uint32_t a0 = C0[k], a1 = C1[k], aE = E[k];  /* word k */
    uint32_t b0 = C0[k1], b1 = C1[k1], bE = E[k1];
    const int nhalf = (lmax + 15) >> 4;          /* half chunks of 16 positions */
    int jbase = 32 * q;
#pragma unroll 1
    for (int h = 0; h < nhalf; h += 2) {
        const int k2 = (k1 + 1 == Wc) ? 0 : k1 + 1;
        const uint32_t c0 = C0[k2], c1 = C1[k2], cE = E[k2];
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
            if (h + half >= nhalf) break;
            const int e0 = 16 * (h + half);
            /* stream bits [e0', e0'+64) seen from this lane: aligned words, or words shifted by 16 */
            const uint32_t lo0 = half ? gkm_funnel(a0, b0, 16) : a0, hi0 = half ? gkm_funnel(b0, c0, 16) : b0;
            const uint32_t lo1 = half ? gkm_funnel(a1, b1, 16) : a1, hi1 = half ? gkm_funnel(b1, c1, 16) : b1;
            const uint32_t loE = half ? gkm_funnel(aE, bE, 16) : aE, hiE = half ? gkm_funnel(bE, cE, 16) : bE;
            const bool need_va = (e0 < L - 1) || (e0 + 16 > lmin);
            if (need_va)
                gkm_diag_steps<L, INV, NB, WEIGHTED, D4, true, 0, 16>(st0, st1, apos + e0, aaux + e0, lo0, hi0, lo1, hi1, loE, hiE,
                                                                  wend, jbase, P, acc0, acc1);
            else
                gkm_diag_steps<L, INV, NB, WEIGHTED, D4, false, 0, 16>(st0, st1, apos + e0, aaux + e0, lo0, hi0, lo1, hi1, loE, hiE,
                                                                   wend, jbase, P, acc0, acc1);
            jbase += 16;
            if (jbase >= P) jbase -= P;
        }
        a0 = b0; a1 = b1; aE = bE;
        b0 = c0; b1 = c1; bE = cE;
        k1 = k2;
    }
}

#endif /* GKM_BITSLICE_H_INCLUDED */
