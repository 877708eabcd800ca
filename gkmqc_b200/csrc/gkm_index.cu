/* gkm_index.cu -- sm_100a kernels of the "index" variant (see gkm_index.h for the idea).
 *
 * Build (once per column block of a problem, a few ms):
 *   gkm_idx_keys_kernel   every valid L-mer window of both strands of the block's columns ->
 *                         64-bit key  code << 32 | column << 8 | weight
 *   cub radix sort        by code, stable: columns stay ascending   [library call, set-up only]
 *   gkm_idx_runs_kernel   run length of every distinct code; overflow demand of runs >= 5
 *   cub exclusive scan    overflow offsets             [library call, set-up only]
 *   gkm_idx_fill_kernel   slots and overflow lists, one posting per thread (formats: gkm_index_slot.h)
 * Hot loop:
 *   gkm_index_rows_kernel one CTA of 1024 threads per query row; histogram row in shared
 *                         memory; fused fp64 epilogue identical to the other variants
 *                         (ascending-m sum, one division, no FMA; libgkm.c:576-582,1169-1179).
 */
#include <cuda_runtime.h>
#include <type_traits>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "gkm_index_dev.h"
#include "gkm_index_slot.h"
#include "gkm_internal.h"

#define GKM_IDX_THREADS 1024
#define GKM_IDX_UNROLL 4
#define GKM_IDX_WUNR 2 /* slot loads in flight per thread of the weighted two-CTA build (A/B: 3, 4) */
#define GKM_IDX_QCAP 64 /* queued overflow walks per warp: < 32 waiting + <= 32 new */
#define GKM_IDX_LQCAP 32 /* long lists waiting for a whole-warp walk, per warp */
/* Problems of several column blocks run two CTAs per SM only while both fit the 196 KB step of the L1/shared split
 * (blocks up to ~10 700 columns): beyond it L1 shrinks to 28 KB, and the two-CTA build then measured 2x SLOWER than
 * one CTA per SM (50k x 50k, 4 blocks of 12 512 columns: 1 300-1 590 ms against 704 ms).  A single block profits from
 * two CTAs up to the 227 KB limit (12 000 columns: 54.9 against 59.6 ms). */
#define GKM_IDX_TWO_SMEM (196u * 1024u)
#define GKM_IDX_SKEW_ONE_CTA 10.0 /* sum len^2 / P of the block: 2.4 on uniform 10k x 300 bp (L = 11), 3 on AT-rich, 6.5 at L = 10, 12.3 at L = 10 with 600-bp
                                      * windows (gkmQC's default: one CTA 220.6 ms, two 227.0), > 100 with 10 % poly-A */
/* queue entry: (list, bin row, weight).  Compact slots: 4 bytes; 16-byte slots: 8 bytes.  The queues are kept small on
 * purpose: at 10 000 columns two CTAs per SM need 2 x (80 KB histogram + queues + query) of shared memory, and
 * every KB beyond 196 KB per SM moves the L1/shared split to its last step (28 KB of L1 instead of 60), which
 * measured 4 % slower (the in-flight slot probes live in L1 lines): tools/ab_variants.sh, DESIGN.md 4.4. */
#define GKM_IDX_QBYTES_FMT(c16) ((GKM_IDX_THREADS / 32) * (GKM_IDX_QCAP + GKM_IDX_LQCAP) * ((c16) ? 4 : 8) + (GKM_IDX_THREADS / 32) * 4)

/* ------------------------------------------------------------------ */
/* build                                                                */
/* ------------------------------------------------------------------ */
template <bool WEIGHTED>
__global__ void __launch_bounds__(128)
gkm_idx_keys_kernel(const uint32_t *__restrict__ planes, const int32_t *__restrict__ lens, const uint8_t *__restrict__ wend,
                    int W, int L, int cb, const uint32_t *__restrict__ offs, unsigned long long *__restrict__ keys)
{
    const int b = (int) blockIdx.x, g = cb + b;
    const int len = lens[g], nk = len - L + 1;
    const uint32_t base = offs[b];
    const uint32_t mask = (L >= 32) ? 0xFFFFFFFFu : ((1u << L) - 1u);
    const uint32_t *pl = planes + (size_t) g * 3 * (size_t) W;
    for (int j = (int) threadIdx.x; j < 2 * len; j += (int) blockDim.x) {
        const int rel = (j < len) ? j : j - len;
        if (rel < L - 1) continue;
        const uint32_t x0 = idx_window(pl, W, j - L + 1, mask), x1 = idx_window(pl + W, W, j - L + 1, mask);
        const uint32_t code = gkm_idx_code(x0, x1, L);
        const uint32_t wt = WEIGHTED ? (uint32_t) wend[(size_t) g * 32 * (size_t) W + (size_t) j] : 1u;
        const uint32_t slot = base + (uint32_t) ((j < len) ? rel - (L - 1) : nk + rel - (L - 1));
        keys[slot] = ((unsigned long long) code << 32) | ((unsigned long long) (uint32_t) b << 8) | (unsigned long long) wt;
    }
}

/* first index in [lo, hi) whose code is > code (keys sorted by code) */
__device__ __forceinline__ uint32_t idx_upper(const unsigned long long *keys, uint32_t lo, uint32_t hi, uint32_t code)
{
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if ((uint32_t) (keys[mid] >> 32) <= code) lo = mid + 1; else hi = mid;
    }
    return lo;
}

/* first index in [lo, hi) whose code is >= code */
__device__ __forceinline__ uint32_t idx_lower(const unsigned long long *keys, uint32_t lo, uint32_t hi, uint32_t code)
{
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if ((uint32_t) (keys[mid] >> 32) < code) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256)
gkm_idx_runs_kernel(const unsigned long long *__restrict__ keys, uint32_t P, int fmt, uint32_t *__restrict__ runlen, uint32_t *__restrict__ need,
                    unsigned long long *__restrict__ sumsq)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t len = 0;
    const uint32_t code = (i < P) ? (uint32_t) (keys[i] >> 32) : 0u;
    if (i < P && (i == 0 || (uint32_t) (keys[i - 1] >> 32) != code)) {
        /* gallop, then bisect: runs are short (mean 1.4 at 10k x 300 bp) but homopolymers make long ones */
        uint32_t lo = i + 1, hi = P, step = 1; /* [i, lo) holds `code`; keys[hi] does not (or hi == P) */
        for (;;) {
            const uint32_t probe = lo + step - 1;
            if (probe >= P) { hi = P; break; }
            if ((uint32_t) (keys[probe] >> 32) != code) { hi = probe; break; }
            lo = probe + 1;
            step <<= 1;
        }
        len = idx_upper(keys, lo, hi, code) - i;
    }
    {   /* sum of squared list lengths of the block: its ratio to P tells uniform input (1 + postings per slot) from
         * input with repeats (one list of 20 000 postings outweighs everything else); one atomic per warp */
        unsigned long long sq = (unsigned long long) len * (unsigned long long) len;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_down_sync(0xFFFFFFFFu, sq, o);
        if ((threadIdx.x & 31u) == 0u && sq) atomicAdd(sumsq, sq);
    }
    if (i >= P) return;
    runlen[i] = len;
    need[i] = gkm_idx_ovf_need(fmt, len);
}

/* the head of the run that holds posting i: gallop back, then bisect */
__device__ __forceinline__ uint32_t idx_run_head(const unsigned long long *keys, const uint32_t *runlen, uint32_t i, uint32_t code)
{
    if (runlen[i] != 0) return i;
    uint32_t hi = i, lo = 0, step = 1; /* [hi, i] holds `code` */
    for (;;) {
        if (hi < step) { lo = 0; break; }
        const uint32_t probe = hi - step;
        if ((uint32_t) (keys[probe] >> 32) != code) { lo = probe + 1; break; }
        hi = probe;
        step <<= 1;
    }
    return idx_lower(keys, lo, hi, code);
}

/* plain stores; the three 20-bit fields of a W20 slot are written by three threads into two 32-bit words: AND */
struct idx_store {
    template <class T> static __device__ __forceinline__ void st(T *p, T v) { *p = v; }
    static __device__ __forceinline__ void and_(uint32_t *p, uint32_t v) { atomicAnd(p, v); }
};

template <int FMT>
__global__ void __launch_bounds__(256)
gkm_idx_fill_kernel(const unsigned long long *__restrict__ keys, uint32_t P, const uint32_t *__restrict__ runlen,
                    const uint32_t *__restrict__ ovfofs, void *__restrict__ tab, uint32_t *__restrict__ ovf)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const unsigned long long key = keys[i];
    const uint32_t code = (uint32_t) (key >> 32), lb = idx_run_head(keys, runlen, i, code);
    uint32_t *slot = reinterpret_cast<uint32_t *>(tab) + (size_t) code * (FMT == GKM_IDX_FMT_P32 ? 4 : 2);
    gkm_idx_place<FMT, idx_store>(i - lb, runlen[lb], ovfofs[lb], (uint32_t) (key >> 8) & GKM_IDX_COL_MASK, (uint32_t) key & 0xFFu, slot, ovf);
}

/* 4^L slots and one spare, always empty: where the probes of lanes that ran out of query L-mers go */
size_t gkm_idx_tab_bytes(int L, int fmt) { return (((size_t) 1 << (2 * L)) + 1) * (fmt == GKM_IDX_FMT_P32 ? sizeof(uint4) : sizeof(uint2)); }

/* overflow demand is at most 2 entries per posting in either format (header unit of the long lists included) */
size_t gkm_idx_ovf_bytes(size_t P, int fmt) { return (2 * P + 16) * (fmt == GKM_IDX_FMT_C16 ? 2 : 4); }

static size_t align256(size_t x) { return (x + 255) & ~(size_t) 255; }

size_t gkm_idx_scratch_bytes(size_t P, int L, size_t *cub_bytes_out)
{
    size_t t1 = 0, t2 = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, t1, (const unsigned long long *) nullptr, (unsigned long long *) nullptr,
                                   (int) P, 32, 32 + 2 * L);
    cub::DeviceScan::ExclusiveSum(nullptr, t2, (const uint32_t *) nullptr, (uint32_t *) nullptr, (int) P);
    const size_t cubb = align256(t1 > t2 ? t1 : t2);
    if (cub_bytes_out) *cub_bytes_out = cubb;
    return 2 * align256(P * 8) + 2 * align256(P * 4) + cubb + 256;
}

/* the scratch of a build: keys as generated | keys sorted | run lengths | overflow demands | cub temporary storage */
struct idx_scratch {
    unsigned long long *keys_a, *keys_b;
    uint32_t *runlen, *need;
    void *cub_tmp;
};

static idx_scratch idx_carve(const gkm_idx_build_args *a)
{
    const size_t P = a->P;
    unsigned char *s = (unsigned char *) a->scratch;
    idx_scratch r;
    r.keys_a = (unsigned long long *) s; s += align256(P * 8);
    r.keys_b = (unsigned long long *) s; s += align256(P * 8);
    r.runlen = (uint32_t *) s; s += align256(P * 4);
    r.need = (uint32_t *) s; s += align256(P * 4);
    r.cub_tmp = s;
    return r;
}

cudaError_t gkm_idx_sort_keys(const gkm_idx_build_args *a, cudaStream_t st, const unsigned long long **sorted)
{
    const idx_scratch sc = idx_carve(a);
    size_t cub_bytes = a->cub_bytes;
    if (a->wend) gkm_idx_keys_kernel<true><<<(unsigned) (a->ce - a->cb), 128, 0, st>>>(a->planes, a->lens, a->wend, a->W, a->L, a->cb, a->offs, sc.keys_a);
    else gkm_idx_keys_kernel<false><<<(unsigned) (a->ce - a->cb), 128, 0, st>>>(a->planes, a->lens, a->wend, a->W, a->L, a->cb, a->offs, sc.keys_a);
    /* the keys are generated in column order and the radix sort is stable: sorting by the code bits alone leaves
     * every run in ascending column order (3 passes instead of 6 at L = 11) */
    *sorted = sc.keys_b;
    return cub::DeviceRadixSort::SortKeys(sc.cub_tmp, cub_bytes, sc.keys_a, sc.keys_b, (int) a->P, 32, 32 + 2 * a->L, st);
}

int gkm_idx_build(const gkm_idx_build_args *a, cudaStream_t st)
{
    const size_t P = a->P;
    if (P == 0 || P > 0x7FFFFFF0u) { gkm_set_error("index block with %zu postings", P); return 1; }
    const idx_scratch sc = idx_carve(a);
    uint32_t *runlen = sc.runlen, *need = sc.need;
    void *cub_tmp = sc.cub_tmp;
    size_t cub_bytes;
    const unsigned long long *sorted;
    cudaError_t e;
    if ((e = cudaMemsetAsync(a->tab, 0xFF, gkm_idx_tab_bytes(a->L, a->fmt), st)) != cudaSuccess) goto fail;
    if ((e = gkm_idx_sort_keys(a, st, &sorted)) != cudaSuccess) goto fail;
    {
        const unsigned blocks = (unsigned) ((P + 255) / 256);
        unsigned long long *sumsq = (unsigned long long *) ((unsigned char *) cub_tmp + a->cub_bytes); /* in the slack behind the cub area */
        if ((e = cudaMemsetAsync(sumsq, 0, sizeof(*sumsq), st)) != cudaSuccess) goto fail;
        gkm_idx_runs_kernel<<<blocks, 256, 0, st>>>(sorted, (uint32_t) P, a->fmt, runlen, need, sumsq);
        if (a->h_sumsq && (e = cudaMemcpyAsync(a->h_sumsq, sumsq, sizeof(*sumsq), cudaMemcpyDeviceToHost, st)) != cudaSuccess) goto fail;
        uint32_t *ovfofs = (uint32_t *) sc.keys_a; /* the unsorted keys are dead now */
        cub_bytes = a->cub_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(cub_tmp, cub_bytes, need, ovfofs, (int) P, st)) != cudaSuccess) goto fail;
        if (a->fmt == GKM_IDX_FMT_C16) gkm_idx_fill_kernel<GKM_IDX_FMT_C16><<<blocks, 256, 0, st>>>(sorted, (uint32_t) P, runlen, ovfofs, a->tab, a->ovf);
        else if (a->fmt == GKM_IDX_FMT_W20) gkm_idx_fill_kernel<GKM_IDX_FMT_W20><<<blocks, 256, 0, st>>>(sorted, (uint32_t) P, runlen, ovfofs, a->tab, a->ovf);
        else gkm_idx_fill_kernel<GKM_IDX_FMT_P32><<<blocks, 256, 0, st>>>(sorted, (uint32_t) P, runlen, ovfofs, a->tab, a->ovf);
    }
    if ((e = cudaGetLastError()) != cudaSuccess) goto fail;
    return 0;
fail:
    gkm_set_error("CUDA: index build: %s", cudaGetErrorString(e));
    return 1;
}

/* ------------------------------------------------------------------ */
/* hot loop                                                             */
/* ------------------------------------------------------------------ */
/* the hit callback of the row kernel: a shared (hot bins) or global (cold bins) atomic into the bin row Hm */
struct idx_add {
    int32_t *Hm;
    __device__ __forceinline__ void operator()(uint32_t i, int v) const { atomicAdd(Hm + i, v); }
};

template <int FMT> using idx_slot_t = std::conditional_t<FMT == GKM_IDX_FMT_P32, uint4, uint2>;

/* inline postings of one slot; returns the offset of the overflow list that still has to be walked, or ~0u */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ uint32_t idx_slot(const idx_slot_t<FMT> sl, int32_t *Hm, uint32_t blo, uint32_t bhi, int w)
{
    if constexpr (FMT == GKM_IDX_FMT_P32) return gkm_idx_slot<FMT, WEIGHTED, RANGE>(sl.x, sl.y, sl.z, sl.w, blo, bhi, w, idx_add{Hm});
    else return gkm_idx_slot<FMT, WEIGHTED, RANGE>(sl.x, sl.y, 0u, 0u, blo, bhi, w, idx_add{Hm});
}

/* the first 16-byte unit of the overflow list at entry ofs (16-bit entries for C16, 32-bit ones otherwise) */
template <int FMT>
__device__ __forceinline__ const uint4 *idx_units(const uint32_t *ovf, uint32_t ofs)
{
    return FMT == GKM_IDX_FMT_C16 ? reinterpret_cast<const uint4 *>(reinterpret_cast<const uint16_t *>(ovf) + ofs)
                                  : reinterpret_cast<const uint4 *>(ovf + ofs);
}

/* one overflow list (lists of five or more: 1.7 % of the slots at 10k x 300 bp) by one lane, 16 bytes at a time; a
 * long one from behind its header unit */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ void idx_walk(const gkm_idx_rowargs &r, uint32_t ofs, bool lng, int32_t *Hm, uint32_t blo, uint32_t bhi, int w)
{
    const uint4 *q = idx_units<FMT>(r.ovf, ofs + (lng ? gkm_idx_unit_entries(FMT) : 0u));
    for (;;) {
        const uint4 v = __ldg(q++);
        if (!gkm_idx_unit<FMT, WEIGHTED, RANGE>(v.x, v.y, v.z, v.w, blo, bhi, w, idx_add{Hm})) break;
    }
}

/* a long list (GKM_IDX_LONG), walked by the whole warp: lane l takes the units l, l + 32, ... */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ void idx_walk_long(const uint32_t *__restrict__ ovf, uint32_t ofs, int32_t *Hm, uint32_t blo, uint32_t bhi, int w, int lane)
{
    const uint4 *q = idx_units<FMT>(ovf, ofs);
    const uint32_t units = __ldg(q).x;
    for (uint32_t u = (uint32_t) lane; u < units; u += 32u) {
        const uint4 v = __ldg(q + 1 + u);
        if (!gkm_idx_unit_folded<FMT, WEIGHTED, RANGE>(v.x, v.y, v.z, v.w, blo, bhi, w, idx_add{Hm})) break;
    }
}

/* queue entries.  o = offset of the overflow list in entries (a multiple of 8 / 4) | GKM_IDX_LONG */
template <bool C16> struct idx_qe;
template <> struct idx_qe<true> {
    typedef uint32_t type; /* offset / 8 : 27 | long : 1 | bin row : 4 */
    static __device__ __forceinline__ type make(uint32_t o, int mrow, int) { return (o >> 3) | ((o & GKM_IDX_LONG) << 27) | ((uint32_t) mrow << 28); }
    static __device__ __forceinline__ uint32_t ofs(type e) { return (e & 0x07FFFFFFu) << 3; }
    static __device__ __forceinline__ bool lng(type e) { return (e >> 27) & 1u; }
    static __device__ __forceinline__ int mrow(type e) { return (int) (e >> 28); }
    static __device__ __forceinline__ int w(type) { return 1; }
    static __device__ __forceinline__ type none() { return 0u; }
};
template <> struct idx_qe<false> {
    typedef uint2 type; /* {offset | long, bin row | weight << 8} */
    static __device__ __forceinline__ type make(uint32_t o, int mrow, int w) { return make_uint2(o, (uint32_t) mrow | ((uint32_t) w << 8)); }
    static __device__ __forceinline__ uint32_t ofs(type e) { return e.x & ~GKM_IDX_LONG; }
    static __device__ __forceinline__ bool lng(type e) { return e.x & GKM_IDX_LONG; }
    static __device__ __forceinline__ int mrow(type e) { return (int) (e.y & 0xFFu); }
    static __device__ __forceinline__ int w(type e) { return (int) (e.y >> 8); }
    static __device__ __forceinline__ type none() { return make_uint2(0u, 0u); }
};

/* the long queue of a warp, one list after the other, each by all 32 lanes */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ void idx_long(const gkm_idx_rowargs &r, const typename idx_qe<FMT == GKM_IDX_FMT_C16>::type *lq, int lqn, int32_t *Hb, int ldh,
                                         uint32_t blo, uint32_t bhi, int lane)
{
    typedef idx_qe<FMT == GKM_IDX_FMT_C16> QE;
    __syncwarp();
    for (int i = 0; i < lqn; i++) {
        const typename QE::type e = lq[i];
        idx_walk_long<WEIGHTED, RANGE, FMT>(r.ovf, QE::ofs(e), Hb + (size_t) QE::mrow(e) * (size_t) ldh, blo, bhi, QE::w(e), lane);
    }
    __syncwarp();
}

/* Probes of the masks [t_begin, t_end) into the COLD bins (global scratch row C; m <= d - 2, ~1 % of the hits and
 * a handful of masks): tiles of <= 1024 masks; inside a tile a thread keeps its mask and walks the query L-mers.
 * A short tile is shared by several "phases" of threads that take interleaved query L-mers.  Overflow lists are
 * walked on the spot, except the long ones (these masks are where a repeat meets itself): a lane parks them in its
 * warp's long queue (shared counter, the lanes are divergent here) and the warp walks them together at the end. */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ void idx_probe_cold(const gkm_idx_rowargs &r, int t_begin, int t_end, const uint32_t *xq, const uint8_t *wq,
                                               int nq, int32_t *C, int ldh, uint32_t blo, uint32_t bhi,
                                               typename idx_qe<FMT == GKM_IDX_FMT_C16>::type *lq, int *lqcnt)
{
    typedef idx_qe<FMT == GKM_IDX_FMT_C16> QE;
    const int tid = (int) threadIdx.x;
    for (int t0 = t_begin; t0 < t_end; t0 += GKM_IDX_THREADS) {
        const int rem = min(GKM_IDX_THREADS, t_end - t0);
        int T = (rem + 31) & ~31;
        if (rem < 32) { T = 1; while (T < rem) T <<= 1; }
        const int nph = GKM_IDX_THREADS / T;
        const int ph = tid / T, tt = tid - ph * T;
        if (ph >= nph || tt >= rem) continue;
        const uint32_t dl = r.deltas[t0 + tt];
        const uint32_t dx = dl & 0x0FFFFFFFu;
        const int mrow = (int) (dl >> 28);
        int32_t *Hm = C + (size_t) mrow * (size_t) ldh;
        for (int xi = ph; xi < nq; xi += nph) {
            const uint32_t y = xq[xi] ^ dx;
            const int w = WEIGHTED ? (int) wq[xi] : 1;
            const uint32_t o = idx_slot<WEIGHTED, RANGE, FMT>(__ldg(reinterpret_cast<const idx_slot_t<FMT> *>(r.tab) + y), Hm, blo, bhi, w);
            if (o == ~0u) continue;
            if (o & GKM_IDX_LONG) {
                const int pos = atomicAdd(lqcnt, 1);
                if (pos < GKM_IDX_LQCAP) { lq[pos] = QE::make(o, mrow, w); continue; }
            }
            idx_walk<WEIGHTED, RANGE, FMT>(r, o & ~GKM_IDX_LONG, o & GKM_IDX_LONG, Hm, blo, bhi, w);
        }
    }
    __syncwarp();
    const int cnt = min(*lqcnt, GKM_IDX_LQCAP);
    if (cnt) idx_long<WEIGHTED, RANGE, FMT>(r, lq, cnt, C, ldh, blo, bhi, tid & 31);
}

/* the queued walks of a warp, one entry per lane that `have`s one.  Short lists: every lane walks its own.  Long
 * lists are only MOVED here, to the warp's long queue lq[0 .. lqn): they are walked by all 32 lanes at the end of
 * the probe iteration (idx_long), where the prefetched slots are dead -- walked here, inside the unrolled probe
 * body, their registers cost the 32-register build spills of exactly those slots (ptxas -v / SASS).  Should the
 * long queue be full, the list is walked like a short one: slow, but only reached by more than 32 long lists in
 * one iteration. */
template <bool WEIGHTED, bool RANGE, int FMT>
__device__ __forceinline__ void idx_drain(const gkm_idx_rowargs &r, typename idx_qe<FMT == GKM_IDX_FMT_C16>::type e, bool have, int32_t *Hb, int ldh,
                                          uint32_t blo, uint32_t bhi, typename idx_qe<FMT == GKM_IDX_FMT_C16>::type *lq, int &lqn, uint32_t lt)
{
    typedef idx_qe<FMT == GKM_IDX_FMT_C16> QE;
    const bool lng = have && QE::lng(e);
    const uint32_t lm = __ballot_sync(0xFFFFFFFFu, lng);
    if (lm && lqn + __popc(lm) <= GKM_IDX_LQCAP) {
        if (lng) lq[lqn + __popc(lm & lt)] = e;
        lqn += __popc(lm);
        have = have && !lng;
    }
    if (have) idx_walk<WEIGHTED, RANGE, FMT>(r, QE::ofs(e), lng, Hb + (size_t) QE::mrow(e) * (size_t) ldh, blo, bhi, QE::w(e));
}

/* Probes of the masks [t_begin, t_end) into the HOT bins (shared memory H; bin row 0 of H holds m = mbase).
 * Same tiling as above, UNR independent slot loads in flight per thread.  Every lane of a warp runs the
 * same iterations (lanes without work probe with an empty column range), so that the overflow lists can be handled
 * at warp level: a lane that meets a list of five or more postings does NOT walk it on the spot -- one walking lane
 * would stall the other 31 behind a dependent load in divergent code, and nearly every warp probe has one -- but
 * pushes (list, bin row, weight) on the warp's queue in shared memory; whenever 32 walks are queued the warp runs
 * them together (idx_drain). */
template <bool WEIGHTED, bool RANGE, int FMT, int UNR>
__device__ __forceinline__ void idx_probe_hot(const gkm_idx_rowargs &r, int t_begin, int t_end, const uint32_t *xq, const uint8_t *wq,
                                              int nq, int32_t *H, int mbase, int ldh, uint32_t blo, uint32_t bhi,
                                              typename idx_qe<FMT == GKM_IDX_FMT_C16>::type *queue)
{
    typedef idx_qe<FMT == GKM_IDX_FMT_C16> QE;
    const int tid = (int) threadIdx.x, lane = tid & 31;
    const uint32_t lt = (1u << lane) - 1u;
    const idx_slot_t<FMT> *__restrict__ tab = reinterpret_cast<const idx_slot_t<FMT> *>(r.tab);
    typename QE::type *lq = queue + GKM_IDX_QCAP; /* long queue of this warp */
    int qn = 0, lqn = 0;                          /* queued walks of this warp (warp-uniform) */
    for (int t0 = t_begin; t0 < t_end; t0 += GKM_IDX_THREADS) {
        const int rem = min(GKM_IDX_THREADS, t_end - t0);
        int T = (rem + 31) & ~31;
        if (rem < 32) { T = 1; while (T < rem) T <<= 1; }
        const int nph = GKM_IDX_THREADS / T;
        const int ph = tid / T, tt = tid - ph * T;
        const bool lane_ok = ph < nph && tt < rem;
        if (!__any_sync(0xFFFFFFFFu, lane_ok)) continue;
        const uint32_t dl = lane_ok ? r.deltas[t0 + tt] : 0u;
        const uint32_t dx = dl & 0x0FFFFFFFu;
        const int mrow = lane_ok ? (int) (dl >> 28) - mbase : 0;
        int32_t *Hm = H + (size_t) mrow * (size_t) ldh;
        const uint32_t bhi_l = lane_ok ? bhi : 0u; /* a lane without a mask never hits */
        const int n_it = (nq + nph - 1) / nph;     /* the same for every lane */
        for (int it = 0; it < n_it; it += UNR) {
            int w[UNR];
            idx_slot_t<FMT> sl[UNR];
#pragma unroll
            for (int u = 0; u < UNR; u++) {
                const int xi = ph + (it + u) * nph;
                const bool ok = xi < nq; /* implies it + u < n_it */
                /* a probe past the last L-mer reads the spare slot behind the table: always empty, never a hit */
                const uint32_t y = ok ? (xq[xi] ^ dx) : r.nslots;
                w[u] = (WEIGHTED && ok) ? (int) wq[xi] : 1;
                sl[u] = __ldg(tab + y);
            }
#pragma unroll
            for (int u = 0; u < UNR; u++) {
                const uint32_t o = idx_slot<WEIGHTED, RANGE, FMT>(sl[u], Hm, blo, bhi_l, w[u]);
                const uint32_t mk = __ballot_sync(0xFFFFFFFFu, o != ~0u);
                if (mk) {
                    if (o != ~0u) queue[qn + __popc(mk & lt)] = QE::make(o, mrow, w[u]);
                    qn += __popc(mk);
                    if (qn >= 32) {
                        __syncwarp();
                        idx_drain<WEIGHTED, RANGE, FMT>(r, queue[qn - 32 + lane], true, H, ldh, blo, bhi, lq, lqn, lt);
                        qn -= 32;
                        __syncwarp();
                    }
                }
            }
            if (lqn) { idx_long<WEIGHTED, RANGE, FMT>(r, lq, lqn, H, ldh, blo, bhi, lane); lqn = 0; }
        }
    }
    __syncwarp();
    idx_drain<WEIGHTED, RANGE, FMT>(r, lane < qn ? queue[lane] : QE::none(), lane < qn, H, ldh, blo, bhi, lq, lqn, lt);
    if (lqn) idx_long<WEIGHTED, RANGE, FMT>(r, lq, lqn, H, ldh, blo, bhi, lane);
}

template <bool WEIGHTED, bool RANGE, int FMT, int MINB>
__global__ void __launch_bounds__(GKM_IDX_THREADS, MINB)
gkm_index_rows_kernel(const __grid_constant__ gkm_kparams p, const __grid_constant__ gkm_idx_rowargs r)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = (int) threadIdx.x;
    const int a = p.row_begin + (int) blockIdx.x;
    const int L = p.L, nb = p.nbins;
    const int nhot = nb < GKM_IDX_HOT_BINS ? nb : GKM_IDX_HOT_BINS, ncoldb = nb - nhot;
    /* wanted columns of this row inside the block, relative to the block's first column */
    uint32_t blo = (uint32_t) r.blo, bhi = (uint32_t) r.bhi;
    if (p.mode == GKM_MODE_LOWER) {
        const int lim = a - r.cb; /* columns < a only */
        if (lim <= (int) blo) return;
        if ((uint32_t) lim < bhi) bhi = (uint32_t) lim;
    }
    if (bhi <= blo) return;
    const int ldh = r.ldh;
    int32_t *H = reinterpret_cast<int32_t *>(smem);                       /* bins ncoldb .. nb-1 */
    int32_t *C = r.cold + (size_t) blockIdx.x * (size_t) ncoldb * (size_t) ldh; /* bins 0 .. ncoldb-1, this row's scratch */
    typedef typename idx_qe<FMT == GKM_IDX_FMT_C16>::type qe_t;
    unsigned char *qbase = smem + (size_t) nhot * (size_t) ldh * 4;
    qe_t *queue = reinterpret_cast<qe_t *>(qbase) + (size_t) (tid >> 5) * (GKM_IDX_QCAP + GKM_IDX_LQCAP); /* this warp's */
    int *lqcnt = reinterpret_cast<int *>(qbase + GKM_IDX_QBYTES_FMT(FMT == GKM_IDX_FMT_C16)) - GKM_IDX_THREADS / 32 + (tid >> 5); /* cold phase only */
    uint32_t *xq = reinterpret_cast<uint32_t *>(qbase + GKM_IDX_QBYTES_FMT(FMT == GKM_IDX_FMT_C16));
    uint8_t *wq = reinterpret_cast<uint8_t *>(xq + r.maxq);

    const int ncol = (int) (bhi - blo);
    for (int m = 0; m < nhot; m++)
        for (int i = tid; i < ncol; i += GKM_IDX_THREADS) H[m * ldh + i] = 0;
    for (int m = 0; m < ncoldb; m++)
        for (int i = tid; i < ncol; i += GKM_IDX_THREADS) __stcg(C + (size_t) m * ldh + i, 0);
    if ((tid & 31) == 0) *lqcnt = 0;
    /* forward L-mers of the query (window ending at e, L-1 <= e < len) */
    const int len = p.lens[a], nq = len - L + 1;
    {
        const uint32_t *pl = p.planes + (size_t) a * 3 * (size_t) p.W;
        const uint32_t mask = (1u << L) - 1u;
        for (int i = tid; i < nq; i += GKM_IDX_THREADS) {
            xq[i] = gkm_idx_code(idx_window(pl, p.W, i, mask), idx_window(pl + p.W, p.W, i, mask), L);
            if (WEIGHTED) wq[i] = p.wend[(size_t) a * 32 * (size_t) p.W + (size_t) (i + L - 1)];
        }
    }
    __syncthreads();

    if (r.ncold > 0) idx_probe_cold<WEIGHTED, RANGE, FMT>(r, 0, r.ncold, xq, wq, nq, C, ldh, blo, bhi, queue + GKM_IDX_QCAP, lqcnt);
    /* weighted types at two CTAs per SM: two loads in flight per thread instead of four (the same number per SM as one
     * CTA with four) keep the 32-register build nearly spill-free: wgkm at 10k 50.7 -> 47.8 ms (tools/wgkm_ab.py) */
    constexpr int UNR = (WEIGHTED && MINB == 2) ? GKM_IDX_WUNR : GKM_IDX_UNROLL;
    idx_probe_hot<WEIGHTED, RANGE, FMT, UNR>(r, r.ncold, r.ndelta, xq, wq, nq, H, ncoldb, ldh, blo, bhi, queue);
    __syncthreads();

    /* epilogue: histogram -> normalised double, the reference's operation order */
    double dsum = 0.0;
    const double sqa = (p.out || p.decision) ? p.sqnorm[a] : 1.0;
    for (int i = tid; i < ncol; i += GKM_IDX_THREADS) {
        const int b_g = r.cb + (int) blo + i;
        int32_t h[GKM_MAX_BINS];
        for (int m = 0; m < ncoldb; m++) h[m] = __ldcg(C + (size_t) m * ldh + i);
        for (int m = 0; m < nhot; m++) h[ncoldb + m] = H[m * ldh + i];
        if (p.hist) {
            int32_t *dst = p.hist + ((size_t) (a - p.row_base) * (size_t) p.hist_cols + (size_t) (b_g - p.col_base)) * (size_t) nb;
            for (int m = 0; m < nb; m++) dst[m] = h[m];
        }
        if (!p.out && !p.decision) continue;
        double kraw = 0.0;
        for (int m = 0; m < nb; m++) kraw = __dadd_rn(kraw, __dmul_rn(p.w[m], (double) h[m]));
        double v = __ddiv_rn(kraw, __dmul_rn(sqa, p.sqnorm[b_g]));
        if (p.kernel_type == 3 || p.kernel_type == 5) v = exp(__dmul_rn(p.gamma, __dadd_rn(v, -1.0)));
        /* streaming store: the matrix is written once and must not push the slot table out of L2 */
        if (p.out) __stcs(p.out + (size_t) (a - p.row_base) * (size_t) p.ld + (size_t) (b_g - p.col_base), v);
        if (p.decision) dsum += p.alpha[b_g - p.col_base] * v;
    }
    if (p.decision) {
        __shared__ double red[GKM_IDX_THREADS / 32];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dsum += __shfl_down_sync(0xFFFFFFFFu, dsum, o);
        if ((tid & 31) == 0) red[tid >> 5] = dsum;
        __syncthreads();
        if (tid < 32) {
            double s = red[tid];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, o);
            if (tid == 0) atomicAdd(p.decision + (a - p.row_base), s);
        }
    }
}

unsigned gkm_idx_row_smem(int nbins, int ldh, int maxq, int weighted, int c16)
{
    const int nhot = nbins < GKM_IDX_HOT_BINS ? nbins : GKM_IDX_HOT_BINS;
    size_t s = (size_t) nhot * (size_t) ldh * 4 + GKM_IDX_QBYTES_FMT(c16) + (size_t) maxq * 4 + (weighted ? (size_t) maxq : 0);
    return (unsigned) ((s + 15) & ~(size_t) 15);
}

size_t gkm_idx_cold_bytes(int nbins, int ldh, int rows)
{
    const int ncoldb = nbins > GKM_IDX_HOT_BINS ? nbins - GKM_IDX_HOT_BINS : 0;
    return (size_t) rows * (size_t) ncoldb * (size_t) ldh * 4;
}

int gkm_idx_max_cols(int nbins, int maxq, int weighted)
{
    const long long budget = 227LL * 1024 - 1024 /* static reduction buffer and slack */ - GKM_IDX_QBYTES_FMT(0) - (long long) maxq * (weighted ? 5 : 4);
    long long cols = budget / (4LL * (nbins < GKM_IDX_HOT_BINS ? nbins : GKM_IDX_HOT_BINS));
    cols &= ~31LL;
    if (cols > (long long) GKM_IDX_MAX_COLS) cols = GKM_IDX_MAX_COLS & ~31;
    return cols < 32 ? 0 : (int) cols;
}

int gkm_idx_rows(const gkm_kparams *kp, const gkm_idx_rowargs *ra, int weighted, cudaStream_t st)
{
    const int rows = kp->row_end - kp->row_begin;
    if (rows <= 0 || ra->bhi <= ra->blo) return 0;
    const bool range = ra->blo != 0;
    const int c16 = ra->fmt == GKM_IDX_FMT_C16;
    const unsigned smem = gkm_idx_row_smem(kp->nbins, ra->ldh, ra->maxq, weighted, c16);
    /* Two CTAs per SM where two full histogram rows of the block fit shared memory (blocks up to ~12 000 columns):
     * that build is held to 32 registers, which the compact-slot code meets without spills (41.0 instead of 46.1 ms
     * at 10k).  The decision is per block, not per launch: mixing the two builds inside one problem measured
     * slower (28 288 sequences: 272 ms against 228 ms), and the 16-byte-slot code spills at 32 registers
     * (wgkm at 10k: 70 ms against 49 ms), so that format always runs one CTA per SM. */
    const unsigned pair = 2u * (gkm_idx_row_smem(kp->nbins, (ra->blk_cols + 31) & ~31, ra->maxq, weighted, c16) + 1280u);
    bool two = ra->fmt != GKM_IDX_FMT_P32 && pair <= (ra->nblk > 1 ? GKM_IDX_TWO_SMEM : 227u * 1024u);
    /* weighted types on input with repeats (long-tailed rows): one CTA per SM (everything-mixed workload of
     * tools/nonuniform.py: 80 against 95 ms; uniform input: 50.4 against 47.4 ms the other way round) */
    if (weighted && ra->skew > GKM_IDX_SKEW_ONE_CTA) two = false;
    if ((ra->fmt == GKM_IDX_FMT_C16 && weighted) || (ra->fmt == GKM_IDX_FMT_W20 && !weighted)) { gkm_set_error("index slot format does not match the kernel type"); return 1; }
    const void *fn;
#define GKM_IDX_PICK(W, F) (range ? (two ? (const void *) gkm_index_rows_kernel<W, true, F, 2> : (const void *) gkm_index_rows_kernel<W, true, F, 1>) \
                                  : (two ? (const void *) gkm_index_rows_kernel<W, false, F, 2> : (const void *) gkm_index_rows_kernel<W, false, F, 1>))
    if (ra->fmt == GKM_IDX_FMT_C16) fn = GKM_IDX_PICK(false, GKM_IDX_FMT_C16);
    else if (ra->fmt == GKM_IDX_FMT_W20) fn = GKM_IDX_PICK(true, GKM_IDX_FMT_W20);
    else if (weighted) fn = GKM_IDX_PICK(true, GKM_IDX_FMT_P32);
    else fn = GKM_IDX_PICK(false, GKM_IDX_FMT_P32);
#undef GKM_IDX_PICK
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    /* Ask for no more shared memory per SM than this launch's CTAs need: what is left is L1, where the in-flight slot
     * probes live.  Without the hint the split of an earlier, larger launch can stay in force (rows issued widest first
     * ran the weighted build 25 % slower than ascending: profiles/r2_chunk_order_carveout_ab.txt). */
    if (e == cudaSuccess) {
        const unsigned per_sm = (two ? 2u : 1u) * (smem + 1280u);
        int pct = (int) ((per_sm * 100u + 228u * 1024u - 1u) / (228u * 1024u));
        if (pct > 100) pct = 100;
        e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    }
    if (e == cudaSuccess) {
        void *args[] = { (void *) kp, (void *) ra };
        e = cudaLaunchKernel(fn, dim3((unsigned) rows, 1, 1), dim3(GKM_IDX_THREADS, 1, 1), args, smem, st);
    }
    if (e != cudaSuccess) { gkm_set_error("CUDA: index row kernel (%u bytes of shared memory): %s", smem, cudaGetErrorString(e)); return 1; }
    return 0;
}
