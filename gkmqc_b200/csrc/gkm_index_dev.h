/* gkm_index_dev.h -- device-side interface of the "index" variant (gkm_index.cu), used by gkm_device.cu */
#ifndef GKM_INDEX_DEV_H_INCLUDED
#define GKM_INDEX_DEV_H_INCLUDED

#include <cuda_runtime.h>
#include <stdint.h>

#include "gkm_index.h"
#include "gkm_kparams.h"

/* the index of one block of columns [cb, ce) on one GPU */
struct gkm_idx_block {
    int cb, ce;
    int fmt;             /* GKM_IDX_FMT_P32 (16-byte slots) or GKM_IDX_FMT_C16 (8-byte slots of 16-bit columns) */
    void *tab;           /* 4^L slots */
    uint32_t *ovf;       /* overflow lists (16-byte aligned, padded with end markers) */
    size_t tab_bytes, ovf_bytes; /* block sizes as handed out by the pool */
    unsigned long long sumsq;    /* sum of squared posting-list lengths (gkm_idx_runs_kernel) */
    double skew;                 /* sumsq / postings: ~1 + postings per slot on uniform input, far more with repeats */
    size_t postings;
    int built;
    /* the row-kernel launches of this block since the compute call began (choose_variant clears them; first GPU only):
     * bit 2 RANGE + MINB - 1 per build gkm_index_rows_kernel<., RANGE, ., MINB> that ran, the most dynamic shared memory
     * one asked for, and the number of launches */
    int inst_mask;
    unsigned max_smem;
    long long launches;
};

struct gkm_idx_build_args {
    const uint32_t *planes; const int32_t *lens; const uint8_t *wend; /* wend = NULL: unit weights */
    int W, L, cb, ce;
    const uint32_t *offs;  /* device, [ce - cb]: first posting of every column (2 * (len - L + 1) each) */
    size_t P;              /* postings of the block */
    void *scratch;         /* gkm_idx_scratch_bytes(P, L) bytes */
    size_t cub_bytes;
    int fmt;
    void *tab; uint32_t *ovf;
    unsigned long long *h_sumsq; /* host, optional: sum of squared list lengths, valid once the stream has drained */
};

struct gkm_idx_rowargs {
    int fmt;
    const void *tab; const uint32_t *ovf; const uint32_t *deltas;
    uint32_t nslots; /* 4^L: index of the spare, always empty slot behind the table */
    int ndelta;    /* masks in all */
    int ncold;     /* the first ncold masks belong to the cold bins (m <= d - 2) */
    int32_t *cold; /* [rows of the launch][cold bins][ldh] scratch in global memory, zeroed by the kernel */
    int cb;        /* first column of the index block */
    int blo, bhi;  /* wanted columns, relative to cb */
    int ldh;       /* histogram row stride in shared memory (>= bhi - blo) */
    int blk_cols;  /* columns of the whole index block (decides the kernel build) */
    int nblk;      /* column blocks of the problem (ditto) */
    double skew;   /* of the block (ditto, weighted types) */
    int maxq;      /* upper bound of query L-mers per row */
};

/* bits [lo, lo + L) of a bit plane of W words (mask = 2^L - 1): the window of the L-mer that starts at lo */
static __device__ __forceinline__ uint32_t idx_window(const uint32_t *pl, int W, int lo, uint32_t mask)
{
    const int w = lo >> 5, s = lo & 31;
    const uint32_t x = pl[w], y = (w + 1 < W) ? pl[w + 1] : 0u;
    return __funnelshift_r(x, y, (uint32_t) s) & mask;
}

size_t gkm_idx_tab_bytes(int L, int fmt);
size_t gkm_idx_ovf_bytes(size_t P, int fmt);
size_t gkm_idx_scratch_bytes(size_t P, int L, size_t *cub_bytes_out);
int gkm_idx_build(const gkm_idx_build_args *a, cudaStream_t st);
/* the first steps of gkm_idx_build, shared with the L-mer table (gkm_lmer_table.cu): the keys code << 32 | column - cb << 8 |
 * weight of every L-mer of both strands of the columns [cb, ce), radix-sorted by code (stable: by column inside a code,
 * and in generation order inside a column).  Only planes .. P, scratch and cub_bytes of `a` are read; *sorted points
 * into the scratch. */
cudaError_t gkm_idx_sort_keys(const gkm_idx_build_args *a, cudaStream_t st, const unsigned long long **sorted);
/* host rules of the row kernel's launch, C linkage so that the CPU tests can call them */
extern "C" {
/* most columns one block may hold so that the hot histogram rows + the query fit 227 KB of shared memory (0: none) */
int gkm_idx_max_cols(int nbins, int maxq, int weighted);
unsigned gkm_idx_row_smem(int nbins, int ldh, int maxq, int weighted, int c16);
/* 1 when the row kernel of a block of blk_cols columns (format fmt, one of nblk blocks, sum len^2 / postings = skew) runs
 * two CTAs per SM, 0 for one */
int gkm_idx_two_cta(int nbins, int blk_cols, int maxq, int weighted, int fmt, int nblk, double skew);
}
/* bytes of cold-bin scratch a launch of `rows` rows needs */
size_t gkm_idx_cold_bytes(int nbins, int ldh, int rows);
/* the build gkm_index_rows_kernel<WEIGHTED, RANGE, FMT, MINB> a launch ran: RANGE, MINB (0: nothing launched) and its
 * dynamic shared memory */
struct gkm_idx_launch {
    int range, minb;
    unsigned smem;
};
/* rows [kp->row_begin, kp->row_end) against the wanted columns of one block; outputs as in gkm_kparams; *ran (may be NULL)
 * tells which build ran */
int gkm_idx_rows(const gkm_kparams *kp, const gkm_idx_rowargs *ra, int weighted, cudaStream_t st, gkm_idx_launch *ran);

#endif
