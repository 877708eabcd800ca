/* gkm_lmer_table_dev.h -- device-side interface of the L-mer table (gkm_lmer_table.cu), used by gkm_device.cu */
#ifndef GKM_LMER_TABLE_DEV_H_INCLUDED
#define GKM_LMER_TABLE_DEV_H_INCLUDED

#include <cuda_runtime.h>
#include <stdint.h>

#include "gkm_index_dev.h"

struct gkm_lt_build_args {
    gkm_idx_build_args keys; /* planes, lens, wend, W, L, cb, ce, offs, P, scratch, cub_bytes: the SV columns' sorted keys */
    int d;
    const double *alpha;     /* device, [ce - cb] */
    const double *norm;      /* device, [ce - cb]: |c| of the columns (sqnorm of the upload, from cb) */
    double *beta;            /* device, [ce - cb] */
    double *A;               /* device, [d + 1][4^L] */
    double *T;               /* device, [4^L] */
    const double *w;         /* host, w[0..d] */
};

/* S, transform and combine on stream st; ev = NULL or four events recorded before S, between the phases and behind
 * the combine */
int gkm_lt_build(const gkm_lt_build_args *a, cudaStream_t st, cudaEvent_t *ev);
/* out[lex] = T[code of lex], 4^L values (device buffers) */
int gkm_lt_export(const double *T, int L, double *out, cudaStream_t st);
/* out[r] = (sum over the forward L-mers of row row0 + r of wt * T[code]) / norm[row0 + r], r < nrows; wend = NULL: unit weights */
int gkm_lt_score(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L,
                 const double *norm, int row0, int nrows, double *out, cudaStream_t st);
/* out[4 i + v] = (numerator of the row row[i] with base pos[i] replaced by v) / its norm, i < nsites (gkm_lmer_subst.h):
 * H = the rows' self histograms, [rows][d + 1] int32 from row hrow0; w[0..d] host; maxlen = the longest row of the
 * problem; row, pos, out device buffers.  Sites of one row are best consecutive: each block of 64 stages a row once per run. */
int gkm_lt_subst(const double *T, const uint32_t *planes, const int32_t *lens, const uint8_t *wend, int W, int L, int d,
                 const double *w, const int32_t *H, int hrow0, int maxlen, const int *row, const int *pos, long long nsites,
                 double *out, cudaStream_t st);

#endif
