/* gkm_kparams.h -- launch parameters shared by the histogram kernels (passed by value) */
#ifndef GKM_KPARAMS_H_INCLUDED
#define GKM_KPARAMS_H_INCLUDED

#include <stdint.h>

enum { GKM_MODE_RECT = 0, GKM_MODE_LOWER = 1, GKM_MODE_DIAG = 2 };

struct gkm_kparams {
    /* device-resident problem image (gkm_pack.h; packed by gkm_device.cu: gkm_pack_kernel) */
    const uint32_t *planes; /* [n][3][W]: code bit 0, code bit 1, valid-window-end plane; both strands, circular */
    const int32_t *lens;    /* [n] */
    const uint8_t *wend;    /* [n][32W], weighted kernel types only */
    const double *sqnorm;   /* [n] */
    /* outputs (any may be null) */
    double *out;            /* out[(row-row_base)*ld + (col-col_base)] = K(row,col) */
    long long ld;
    int32_t *hist;          /* hist[((row-row_base)*hist_cols + (col-col_base))*nbins + m] = H_m(row,col) */
    int hist_cols;
    double *sqnorm_out;     /* GKM_MODE_DIAG: sqnorm_out[row] = sqrt(Kraw(row,row)) */
    const double *alpha;    /* decision values: decision[row-row_base] += alpha[col-col_base]*K(row,col) */
    double *decision;
    /* the block of the matrix this launch covers */
    int row_begin, row_end, col_begin, col_end;
    int row_base, col_base;
    int mode;
    /* shapes */
    int W;      /* words per bit plane (2*maxlen bits) */
    int WA;     /* 32-position chunks of the longest query */
    int TA, TB; /* query rows / target columns per CTA */
    int L, d, nbins, kernel_type;
    double gamma;
    double w[16];
};

#endif
