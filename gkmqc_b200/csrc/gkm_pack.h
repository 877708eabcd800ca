/* gkm_pack.h -- the packing rule of the problem image, position by position.  The device packer (gkm_device.cu:
 * gkm_pack_kernel) and the host packer of the CPU emulators (gkm_seq.c: gkm_pack_problem) both include it verbatim.
 *
 * Per sequence one circular string of 32 W positions: the forward strand at [0, len), its reverse complement (3 - code,
 * mirrored: libgkm.c:878-888) at [len, 2 len), zero padding behind.  The image holds, per position j, the two bits of the
 * base code, bit E (an L-mer of either strand ends at j) and, for the weighted kernel types, wend[j], the positional weight
 * of that L-mer: the reference gives the L-mer starting at t the weight wt[t] = f(|nk / 2 - t|) (libgkm.c:910-932) and its
 * reverse-complement strand wt_rc[t] = wt[nk - 1 - t]. */
#ifndef GKM_PACK_H_INCLUDED
#define GKM_PACK_H_INCLUDED

#include <stdint.h>
#include <stdlib.h>

#include "gkm_internal.h"

/* position j of the circular string of a sequence of `len` letters c[]: returns the base code and sets *s to the start,
 * in forward-strand numbering of wt[], of the L-mer that ends at j, or to -1 if none does */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline uint32_t gkm_pack_code(const uint8_t *c, int len, int L, int j, int *s)
{
    const int nk = len - L + 1;
    uint32_t code = 0;
    int start = -1;
    if (j < len) {
        code = gkm_base_code(c[j]);
        if (j >= L - 1) start = j - (L - 1);
    } else if (j < 2 * len) {
        code = 3u - gkm_base_code(c[2 * len - 1 - j]);
        const int rel = j - len;
        if (rel >= L - 1) start = nk - 1 - (rel - (L - 1)); /* wt_rc[t] = wt[nk - 1 - t] */
    }
    *s = start;
    return code;
}

/* wend at that position, centre = nk / 2 = (len - L + 1) / 2: tab[dist] = weight of the L-mer dist starts away from the
 * centre one (gkm_posweight_table), so that exp() never runs on the device and the bytes are the host's */
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline uint8_t gkm_pack_weight(const uint8_t *tab, int centre, int s)
{
    return (s >= 0) ? tab[abs(centre - s)] : (uint8_t) 0;
}

#endif
