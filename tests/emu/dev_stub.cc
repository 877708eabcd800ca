/* tests/emu/dev_stub.cc -- a host stand-in for the device layer (the gkm_dev_* functions of
 * gkm_device.cu, gkm_compute.cu, gkm_resident.cu and gkm_microbench.cu), to run the
 * reference-ABI shim gkm_capi.c (gkmkernel_init / read_problems / new_object / build_tree / kernelfunc_batch[_all] /
 * swap_index / update_index, libgkm.h:132-147) in the CPU-only test tier, also under ASan + UBSan
 * (tools/asan_host.sh).  gkm_capi.c is pointer bookkeeping over caller-visible structs -- the code ADVICE r1 found a heap
 * overflow in -- and on the GPU box it can only be exercised unsanitised.  It also hands out the host packer's image
 * (gkmb200_problem_image), so that the CPU tier can check the packing rule the device packer shares with it.
 *
 * TEST INFRASTRUCTURE, not a fallback: this file is linked into build/libgkm_abi_emu.so only; the product
 * (gkmqc_b200/bin/gkmkern_pylib.so) has no CPU path and fails loudly without a B200.
 *
 * Histograms come from the lane emulator of the bit-sliced kernel (diag_emu.cc: the arithmetic of gkm_bitslice.h over
 * the product's own packed image); the epilogue below is gkm_emit_entry (gkm_diag_kernel.cuh) in plain C: ascending-m
 * multiply-add without contraction, one division, optional exp -- the reference's order (libgkm.c:576-582,1169-1179).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../gkmqc_b200/csrc/gkm_internal.h"

extern "C" int gkm_emu_hist(gkmb200_problem *p, int a, int b, int32_t *H);

static double kraw_of(const gkmb200_problem *p, const int32_t *H)
{
    volatile double sum = 0.0; /* volatile: no fused multiply-add, whatever the compiler flags */
    for (int m = 0; m < p->nbins; m++) {
        volatile double t = p->w[m] * (double) H[m];
        sum = sum + t;
    }
    return sum;
}

static double entry_of(const gkmb200_problem *p, int a, int b, const int32_t *H)
{
    volatile double den = p->sqnorm[a] * p->sqnorm[b];
    double v = kraw_of(p, H) / den;
    if (p->param.kernel_type == EST_TRUNC_RBF || p->param.kernel_type == EST_TRUNC_PW_RBF) {
        volatile double t = v + -1.0;
        volatile double u = p->param.gamma * t;
        v = exp(u);
    }
    return v;
}

extern "C" {

int gkm_dev_count(void) { return 0; }
int gkm_dev_select(const int *, int) { gkm_set_error("emulator build: no devices"); return 1; }

int gkm_dev_upload(gkmb200_problem *p)
{
    if (!p) { gkm_set_error("null problem"); return 1; }
    if (p->packed && p->planes && p->have_sqnorm) return 0;
    if (gkm_pack_problem(p)) return 1;
    int32_t H[GKM_MAX_BINS];
    for (int i = 0; i < p->n; i++) {
        if (gkm_emu_hist(p, i, i, H)) { gkm_set_error("emulator: no lane code for L=%d", p->param.L); return 1; }
        p->sqnorm[i] = sqrt(kraw_of(p, H));
    }
    p->have_sqnorm = 1;
    p->host_sqnorm = 1;
    return 0;
}

int gkm_dev_compute(gkmb200_problem *p, int row0, int nrows, int col0, int ncols, int lower,
                    double *out, long ld, double **rows, int32_t *hist, int copy_threads)
{
    (void) copy_threads;
    if (!p) { gkm_set_error("null problem"); return 1; }
    if (row0 < 0 || col0 < 0 || nrows < 0 || ncols < 0 || row0 + nrows > p->n || col0 + ncols > p->n) {
        gkm_set_error("block [%d,+%d) x [%d,+%d) outside the problem (n=%d)", row0, nrows, col0, ncols, p->n);
        return 1;
    }
    if (gkm_dev_upload(p)) return 1;
    int32_t H[GKM_MAX_BINS];
    long long entries = 0;
    for (int r = row0; r < row0 + nrows; r++) {
        int hi = col0 + ncols;
        if (lower && hi > r) hi = r;
        for (int c = col0; c < hi; c++) {
            if (gkm_emu_hist(p, r, c, H)) { gkm_set_error("emulator: no lane code for L=%d", p->param.L); return 1; }
            if (hist) memcpy(hist + ((size_t) (r - row0) * (size_t) ncols + (size_t) (c - col0)) * (size_t) p->nbins, H, sizeof(int32_t) * (size_t) p->nbins);
            const double v = entry_of(p, r, c, H);
            if (rows) rows[r][c] = v;
            else if (out) out[(size_t) (r - row0) * (size_t) ld + (size_t) (c - col0)] = v;
            entries++;
        }
        if (lower && r >= col0 && r < col0 + ncols) {
            if (rows) rows[r][r] = 1.0; /* gkmkern_pylib.c:219-221 */
            else if (out) out[(size_t) (r - row0) * (size_t) ld + (size_t) (r - col0)] = 1.0;
        }
    }
    p->stats.entries = entries;
    p->stats.devices = 0;
    p->stats.shard_rank = 0; p->stats.shard_world = 1;
    return 0;
}

static int no_device(const char *what) { gkm_set_error("emulator build: %s needs the device", what); return 1; }
int gkm_dev_decision(gkmb200_problem *, int, int, int, int, const double *, double, double *) { return no_device("decision values"); }
int gkm_dev_bench_lower(gkmb200_problem *, int, int, int, double *) { return no_device("the resident bench"); }
int gkm_dev_microbench(const char *, double *) { return no_device("a micro-benchmark"); }
int gkm_dev_svm_cv(gkmb200_problem *, const double *, long, int, int, const gkmb200_svm_task *, const int *, const signed char *,
                   const int *, double, double, int, double *, gkmb200_svm_fit *, double *) { return no_device("the SVM consumer"); }
/* the image as the host packer builds it (gkm_seq.c: gkm_pack_problem, the rule of gkm_pack.h), in the layout of the
 * device's gkmb200_problem_image: the CPU tier checks it against an independent model of the image */
int gkmb200_problem_image(gkmb200_problem *p, uint32_t *planes, uint8_t *wend, int *out_shape)
{
    if (!p) { gkm_set_error("null problem"); return 1; }
    if (gkm_pack_problem(p)) return 1;
    const size_t n = (size_t) p->n, W = (size_t) p->Wmax;
    if (out_shape) { out_shape[0] = p->n; out_shape[1] = p->Wmax; }
    if (planes) memcpy(planes, p->planes, n * 3 * W * sizeof(uint32_t));
    if (wend && p->weighted) memcpy(wend, p->wend, n * 32 * W);
    return 0;
}

/* the index variant never runs here: the launch record (gkm_device.cu) has nothing to report */
int gkmb200_problem_index_blocks(const gkmb200_problem *, long long *, int) { no_device("the index launch record"); return -1; }

} /* extern "C" */
