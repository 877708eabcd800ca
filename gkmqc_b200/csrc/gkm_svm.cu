/* gkm_svm.cu -- SURVEY.md 8f/f4: the device-resident consumer of the kernel matrix.
 *
 * gkmQC's `evaluate` trains 5-fold x 10-repeat C-SVCs on the precomputed gkm kernel
 * (scripts/gkmsvm.py:104-160: sklearn.svm.SVC(kernel="precomputed", C, tol, shrinking=0) .fit()
 * .decision_function(), 50 fits per bin) -- once the kernel matrix takes 50 ms that is the whole run time.
 * sklearn hands the work to its bundled libsvm (third-party, not in /root/reference; scikit-learn 1.9.0,
 * libsvm 3.x "svm.cpp": Solver::Solve / select_working_set / calculate_rho, Fan, Chen & Lin 2005, WSS 2).
 * This file restates that solver for the GPU, one CTA per fit, and keeps libsvm's arithmetic so that the
 * iterates -- not just the optimum -- coincide:
 *   - the training points are grouped by class, label 0 first, and that class gets y = +1 (svm_group_classes
 *     with sklearn's label sort; svm_train's sub-problem), sklearn flips the sign of the decision value back;
 *   - Q_ij = (float)(y_i y_j K_ij): libsvm caches kernel rows as `Qfloat` = float; QD_i = K_ii stays double;
 *   - maximal violating pair: i = argmax over I_up of -y G with `>=` (the LAST index wins a tie), j = argmin of
 *     -(b*b)/a over I_low with `<=`, a = QD_i + QD_j -/+ 2 y_i Q_ij (TAU = 1e-12 when a <= 0);
 *   - the two-case clipped update of (alpha_i, alpha_j), G_k += Q_ik*dalpha_i + Q_jk*dalpha_j without FMA;
 *   - stop when Gmax + Gmax2 < eps; rho = mean of y G over the free vectors in index order (or the midpoint);
 *   - decision value = sum over support vectors in model order of coef * K(x, sv), minus rho, no FMA.
 * Shrinking (SVC(shrinking=True); gkmQC's default is off, bin/gkmqc.py:209) is the SHRINK instance of the same kernel:
 * libsvm's do_shrinking every min(l, 1000) iterations with its exact permutation, the unshrink at Gmax1 + Gmax2 <=
 * 10 eps, reconstruct_gradient in whichever of its two loop orders libsvm picks, G_bar updated on every change of
 * an upper-bound status, rho over the active set -- the same iterates as sklearn with shrinking.
 *
 * Data: the symmetric n x n matrix is resident in HBM (ld doubles per row); per fit G, alpha, the gather index
 * and y live in shared memory (21 bytes per training point: 10 724 points fit), every iteration reads two
 * kernel rows through the gather index; the shrinking solver's G_bar and position map stay in global memory.
 * Bound: latency of two block-wide arg-reductions per iteration; the 50 fits of a bin run concurrently, one per SM.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "gkm_internal.h"
#include "gkm_svm.h"

#define SVM_THREADS 1024
#define SVM_TAU 1e-12

struct svm_pick { double v; int i; };

/* global scratch of the shrinking solver, indexed like train_idx (idx, y: the global-state path only) */
struct svm_shrink_buf {
    double *gbar;
    int *aset, *pairs, *idx;
    signed char *y;
    gkm_svm_shrink_stats *stats;
};

/* block-wide arg-max of (v, i): larger v wins, equal v -> larger i (libsvm scans upwards with >= / <=) */
__device__ __forceinline__ svm_pick svm_block_argmax(svm_pick x, svm_pick *red /* [32] shared */)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xFFFFFFFFu, x.v, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, x.i, o);
        if (ov > x.v || (ov == x.v && oi > x.i)) { x.v = ov; x.i = oi; }
    }
    __syncthreads(); /* red[] may still be read from the previous reduction */
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
    __syncthreads();
    x = red[threadIdx.x & 31];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xFFFFFFFFu, x.v, o);
        const int oi = __shfl_xor_sync(0xFFFFFFFFu, x.i, o);
        if (ov > x.v || (ov == x.v && oi > x.i)) { x.v = ov; x.i = oi; }
    }
    return x;
}

__device__ __forceinline__ double svm_block_max(double x, double *red /* [32] shared */)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
    __syncthreads();
    x = red[threadIdx.x & 31];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
    return x;
}

/* libsvm's select_working_set over [0, act): the working pair (i, j), or i = -1 once that set is optimal within eps */
__device__ __forceinline__ int2 svm_select(const double *__restrict__ K, long long ld, const double *__restrict__ qd,
                                           const double *G, const double *A, const int *idx, const signed char *y, int act,
                                           double C, double eps, svm_pick *red_pick, double *red_max)
{
    const int tid = (int) threadIdx.x;
    /* ---- i: maximal -y G over I_up ---- */
    svm_pick pi; pi.v = -INFINITY; pi.i = -1;
    for (int k = tid; k < act; k += SVM_THREADS) {
        const double a = A[k], g = G[k];
        if (y[k] > 0) { if (a < C && -g >= pi.v) { pi.v = -g; pi.i = k; } }
        else          { if (a > 0.0 && g >= pi.v) { pi.v = g; pi.i = k; } }
    }
    pi = svm_block_argmax(pi, red_pick);
    const int i = pi.i;
    const double Gmax = pi.v;
    if (i < 0) return make_int2(-1, -1);
    /* ---- j: second-order choice over I_low; Q_i row through the gather index ---- */
    const double *Ki = K + (size_t) idx[i] * (size_t) ld;
    const int yi = y[i];
    const double QDi = qd[idx[i]];
    svm_pick pj; pj.v = -INFINITY; pj.i = -1; /* maximise -obj_diff = b*b/a, ties -> last index */
    double gmax2 = -INFINITY;
    for (int k = tid; k < act; k += SVM_THREADS) {
        const double a = A[k], g = G[k];
        const int yk = y[k];
        const float qik = (float) ((double) (yi * yk) * Ki[idx[k]]);
        if (yk > 0) {
            if (a > 0.0) {
                const double gd = Gmax + g;
                if (g >= gmax2) gmax2 = g;
                if (gd > 0.0) {
                    const double qdk = qd[idx[k]];
                    const double qc = __dadd_rn(__dadd_rn(QDi, qdk), -__dmul_rn(2.0 * (double) yi, (double) qik));
                    const double od = (qc > 0.0) ? -__ddiv_rn(__dmul_rn(gd, gd), qc) : -__ddiv_rn(__dmul_rn(gd, gd), SVM_TAU);
                    if (-od >= pj.v) { pj.v = -od; pj.i = k; }
                }
            }
        } else {
            if (a < C) {
                const double gd = Gmax - g;
                if (-g >= gmax2) gmax2 = -g;
                if (gd > 0.0) {
                    const double qdk = qd[idx[k]];
                    const double qc = __dadd_rn(__dadd_rn(QDi, qdk), __dmul_rn(2.0 * (double) yi, (double) qik));
                    const double od = (qc > 0.0) ? -__ddiv_rn(__dmul_rn(gd, gd), qc) : -__ddiv_rn(__dmul_rn(gd, gd), SVM_TAU);
                    if (-od >= pj.v) { pj.v = -od; pj.i = k; }
                }
            }
        }
    }
    pj = svm_block_argmax(pj, red_pick);
    gmax2 = svm_block_max(gmax2, red_max);
    const int j = pj.i;
    if (Gmax + gmax2 < eps || j < 0) return make_int2(-1, -1);
    return make_int2(i, j);
}

/* One fit per CTA.  SHRINK: libsvm's shrinking heuristic (Solver::Solve with shrinking = 1).  Positions [0, act) are
 * the active set; do_shrinking moves shrunk points behind it with the swaps of libsvm's own loop, so the state
 * arrays are permuted and aset maps a position to its grouped training position.  G_bar (the gradient part of the
 * points at the upper bound) and aset are touched only on a status change, at a shrink pass and at a gradient
 * reconstruction: they live in global memory (L2), so the per-iteration state keeps its 21 bytes per point. */
template <bool SHRINK>
__global__ void __launch_bounds__(SVM_THREADS, 1)
gkm_svm_smo_kernel(const double *__restrict__ K, long long ld, const double *__restrict__ qd, const gkm_svm_task *__restrict__ tasks,
                   const int *__restrict__ train_idx, const signed char *__restrict__ train_y,
                   double C, double eps, int max_iter, int in_smem,
                   double *__restrict__ alpha_out, double *__restrict__ g_scratch, svm_shrink_buf sb, gkm_svm_fit *__restrict__ fits)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ svm_pick red_pick[32];
    __shared__ double red_max[32];
    __shared__ double sh_d[4];
    __shared__ int sh_u[2];
    __shared__ int warp_cnt[32];

    const gkm_svm_task t = tasks[blockIdx.x];
    const int l = t.ntrain;
    const int tid = (int) threadIdx.x;
    const int *gidx = train_idx + t.train_off;
    const signed char *gy = train_y + t.train_off;
    double *G, *A;
    int *idx;
    signed char *y;
    if (in_smem) {
        G = reinterpret_cast<double *>(smem);
        A = G + l;
        idx = reinterpret_cast<int *>(A + l);
        y = reinterpret_cast<signed char *>(idx + l);
    } else { /* longer problems: the state stays in global memory (L2) */
        G = g_scratch + 2 * t.train_off;
        A = G + l;
        if (SHRINK) { idx = sb.idx + t.train_off; y = sb.y + t.train_off; } /* shrinking permutes them: own copies */
        else { idx = const_cast<int *>(gidx); y = const_cast<signed char *>(gy); }
    }
    double *gbar = SHRINK ? sb.gbar + t.train_off : NULL;
    int *aset = SHRINK ? sb.aset + t.train_off : NULL;
    int *pairs = SHRINK ? sb.pairs + t.train_off : NULL;
    for (int k = tid; k < l; k += SVM_THREADS) {
        G[k] = -1.0; /* p_i = -1, alpha = 0 */
        A[k] = 0.0;
        if (in_smem || SHRINK) { idx[k] = gidx[k]; y[k] = gy[k]; }
        if (SHRINK) { gbar[k] = 0.0; aset[k] = k; }
    }
    __syncthreads();

    int iter = 0, act = l;
    /* shrinking state and statistics: every thread keeps the same copy */
    int counter = (l < 1000 ? l : 1000) + 1, passes = 0, min_act = l, unshrink_iter = -1, recon_a = 0, recon_b = 0;
    bool unshrunk = false;

    /* reconstruct_gradient: G of the inactive points from G_bar and the free active points, each G entry summed in
     * libsvm's order by one thread; the row read is the one libsvm's loop order reads */
    auto reconstruct = [&]() {
        if (act == l) return;
        int nr_free = 0;
        for (int b = 0; b < act; b += SVM_THREADS) {
            const int k = b + tid;
            nr_free += __syncthreads_count(k < act && A[k] > 0.0 && A[k] < C);
        }
        const bool order_a = nr_free * l > 2 * act * (l - act); /* libsvm's int arithmetic */
        recon_a += order_a;
        recon_b += !order_a;
        for (int i = act + tid; i < l; i += SVM_THREADS) {
            double g = __dadd_rn(gbar[i], -1.0);
            const long long ci = idx[i];
            const int yi = y[i];
            for (int j = 0; j < act; j++) {
                const double a = A[j];
                if (a > 0.0 && a < C) {
                    const double kv = order_a ? K[ci * ld + idx[j]] : K[(long long) idx[j] * ld + ci];
                    const float q = (float) ((double) (yi * y[j]) * kv);
                    g = __dadd_rn(g, __dmul_rn(a, (double) q));
                }
            }
            G[i] = g;
        }
        __syncthreads();
    };

    /* do_shrinking: libsvm's two-pointer loop swaps the k-th shrunk position below n_keep (counting up) with the k-th
     * kept position at or above it (counting down); one block-wide prefix count of the kept points finds both ranks */
    auto shrink = [&]() {
        double g1 = -INFINITY, g2 = -INFINITY;
        for (int k = tid; k < act; k += SVM_THREADS) {
            const double a = A[k], g = G[k];
            if (y[k] > 0) { if (a < C) g1 = fmax(g1, -g); if (a > 0.0) g2 = fmax(g2, g); }
            else          { if (a < C) g2 = fmax(g2, -g); if (a > 0.0) g1 = fmax(g1, g); }
        }
        g1 = svm_block_max(g1, red_max);
        g2 = svm_block_max(g2, red_max);
        if (!unshrunk && __dadd_rn(g1, g2) <= __dmul_rn(eps, 10.0)) {
            unshrunk = true;
            unshrink_iter = iter;
            reconstruct();
            act = l;
        }
        auto shrunk = [&](int k) -> bool {
            const double a = A[k], g = G[k];
            if (a >= C) return y[k] > 0 ? -g > g1 : -g > g2;
            if (a <= 0.0) return y[k] > 0 ? g > g2 : g > g1;
            return false;
        };
        int n_keep = 0;
        for (int b = 0; b < act; b += SVM_THREADS) {
            const int k = b + tid;
            n_keep += __syncthreads_count(k < act && !shrunk(k));
        }
        const int lane = tid & 31, warp = tid >> 5;
        int before = 0, m = 0; /* kept points before the tile; pairs to swap */
        for (int b = 0; b < act; b += SVM_THREADS) {
            const int k = b + tid;
            const bool in = k < act;
            const bool keep = in && !shrunk(k);
            const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
            if (lane == 0) warp_cnt[warp] = __popc(bal);
            __syncthreads();
            int woff = 0, tile = 0;
            for (int w = 0; w < SVM_THREADS / 32; w++) { const int c = warp_cnt[w]; woff += w < warp ? c : 0; tile += c; }
            const int P = before + woff + __popc(bal & ((1u << lane) - 1u)); /* kept points before k */
            if (in && !keep && k < n_keep) pairs[k - P] = k;             /* upward rank among the shrunk */
            if (keep && k >= n_keep) pairs[l - n_keep + P] = k;          /* = l - 1 - downward rank among the kept */
            m += __syncthreads_count(in && !keep && k < n_keep);
            before += tile;
        }
        for (int r = tid; r < m; r += SVM_THREADS) {
            const int p = pairs[r], q = pairs[l - 1 - r];
            double d = G[p]; G[p] = G[q]; G[q] = d;
            d = A[p]; A[p] = A[q]; A[q] = d;
            d = gbar[p]; gbar[p] = gbar[q]; gbar[q] = d;
            int s = idx[p]; idx[p] = idx[q]; idx[q] = s;
            s = aset[p]; aset[p] = aset[q]; aset[q] = s;
            const signed char c = y[p]; y[p] = y[q]; y[q] = c;
        }
        __syncthreads();
        act = n_keep;
        passes++;
        if (act < min_act) min_act = act;
    };

    for (;;) {
        if (SHRINK) {
            if (iter >= max_iter) break;
            if (--counter == 0) { counter = l < 1000 ? l : 1000; shrink(); }
        }
        int2 ij = svm_select(K, ld, qd, G, A, idx, y, act, C, eps, red_pick, red_max);
        if (ij.x < 0) {
            if (!SHRINK) break;
            reconstruct(); /* the whole gradient, then the whole set */
            act = l;
            ij = svm_select(K, ld, qd, G, A, idx, y, act, C, eps, red_pick, red_max);
            if (ij.x < 0) break;
            counter = 1; /* shrink in the next iteration */
        }
        if (!SHRINK && iter >= max_iter) break;
        iter++;
        const int i = ij.x, j = ij.y;
        /* ---- analytic step on (alpha_i, alpha_j) ---- */
        const double *Ki = K + (size_t) idx[i] * (size_t) ld;
        const double *Kj = K + (size_t) idx[j] * (size_t) ld;
        const int yi = y[i];
        const int yj = y[j];
        if (tid == 0) {
            const float qij = (float) ((double) (yi * yj) * Ki[idx[j]]);
            const double QDi = qd[idx[i]];
            const double QDj = qd[idx[j]];
            const double oai = A[i], oaj = A[j];
            double ai = oai, aj = oaj;
            if (yi != yj) {
                double qc = __dadd_rn(__dadd_rn(QDi, QDj), (double) (2.0f * qij));
                if (qc <= 0.0) qc = SVM_TAU;
                const double delta = __ddiv_rn(__dadd_rn(-G[i], -G[j]), qc);
                const double diff = ai - aj;
                ai = __dadd_rn(ai, delta);
                aj = __dadd_rn(aj, delta);
                if (diff > 0.0) { if (aj < 0.0) { aj = 0.0; ai = diff; } }
                else            { if (ai < 0.0) { ai = 0.0; aj = -diff; } }
                if (diff > 0.0 /* C_i - C_j = 0 */) { if (ai > C) { ai = C; aj = C - diff; } }
                else                                 { if (aj > C) { aj = C; ai = C + diff; } }
            } else {
                double qc = __dadd_rn(__dadd_rn(QDi, QDj), -(double) (2.0f * qij));
                if (qc <= 0.0) qc = SVM_TAU;
                const double delta = __ddiv_rn(__dadd_rn(G[i], -G[j]), qc);
                const double sum = __dadd_rn(ai, aj);
                ai = __dadd_rn(ai, -delta);
                aj = __dadd_rn(aj, delta);
                if (sum > C) { if (ai > C) { ai = C; aj = sum - C; } }
                else         { if (aj < 0.0) { aj = 0.0; ai = sum; } }
                if (sum > C) { if (aj > C) { aj = C; ai = sum - C; } }
                else         { if (ai < 0.0) { ai = 0.0; aj = sum; } }
            }
            A[i] = ai; A[j] = aj;
            sh_d[0] = ai - oai;
            sh_d[1] = aj - oaj;
            /* +1: moved onto the upper bound, -1: off it */
            sh_u[0] = (ai >= C) - (oai >= C);
            sh_u[1] = (aj >= C) - (oaj >= C);
        }
        __syncthreads();
        const double dai = sh_d[0], daj = sh_d[1];
        /* ---- gradient ---- */
        for (int k = tid; k < act; k += SVM_THREADS) {
            const int yk = y[k];
            const int c = idx[k];
            const float qik = (float) ((double) (yi * yk) * Ki[c]);
            const float qjk = (float) ((double) (yj * yk) * Kj[c]);
            G[k] = __dadd_rn(G[k], __dadd_rn(__dmul_rn((double) qik, dai), __dmul_rn((double) qjk, daj)));
        }
        /* ---- G_bar over all l: C * Q_i for a status change of i, then of j ---- */
        if (SHRINK && (sh_u[0] | sh_u[1])) {
            const int ui = sh_u[0], uj = sh_u[1];
            for (int k = tid; k < l; k += SVM_THREADS) {
                const int yk = y[k];
                const int c = idx[k];
                double gb = gbar[k];
                if (ui) { const double d = __dmul_rn(C, (double) (float) ((double) (yi * yk) * Ki[c])); gb = __dadd_rn(gb, ui > 0 ? d : -d); }
                if (uj) { const double d = __dmul_rn(C, (double) (float) ((double) (yj * yk) * Kj[c])); gb = __dadd_rn(gb, uj > 0 ? d : -d); }
                gbar[k] = gb;
            }
        }
        __syncthreads();
    }
    __syncthreads();
    /* ---- rho over the active set, objective and nu over all: in position order, one thread (libsvm sums
     * sequentially) ---- */
    if (tid == 0) {
        int nr_free = 0, nsv = 0;
        double ub = INFINITY, lb = -INFINITY, sum_free = 0.0, obj = 0.0, asum = 0.0;
        for (int k = 0; k < l; k++) {
            const double a = A[k], yG = (double) y[k] * G[k];
            if (k < act) {
                if (a >= C) { if (y[k] < 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
                else if (a <= 0.0) { if (y[k] > 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
                else { nr_free++; sum_free = __dadd_rn(sum_free, yG); }
            }
            obj = __dadd_rn(obj, __dmul_rn(a, __dadd_rn(G[k], -1.0)));
            if (a > 0.0) { nsv++; asum += a; }
        }
        gkm_svm_fit f;
        f.rho = nr_free > 0 ? sum_free / (double) nr_free : (ub + lb) / 2.0;
        f.obj = obj / 2.0;
        f.n_iter = iter;
        f.n_sv = nsv;
        f.nu = asum / (double) l; /* what gkmsvm.py:120 logs: sum |dual_coef| / len(y_train) */
        f.reserved = 0;
        fits[blockIdx.x] = f;
        if (SHRINK) {
            gkm_svm_shrink_stats s;
            s.shrink_passes = passes;
            s.min_active = min_act;
            s.unshrink_iter = unshrink_iter;
            s.recon_a = recon_a;
            s.recon_b = recon_b;
            s.reserved = 0;
            sb.stats[blockIdx.x] = s;
        }
    }
    /* alpha back in grouped order (libsvm: alpha_[active_set[i]] = alpha[i]) */
    for (int k = tid; k < l; k += SVM_THREADS) alpha_out[t.train_off + (SHRINK ? aset[k] : k)] = A[k];
}

/* decision values of the test points of every fit: one thread per test point, support vectors in model order */
__global__ void __launch_bounds__(256)
gkm_svm_decision_kernel(const double *__restrict__ K, long long ld, const gkm_svm_task *__restrict__ tasks,
                        const int *__restrict__ train_idx, const signed char *__restrict__ train_y,
                        const int *__restrict__ test_idx, const double *__restrict__ alpha,
                        const gkm_svm_fit *__restrict__ fits, double *__restrict__ scores)
{
    const gkm_svm_task t = tasks[blockIdx.y];
    const int r = (int) (blockIdx.x * blockDim.x + threadIdx.x);
    if (r >= t.ntest) return;
    const double *Kr = K + (size_t) test_idx[t.test_off + r] * (size_t) ld;
    const int *gi = train_idx + t.train_off;
    const signed char *gy = train_y + t.train_off;
    const double *a = alpha + t.train_off;
    double sum = 0.0;
    for (int k = 0; k < t.ntrain; k++) {
        const double ak = a[k];
        if (ak > 0.0) sum = __dadd_rn(sum, __dmul_rn(__dmul_rn(ak, (double) gy[k]), Kr[gi[k]]));
    }
    /* libsvm's value is positive for the class that got y = +1 (label 0); sklearn reports its negative */
    scores[t.test_off + r] = -__dadd_rn(sum, -fits[blockIdx.y].rho);
}

/* lower triangle + unit diagonal (what the kernel pass leaves resident) -> full symmetric matrix */
__global__ void gkm_svm_symmetrize_kernel(double *K, long long ld, int n)
{
    __shared__ double tile[32][33];
    const int bx = (int) blockIdx.x, by = (int) blockIdx.y;
    if (bx > by) return; /* tiles on and below the diagonal carry the data */
    const int r0 = by * 32, c0 = bx * 32;
    for (int dy = (int) threadIdx.y; dy < 32; dy += (int) blockDim.y) {
        const int r = r0 + dy, c = c0 + (int) threadIdx.x;
        double v = 0.0;
        if (r < n && c < n) v = (c < r) ? K[(size_t) r * (size_t) ld + c] : (c == r ? 1.0 : K[(size_t) c * (size_t) ld + r]);
        tile[dy][threadIdx.x] = v;
    }
    __syncthreads();
    for (int dy = (int) threadIdx.y; dy < 32; dy += (int) blockDim.y) {
        /* write the tile itself (diagonal tiles: completes the upper part) and its mirror image */
        const int r = r0 + dy, c = c0 + (int) threadIdx.x;
        if (r < n && c < n) K[(size_t) r * (size_t) ld + c] = tile[dy][threadIdx.x];
        const int mr = c0 + dy, mc = r0 + (int) threadIdx.x;
        if (bx != by && mr < n && mc < n) K[(size_t) mr * (size_t) ld + mc] = tile[threadIdx.x][dy];
    }
}

__global__ void gkm_svm_diag_kernel(const double *K, long long ld, int n, double *qd)
{
    const int i = (int) (blockIdx.x * blockDim.x + threadIdx.x);
    if (i < n) qd[i] = K[(size_t) i * (size_t) ld + i];
}

int gkm_svm_diagonal(const double *d_K, long long ld, int n, double *d_qd, cudaStream_t st)
{
    gkm_svm_diag_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>(d_K, ld, n, d_qd);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int gkm_svm_symmetrize(double *d_K, long long ld, int n, cudaStream_t st)
{
    const unsigned nt = (unsigned) ((n + 31) / 32);
    gkm_svm_symmetrize_kernel<<<dim3(nt, nt, 1), dim3(32, 8, 1), 0, st>>>(d_K, ld, n);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

/* all device work of a batch of fits on a resident symmetric matrix; the arrays are host pointers */
int gkm_svm_run(const double *d_K, long long ld, int n, int ntasks, const gkm_svm_task *tasks,
                const int *train_idx, const signed char *train_y, const int *test_idx,
                double C, double eps, int max_iter, int shrinking, double *scores, gkm_svm_fit *fits, double *alpha,
                gkm_svm_shrink_stats *stats, cudaStream_t st)
{
    if (ntasks <= 0) return 0;
    long long ntrain = 0, ntest = 0;
    int lmax = 0, tmax = 0;
    for (int t = 0; t < ntasks; t++) {
        if (tasks[t].ntrain < 2 || tasks[t].ntest < 0) { gkm_set_error("svm task %d: needs at least two training points", t); return 1; }
        if (tasks[t].train_off != ntrain || tasks[t].test_off != ntest) { gkm_set_error("svm task %d: offsets must be consecutive", t); return 1; }
        ntrain += tasks[t].ntrain; ntest += tasks[t].ntest;
        if (tasks[t].ntrain > lmax) lmax = tasks[t].ntrain;
        if (tasks[t].ntest > tmax) tmax = tasks[t].ntest;
    }
    for (long long k = 0; k < ntrain; k++) if (train_idx[k] < 0 || train_idx[k] >= n || (train_y[k] != 1 && train_y[k] != -1)) { gkm_set_error("svm: bad training index or label"); return 1; }
    for (long long k = 0; k < ntest; k++) if (test_idx[k] < 0 || test_idx[k] >= n) { gkm_set_error("svm: bad test index"); return 1; }
    /* one class only: the solver would stop at once and rho = (ub + lb) / 2 would be infinite */
    for (int t = 0; t < ntasks; t++) {
        int npos = 0;
        for (int k = 0; k < tasks[t].ntrain; k++) npos += train_y[tasks[t].train_off + k] > 0;
        if (npos == 0 || npos == tasks[t].ntrain) { gkm_set_error("svm task %d: the training labels must contain both +1 and -1", t); return 1; }
    }
    if (max_iter < 0) max_iter = 10000000 > 100 * lmax ? 10000000 : 100 * lmax; /* libsvm's own ceiling */

    gkm_svm_task *d_tasks = NULL; int *d_tr = NULL, *d_te = NULL; signed char *d_y = NULL;
    double *d_alpha = NULL, *d_g = NULL, *d_scores = NULL, *d_qd = NULL; gkm_svm_fit *d_fits = NULL;
    svm_shrink_buf sb = {NULL, NULL, NULL, NULL, NULL, NULL};
    const size_t smem_need = (size_t) lmax * 21 + 64;
    const int in_smem = smem_need <= 220u * 1024u;
    int rc = 0;
    cudaError_t e = cudaSuccess;
#define SVM_CK(call) do { if (!rc && (e = (call)) != cudaSuccess) { gkm_set_error("CUDA: %s -> %s", #call, cudaGetErrorString(e)); rc = 1; } } while (0)
    SVM_CK(cudaMalloc(&d_tasks, sizeof(gkm_svm_task) * (size_t) ntasks));
    SVM_CK(cudaMalloc(&d_tr, sizeof(int) * (size_t) (ntrain ? ntrain : 1)));
    SVM_CK(cudaMalloc(&d_te, sizeof(int) * (size_t) (ntest ? ntest : 1)));
    SVM_CK(cudaMalloc(&d_y, (size_t) (ntrain ? ntrain : 1)));
    SVM_CK(cudaMalloc(&d_alpha, sizeof(double) * (size_t) (ntrain ? ntrain : 1)));
    SVM_CK(cudaMalloc(&d_scores, sizeof(double) * (size_t) (ntest ? ntest : 1)));
    SVM_CK(cudaMalloc(&d_fits, sizeof(gkm_svm_fit) * (size_t) ntasks));
    SVM_CK(cudaMalloc(&d_qd, sizeof(double) * (size_t) n));
    if (!rc && gkm_svm_diagonal(d_K, ld, n, d_qd, st)) { gkm_set_error("CUDA: svm diagonal kernel failed"); rc = 1; }
    if (!in_smem) SVM_CK(cudaMalloc(&d_g, sizeof(double) * 2 * (size_t) ntrain));
    if (shrinking) {
        SVM_CK(cudaMalloc(&sb.gbar, sizeof(double) * (size_t) ntrain));
        SVM_CK(cudaMalloc(&sb.aset, sizeof(int) * (size_t) ntrain));
        SVM_CK(cudaMalloc(&sb.pairs, sizeof(int) * (size_t) ntrain));
        SVM_CK(cudaMalloc(&sb.stats, sizeof(gkm_svm_shrink_stats) * (size_t) ntasks));
        if (!in_smem) {
            SVM_CK(cudaMalloc(&sb.idx, sizeof(int) * (size_t) ntrain));
            SVM_CK(cudaMalloc(&sb.y, (size_t) ntrain));
        }
    }
    SVM_CK(cudaMemcpyAsync(d_tasks, tasks, sizeof(gkm_svm_task) * (size_t) ntasks, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_tr, train_idx, sizeof(int) * (size_t) ntrain, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_te, test_idx, sizeof(int) * (size_t) ntest, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_y, train_y, (size_t) ntrain, cudaMemcpyHostToDevice, st));
    if (!rc) {
        const unsigned smem = in_smem ? (unsigned) ((smem_need + 15) & ~(size_t) 15) : 0u;
        const void *kfn = shrinking ? (const void *) gkm_svm_smo_kernel<true> : (const void *) gkm_svm_smo_kernel<false>;
        SVM_CK(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
        if (!rc) {
            if (shrinking)
                gkm_svm_smo_kernel<true><<<(unsigned) ntasks, SVM_THREADS, smem, st>>>(d_K, ld, d_qd, d_tasks, d_tr, d_y, C, eps, max_iter, in_smem, d_alpha, d_g, sb, d_fits);
            else
                gkm_svm_smo_kernel<false><<<(unsigned) ntasks, SVM_THREADS, smem, st>>>(d_K, ld, d_qd, d_tasks, d_tr, d_y, C, eps, max_iter, in_smem, d_alpha, d_g, sb, d_fits);
            SVM_CK(cudaGetLastError());
        }
        if (!rc && tmax > 0) {
            gkm_svm_decision_kernel<<<dim3((unsigned) ((tmax + 255) / 256), (unsigned) ntasks, 1), 256, 0, st>>>(d_K, ld, d_tasks, d_tr, d_y, d_te, d_alpha, d_fits, d_scores);
            SVM_CK(cudaGetLastError());
        }
    }
    if (scores && ntest) SVM_CK(cudaMemcpyAsync(scores, d_scores, sizeof(double) * (size_t) ntest, cudaMemcpyDeviceToHost, st));
    if (fits) SVM_CK(cudaMemcpyAsync(fits, d_fits, sizeof(gkm_svm_fit) * (size_t) ntasks, cudaMemcpyDeviceToHost, st));
    if (alpha && ntrain) SVM_CK(cudaMemcpyAsync(alpha, d_alpha, sizeof(double) * (size_t) ntrain, cudaMemcpyDeviceToHost, st));
    if (stats && shrinking) SVM_CK(cudaMemcpyAsync(stats, sb.stats, sizeof(gkm_svm_shrink_stats) * (size_t) ntasks, cudaMemcpyDeviceToHost, st));
    SVM_CK(cudaStreamSynchronize(st));
#undef SVM_CK
    if (!rc && stats && !shrinking)
        for (int t = 0; t < ntasks; t++) {
            const gkm_svm_shrink_stats s = {0, tasks[t].ntrain, -1, 0, 0, 0}; /* the whole set stays active */
            stats[t] = s;
        }
    cudaFree(d_tasks); cudaFree(d_tr); cudaFree(d_te); cudaFree(d_y); cudaFree(d_alpha); cudaFree(d_g); cudaFree(d_scores); cudaFree(d_fits); cudaFree(d_qd);
    cudaFree(sb.gbar); cudaFree(sb.aset); cudaFree(sb.pairs); cudaFree(sb.idx); cudaFree(sb.y); cudaFree(sb.stats);
    return rc;
}
