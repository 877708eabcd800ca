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
 * Shrinking (gkmQC's default is off, bin/gkmqc.py:209) is not implemented: it changes the path, not the optimum.
 *
 * Data: the symmetric n x n matrix is resident in HBM (ld doubles per row); per fit G, alpha, the gather index
 * and y live in shared memory (21 bytes per training point: 10 800 points fit), every iteration reads two
 * kernel rows through the gather index.  Bound: latency of two block-wide arg-reductions per iteration; the
 * 50 fits of a bin run concurrently, one per SM.
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

/* one fit per CTA */
__global__ void __launch_bounds__(SVM_THREADS, 1)
gkm_svm_smo_kernel(const double *__restrict__ K, long long ld, const double *__restrict__ qd, const gkm_svm_task *__restrict__ tasks,
                   const int *__restrict__ train_idx, const signed char *__restrict__ train_y,
                   double C, double eps, int max_iter, int in_smem,
                   double *__restrict__ alpha_out, double *__restrict__ g_scratch, gkm_svm_fit *__restrict__ fits)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ svm_pick red_pick[32];
    __shared__ double red_max[32];
    __shared__ double sh_d[4];

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
        idx = const_cast<int *>(gidx);
        y = const_cast<signed char *>(gy);
    }
    for (int k = tid; k < l; k += SVM_THREADS) {
        G[k] = -1.0; /* p_i = -1, alpha = 0 */
        A[k] = 0.0;
        if (in_smem) { idx[k] = gidx[k]; y[k] = gy[k]; }
    }
    __syncthreads();

    int iter = 0;
    for (;;) {
        /* ---- i: maximal -y G over I_up ---- */
        svm_pick pi; pi.v = -INFINITY; pi.i = -1;
        for (int k = tid; k < l; k += SVM_THREADS) {
            const double a = A[k], g = G[k];
            if (y[k] > 0) { if (a < C && -g >= pi.v) { pi.v = -g; pi.i = k; } }
            else          { if (a > 0.0 && g >= pi.v) { pi.v = g; pi.i = k; } }
        }
        pi = svm_block_argmax(pi, red_pick);
        const int i = pi.i;
        const double Gmax = pi.v;
        if (i < 0) break;
        /* ---- j: second-order choice over I_low; Q_i row through the gather index ---- */
        const double *Ki = K + (size_t) idx[i] * (size_t) ld;
        const int yi = y[i];
        const double QDi = qd[idx[i]];
        svm_pick pj; pj.v = -INFINITY; pj.i = -1; /* maximise -obj_diff = b*b/a, ties -> last index */
        double gmax2 = -INFINITY;
        for (int k = tid; k < l; k += SVM_THREADS) {
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
        if (Gmax + gmax2 < eps || j < 0) break;
        if (iter >= max_iter) break;
        iter++;
        /* ---- analytic step on (alpha_i, alpha_j) ---- */
        const double *Kj = K + (size_t) idx[j] * (size_t) ld;
        const int yj = y[j];
        if (tid == 0) {
            const float qij = (float) ((double) (yi * yj) * Ki[idx[j]]);
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
        }
        __syncthreads();
        const double dai = sh_d[0], daj = sh_d[1];
        /* ---- gradient ---- */
        for (int k = tid; k < l; k += SVM_THREADS) {
            const int yk = y[k];
            const int c = idx[k];
            const float qik = (float) ((double) (yi * yk) * Ki[c]);
            const float qjk = (float) ((double) (yj * yk) * Kj[c]);
            G[k] = __dadd_rn(G[k], __dadd_rn(__dmul_rn((double) qik, dai), __dmul_rn((double) qjk, daj)));
        }
        __syncthreads();
    }
    __syncthreads();
    /* ---- rho, objective, nu: in index order, one thread (libsvm sums sequentially) ---- */
    if (tid == 0) {
        int nr_free = 0, nsv = 0;
        double ub = INFINITY, lb = -INFINITY, sum_free = 0.0, obj = 0.0, asum = 0.0;
        for (int k = 0; k < l; k++) {
            const double a = A[k], yG = (double) y[k] * G[k];
            if (a >= C) { if (y[k] < 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
            else if (a <= 0.0) { if (y[k] > 0) ub = fmin(ub, yG); else lb = fmax(lb, yG); }
            else { nr_free++; sum_free = __dadd_rn(sum_free, yG); }
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
    }
    for (int k = tid; k < l; k += SVM_THREADS) alpha_out[t.train_off + k] = A[k];
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
                double C, double eps, int max_iter, double *scores, gkm_svm_fit *fits, double *alpha, cudaStream_t st)
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
    SVM_CK(cudaMemcpyAsync(d_tasks, tasks, sizeof(gkm_svm_task) * (size_t) ntasks, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_tr, train_idx, sizeof(int) * (size_t) ntrain, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_te, test_idx, sizeof(int) * (size_t) ntest, cudaMemcpyHostToDevice, st));
    SVM_CK(cudaMemcpyAsync(d_y, train_y, (size_t) ntrain, cudaMemcpyHostToDevice, st));
    if (!rc) {
        const unsigned smem = in_smem ? (unsigned) ((smem_need + 15) & ~(size_t) 15) : 0u;
        SVM_CK(cudaFuncSetAttribute((const void *) gkm_svm_smo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
        if (!rc) {
            gkm_svm_smo_kernel<<<(unsigned) ntasks, SVM_THREADS, smem, st>>>(d_K, ld, d_qd, d_tasks, d_tr, d_y, C, eps, max_iter, in_smem, d_alpha, d_g, d_fits);
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
    SVM_CK(cudaStreamSynchronize(st));
#undef SVM_CK
    cudaFree(d_tasks); cudaFree(d_tr); cudaFree(d_te); cudaFree(d_y); cudaFree(d_alpha); cudaFree(d_g); cudaFree(d_scores); cudaFree(d_fits); cudaFree(d_qd);
    return rc;
}
