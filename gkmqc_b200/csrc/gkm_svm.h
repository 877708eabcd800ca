/* gkm_svm.h -- device side of the C-SVC cross-validation consumer (gkm_svm.cu), used by gkm_resident.cu */
#ifndef GKM_SVM_H_INCLUDED
#define GKM_SVM_H_INCLUDED

#include <cuda_runtime.h>

#include "../../include/gkm_b200.h"

typedef gkmb200_svm_task gkm_svm_task;
typedef gkmb200_svm_fit gkm_svm_fit;
typedef gkmb200_svm_shrink_stats gkm_svm_shrink_stats;

/* lower triangle (+ anything on and above the diagonal) -> symmetric matrix with unit diagonal, in place */
int gkm_svm_symmetrize(double *d_K, long long ld, int n, cudaStream_t st);
/* d_qd[i] = d_K[i][i] */
int gkm_svm_diagonal(const double *d_K, long long ld, int n, double *d_qd, cudaStream_t st);
/* ntasks fits + the decision values of their test points on the resident symmetric matrix d_K; shrinking = 1 runs
 * libsvm's shrinking heuristic.  tasks / train_idx / train_y / test_idx and the outputs are HOST arrays (scores, fits,
 * alpha, stats may be NULL); synchronises the stream. */
int gkm_svm_run(const double *d_K, long long ld, int n, int ntasks, const gkm_svm_task *tasks,
                const int *train_idx, const signed char *train_y, const int *test_idx,
                double C, double eps, int max_iter, int shrinking, double *scores, gkm_svm_fit *fits, double *alpha,
                gkm_svm_shrink_stats *stats, cudaStream_t st);

#endif
