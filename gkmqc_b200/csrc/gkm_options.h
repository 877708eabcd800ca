#ifndef GKM_OPTIONS_H_INCLUDED
#define GKM_OPTIONS_H_INCLUDED
#ifdef __cplusplus
extern "C" {
#endif
enum { GKM_KERNEL_AUTO = 0, GKM_KERNEL_LMER = 1, GKM_KERNEL_DIAG = 2, GKM_KERNEL_MMA = 3, GKM_KERNEL_INDEX = 4 };
int gkm_opt_kernel(void);
int gkm_opt_max_L(void);
int gkm_opt_chunk_mb(void);
int gkm_opt_index_cols(void);
int gkm_opt_index_wide(void);
int gkm_opt_index_greedy(void); /* 1 greedy, 0 equal, -1 per call */
#ifdef __cplusplus
}
#endif
#endif
