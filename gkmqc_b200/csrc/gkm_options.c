/* gkm_options.c -- process-wide knobs.  The reference's whole configuration surface is
 * the gkmOpt struct (libgkm.h:149-161), which cannot grow without breaking the ABI, so
 * everything GPU-specific comes from gkmb200_set_option() or the environment:
 *   GKM_KERNEL   = auto | lmer | diag | mma | index   kernel variant (mma = tcgen05 one-hot GEMM candidate,
 *                                           index = inverted L-mer index; auto picks diag or index by a cost model)
 *   GKM_MAX_L    = 12 | 16                 ceiling of the parameter gate in gkm_main_pywrapper
 *   GKM_CHUNK_MB = n                       upper bound of one chunk's dense output
 *   GKM_INDEX_COLS = n                     upper bound of the columns of one index block (tests: forces several blocks)
 *   GKM_INDEX_SPLIT = equal | greedy       how a column range is cut into index blocks: equal shares, or full blocks first
 *   GKM_DEVICES  = "0,1,.."                GPUs to use (gkm_device.cu)
 */
#include <stdlib.h>
#include <string.h>

#include "gkm_internal.h"
#include "gkm_options.h"

static int g_loaded = 0;
static int g_kernel = GKM_KERNEL_AUTO;
static int g_max_L = 12;
static int g_chunk_mb = 128; /* 50k x 50k: 686 ms per pass with 64 MB chunks (one wave of 148 rows each), 671 with 128, 669 with 256 */
static int g_index_cols = 0;
static int g_index_wide = 0;
static int g_index_greedy = -1; /* -1: the library decides per call */

static int parse_kernel(const char *v, int *out)
{
    if (!strcmp(v, "auto")) *out = GKM_KERNEL_AUTO;
    else if (!strcmp(v, "lmer")) *out = GKM_KERNEL_LMER;
    else if (!strcmp(v, "diag")) *out = GKM_KERNEL_DIAG;
    else if (!strcmp(v, "mma")) *out = GKM_KERNEL_MMA;
    else if (!strcmp(v, "index")) *out = GKM_KERNEL_INDEX;
    else return 1;
    return 0;
}

static void load_env(void)
{
    if (g_loaded) return;
    g_loaded = 1;
    const char *v;
    if ((v = getenv("GKM_KERNEL")) != NULL) parse_kernel(v, &g_kernel);
    if ((v = getenv("GKM_MAX_L")) != NULL) { int x = atoi(v); if (x == 12 || x == 16) g_max_L = x; }
    if ((v = getenv("GKM_CHUNK_MB")) != NULL) { int x = atoi(v); if (x >= 1 && x <= 4096) g_chunk_mb = x; }
    if ((v = getenv("GKM_INDEX_COLS")) != NULL) { int x = atoi(v); if (x >= 32) g_index_cols = x & ~31; }
    if ((v = getenv("GKM_INDEX_WIDE")) != NULL) g_index_wide = atoi(v) != 0;
    if ((v = getenv("GKM_INDEX_SPLIT")) != NULL) g_index_greedy = !strcmp(v, "greedy") ? 1 : !strcmp(v, "equal") ? 0 : -1;
}

int gkm_opt_kernel(void) { load_env(); return g_kernel; }
int gkm_opt_max_L(void) { load_env(); return g_max_L; }
int gkm_opt_chunk_mb(void) { load_env(); return g_chunk_mb; }
int gkm_opt_index_cols(void) { load_env(); return g_index_cols; }
int gkm_opt_index_wide(void) { load_env(); return g_index_wide; }
int gkm_opt_index_greedy(void) { load_env(); return g_index_greedy; }

int gkmb200_set_option(const char *key, const char *value)
{
    load_env();
    if (!key || !value) { gkm_set_error("null option"); return 1; }
    if (!strcmp(key, "kernel")) {
        if (parse_kernel(value, &g_kernel)) { gkm_set_error("kernel must be auto, lmer, diag, mma or index"); return 1; }
        return 0;
    }
    int x = atoi(value);
    if (!strcmp(key, "max_L")) {
        if (x != 12 && x != 16) { gkm_set_error("max_L must be 12 or 16"); return 1; }
        g_max_L = x;
        return 0;
    }
    if (!strcmp(key, "chunk_mb")) {
        if (x < 1 || x > 4096) { gkm_set_error("chunk_mb out of range"); return 1; }
        g_chunk_mb = x;
        return 0;
    }
    if (!strcmp(key, "index_cols")) { /* upper bound of the columns of one index block (0 = what fits shared memory) */
        if (x != 0 && x < 32) { gkm_set_error("index_cols must be 0 or >= 32"); return 1; }
        g_index_cols = x & ~31;
        return 0;
    }
    if (!strcmp(key, "index_wide")) { /* 1: 16-byte slots even where the compact 8-byte ones would do (A/B, tests) */
        g_index_wide = x != 0;
        return 0;
    }
    if (!strcmp(key, "index_split")) { /* equal: blocks of equal size; greedy: full blocks first, the rest last; auto: per call */
        if (strcmp(value, "equal") && strcmp(value, "greedy") && strcmp(value, "auto")) { gkm_set_error("index_split must be equal, greedy or auto"); return 1; }
        g_index_greedy = !strcmp(value, "greedy") ? 1 : !strcmp(value, "equal") ? 0 : -1;
        return 0;
    }
    gkm_set_error("unknown option %s", key);
    return 1;
}

int gkmb200_abi_version(void) { return 1; }
