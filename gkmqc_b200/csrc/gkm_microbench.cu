/* gkm_microbench.cu -- micro-benchmarks of the B200 (gkm_dev_microbench): integer issue rates, the denominators of the
 * integer roofline; random 16-byte gathers from L2; shared-memory atomics the way the index variant issues them. */
#include "gkm_dev.h"

template <int OP>
__global__ void __launch_bounds__(256) gkm_mb_kernel(uint32_t *out, int iters, uint32_t seed)
{
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = seed * (uint32_t) (threadIdx.x + 1) + (uint32_t) i * 0x9E3779B9u;
    uint32_t y = seed ^ 0x5bd1e995u, z = seed + (uint32_t) blockIdx.x;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (OP == 0) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                if (OP == 1) asm volatile("shf.r.wrap.b32 %0, %0, %1, 7;" : "+r"(x[i]) : "r"(y));
                if (OP == 2) asm volatile("popc.b32 %0, %0;" : "+r"(x[i]));
                if (OP == 3) asm volatile("add.u32 %0, %0, %1;" : "+r"(x[i]) : "r"(y));
                if (OP == 4) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z));
                if (OP == 5) asm volatile("mad.hi.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z));
                /* mixes: do the pipes run side by side?  (ops counted: all of them) */
                if (OP == 6) { if (i & 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z)); }
                if (OP == 7) { if (i & 3) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("popc.b32 %0, %0;" : "+r"(x[i])); }
                if (OP == 8) { if (i == 0) asm volatile("popc.b32 %0, %0;" : "+r"(x[i]));
                               else if (i < 5) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[i]) : "r"(y), "r"(z));
                               else asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[i]) : "r"(y), "r"(z)); }
            }
        }
    }
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s ^= x[i];
    if (s == 0x12345u) out[0] = s;
}

/* random 16-byte gathers from a 64 MB (L2-resident) table, four independent loads per thread in flight:
 * the sector rate the "index" variant's slot probes can reach at best */
__global__ void __launch_bounds__(1024, 1) gkm_mb_gather_kernel(const uint4 *__restrict__ tab, uint32_t mask, int iters, uint32_t *out)
{
    uint32_t s = (blockIdx.x * 1024u + threadIdx.x) * 2654435761u + 12345u;
    uint32_t acc = 0;
    for (int i = 0; i < iters; i++) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            s = s * 1664525u + 1013904223u;
            v[u] = __ldg(tab + ((s >> 4) & mask));
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc ^= v[u].x ^ v[u].y ^ v[u].z ^ v[u].w;
    }
    if (acc == 0x9E3779B9u) out[0] = acc;
}

/* shared-memory atomic adds the way the index variant's hit path issues them: each warp instruction has ~`active` of
 * its 32 lanes on (a probe finds a posting in the wanted range for a few lanes only), each on a random column of an
 * 80 KB histogram row; two CTAs of 1024 threads per SM like the hot loop.  Result: atomics per second. */
__global__ void __launch_bounds__(1024, 2) gkm_mb_atoms_kernel(int iters, uint32_t ncols, uint32_t active, unsigned long long *total)
{
    extern __shared__ int32_t mbH[];
    for (uint32_t i = threadIdx.x; i < ncols; i += 1024u) mbH[i] = 0;
    __syncthreads();
    uint32_t s = (blockIdx.x * 1024u + threadIdx.x) * 2654435761u + 12345u;
    uint32_t cnt = 0;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            s ^= s << 13; s ^= s >> 17; s ^= s << 5;
            const uint32_t col = __umulhi(s, ncols);
            const bool on = ((s >> 3) & 31u) < active;
            if (on) atomicAdd(&mbH[col], 1);
            cnt += on;
        }
    }
    __syncthreads();
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xFFFFFFFFu, cnt, o);
    if ((threadIdx.x & 31u) == 0u) atomicAdd(total, (unsigned long long) cnt + (mbH[threadIdx.x % ncols] < 0 ? 1ull : 0ull));
}

/* device time of launch(rep) on g->sc: the best of repetitions 1..3 (repetition 0 warms up) */
template <class F>
static int best_ms(gkm_gpu *g, const F &launch, float *best)
{
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    *best = 1e30f;
    int rc = 0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, g->sc);
        launch(rep);
        cudaEventRecord(e1, g->sc);
        if (cudaEventSynchronize(e1) != cudaSuccess) { gkm_set_error("CUDA: microbench failed: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms < *best) *best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

static int microbench_atoms(gkm_gpu *g, int sms, uint32_t active, double *result)
{
    gkm_dbuf<unsigned long long> d(g); /* one counter per repetition */
    unsigned long long h = 0;
    if (d.alloc(4) != cudaSuccess) { gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    cudaMemsetAsync(d, 0, 4 * sizeof(h), g->sc);
    const uint32_t ncols = 20000;
    const unsigned smem = ncols * 4;
    const int iters = 4096;
    cudaFuncSetAttribute(gkm_mb_atoms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    float best;
    const int rc = best_ms(g, [&](int rep) { gkm_mb_atoms_kernel<<<2 * sms, 1024, smem, g->sc>>>(iters, ncols, active, d + rep); }, &best);
    if (!rc) cudaMemcpy(&h, d + 3, sizeof(h), cudaMemcpyDeviceToHost);
    if (!rc) *result = (double) h / ((double) best * 1e-3) / 1e9;
    return rc;
}

static int microbench_gather(gkm_gpu *g, int sms, double *result)
{
    const size_t slots = (size_t) 1 << 22; /* 4 Mi x 16 B = 64 MB, the size of the L = 11 slot table */
    gkm_dbuf<uint4> tab(g);
    gkm_dbuf<uint32_t> d(g);
    if (tab.alloc(slots) != cudaSuccess || d.alloc(16) != cudaSuccess) { gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError())); return 1; }
    cudaMemsetAsync(tab, 0x5A, slots * sizeof(uint4), g->sc);
    const int iters = 2048;
    float best;
    const int rc = best_ms(g, [&](int) { gkm_mb_gather_kernel<<<sms, 1024, 0, g->sc>>>(tab, (uint32_t) (slots - 1), iters, d); }, &best);
    if (!rc) *result = (double) sms * 1024.0 * (double) iters * 4.0 / ((double) best * 1e-3) / 1e9; /* 1e9 gathers (sectors) per second */
    return rc;
}

extern "C" int gkm_dev_microbench(const char *what, double *result)
{
    if (!what || !result) { gkm_set_error("null argument"); return 1; }
    static const struct { const char *name; void (*fn)(uint32_t *, int, uint32_t); } ops[] = {
        { "lop3", gkm_mb_kernel<0> }, { "shf", gkm_mb_kernel<1> }, { "popc", gkm_mb_kernel<2> }, { "iadd3", gkm_mb_kernel<3> },
        { "imad", gkm_mb_kernel<4> }, { "imadhi", gkm_mb_kernel<5> }, { "lop3+imad", gkm_mb_kernel<6> },
        { "lop3+popc", gkm_mb_kernel<7> }, { "lop3+imad+popc", gkm_mb_kernel<8> } };
    pthread_mutex_lock(&g_lock);
    int rc = ensure_selected();
    gkm_gpu *g = rc ? NULL : &g_gpu[g_sel[0]];
    if (!rc) rc = gpu_prepare(g, g_sel[0], 0, 0);
    if (!rc) {
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->id);
        int op = -1;
        for (int i = 0; i < (int) (sizeof(ops) / sizeof(ops[0])); i++) if (!strcmp(what, ops[i].name)) op = i;
        if (!strcmp(what, "gather16")) rc = microbench_gather(g, sms, result);
        else if (!strcmp(what, "atoms7")) rc = microbench_atoms(g, sms, 7u, result);
        else if (!strcmp(what, "atoms14")) rc = microbench_atoms(g, sms, 14u, result);
        else if (!strcmp(what, "atoms32")) rc = microbench_atoms(g, sms, 32u, result);
        else if (op < 0) { gkm_set_error("unknown microbench %s", what); rc = 1; }
        else {
            gkm_dbuf<uint32_t> d(g);
            const int iters = 4096, blocks = sms * 8;
            float best;
            if (d.alloc(16) != cudaSuccess) { gkm_set_error("CUDA: microbench buffers: %s", cudaGetErrorString(cudaGetLastError())); rc = 1; }
            else rc = best_ms(g, [&](int rep) { ops[op].fn<<<blocks, 256, 0, g->sc>>>(d, iters, 12345u + rep); }, &best);
            if (!rc) *result = (double) blocks * 256.0 * (double) iters * 32.0 / ((double) best * 1e-3) / 1e9;
        }
    }
    pthread_mutex_unlock(&g_lock);
    return rc;
}
