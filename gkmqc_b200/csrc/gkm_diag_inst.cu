/* gkm_diag_inst.cu -- instantiates the bit-sliced kernel for ONE word length.
 * Compiled once per L = 2..16 with -DGKM_INST_L=<L> (see Makefile) so that the
 * specialisations (15 L x {4,8,16} bins x {plain, weighted}, + d = 4) build in parallel. */
#include "gkm_diag_kernel.cuh"

#ifndef GKM_INST_L
#error "compile with -DGKM_INST_L=<word length>"
#endif

#define GKM_CAT2(a, b) a##b
#define GKM_CAT(a, b) GKM_CAT2(a, b)

template <int NB, bool WEIGHTED>
static const void *pick(int d)
{
    return gkm_diag_instance<NB, WEIGHTED>(d, [](auto d4) {
        return (const void *) gkm_diag_kernel<GKM_INST_L, NB, WEIGHTED, decltype(d4)::value>;
    });
}

extern "C" const void *GKM_CAT(gkm_diag_fn_L, GKM_INST_L)(int nb, int weighted, int d)
{
    if (nb == 4) return weighted ? pick<4, true>(d) : pick<4, false>(d);
    if (nb == 8) return weighted ? pick<8, true>(d) : pick<8, false>(d);
    if (nb == 16) return weighted ? pick<16, true>(d) : pick<16, false>(d);
    return nullptr;
}
