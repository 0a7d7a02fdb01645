// inst_direct.cuh -- instantiates k_direct for one translation unit: INST_TK = TK_DENSE / TK_HAWEEL / TK_DENSE_SYM,
// INST_Q = its quantiser (Q_IMM / Q_PARAM / Q_PARAM_DIV) or list of them (Q_IMM_K6..K10), INST_TAG = name suffix.
// Every (mode, pixel type, factored inverse, metrics) that direct_compiled() allows is compiled here.
// One small translation unit per (T family, quantiser) keeps the parallel build short.
#include "dct_kernels.cuh"

namespace b200dct {

// ctas_per_sm != NULL: no launch, only the occupancy of the kernel the arguments select
cudaError_t B200_CAT(launch_direct_, INST_TAG)(int qm, int mode, int pix, bool finv, bool metrics, const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    return pick_kernel<INST_Q>(qm, mode, pix, finv, metrics, [&](auto q, auto m, auto x, auto fi, auto me) {
        if constexpr (direct_compiled(INST_TK, IC(q), IC(m), IC(x), IC(fi), IC(me)))
            return launch_kernel<k_direct<IC(m), INST_TK, IC(q), IC(x), IC(me), IC(fi)>>(P, grid, block, P.zz_smem ? ZZ_SMEM_BYTES : 0, s, pdl, ctas_per_sm);
        else
            return cudaErrorInvalidValue;
    });
}

} // namespace b200dct
