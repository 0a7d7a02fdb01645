// inst_tma.cuh -- instantiates k_tma for one translation unit (see inst_direct.cuh): every (mode, pixel type, factored
// inverse, metrics) that tma_compiled() allows.
#include "dct_kernels.cuh"

namespace b200dct {

cudaError_t B200_CAT(launch_tma_, INST_TAG)(int qm, int mode, int pix, bool finv, bool metrics, const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl)
{
    return pick_kernel<INST_Q>(qm, mode, pix, finv, metrics, [&](auto q, auto m, auto x, auto fi, auto me) {
        if constexpr (tma_compiled(INST_TK, IC(q), IC(m), IC(x), IC(fi), IC(me))) {
            constexpr auto kern = k_tma<IC(m), INST_TK, IC(q), IC(x), IC(fi), IC(me)>;
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            return launch_kernel<kern>(P, dim3((unsigned)grid), dim3((unsigned)block), smem, s, pdl);
        } else {
            return cudaErrorInvalidValue;
        }
    });
}

} // namespace b200dct
