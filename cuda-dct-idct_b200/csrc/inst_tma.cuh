// inst_tma.cuh -- instantiates k_tma for one (T family, quantiser) pair (see inst_direct.cuh).
#include "dct_kernels.cuh"

namespace b200dct {

#define B200_CAT_(a, b) a##b
#define B200_CAT(a, b) B200_CAT_(a, b)

#define B200_TMA_CASE(M, X, F) B200_TMA_CASE_M(M, X, F, false)
#define B200_TMA_CASE_M(M, X, F, MET)                                                                 \
    if (mode == (M) && pix == (X) && finv == (F) && (P.macc != nullptr) == (MET)) {                   \
        constexpr auto kern = k_tma<M, INST_SPARSE, INST_Q, X, F, MET>;                               \
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        if (e != cudaSuccess) return e;                                                               \
        return launch_kernel<kern>(P, dim3((unsigned)grid), dim3((unsigned)block), smem, s, pdl);     \
    }

cudaError_t B200_CAT(launch_tma_, INST_TAG)(int mode, int pix, bool finv, const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl)
{
    B200_TMA_CASE(MODE_RT, DT_F32, false)
    B200_TMA_CASE(MODE_RT, DT_U8, false)
#if INST_SPARSE == 1
    B200_TMA_CASE(MODE_RT, DT_U8, true)
    B200_TMA_CASE_M(MODE_RT, DT_F32, false, true) // fused MSE / PEEN / non-zero count (P.macc != NULL)
#endif
    B200_TMA_CASE(MODE_FWD, DT_F32, false)
    B200_TMA_CASE(MODE_FWD, DT_U8, false)
    B200_TMA_CASE(MODE_INV, DT_F32, false)
    B200_TMA_CASE(MODE_INV, DT_U8, false)
#if INST_SPARSE == 1
    B200_TMA_CASE(MODE_INV, DT_U8, true)
#endif
    return cudaErrorInvalidValue;
}

} // namespace b200dct
