// inst_tma_k.cu -- fused round trips of the TMA family with the retained-coefficient mask
// (first k = 6..10 zig-zag coefficients, JPEG Q, Haweel's T) as a compile-time constant
// (see inst_direct_k.cu).
#include "dct_kernels.cuh"

namespace b200dct {

template <int QM, int PIX>
static cudaError_t launch_one(const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl)
{
    constexpr auto kern = k_tma<MODE_RT, TK_HAWEEL, QM, PIX>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    return launch_kernel<kern>(P, dim3((unsigned)grid), dim3((unsigned)block), smem, s, pdl);
}

template <int PIX>
static cudaError_t launch_k(int k, const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl)
{
    switch (k) {
    case 6: return launch_one<Q_IMM_K6, PIX>(P, grid, block, smem, s, pdl);
    case 7: return launch_one<Q_IMM_K7, PIX>(P, grid, block, smem, s, pdl);
    case 8: return launch_one<Q_IMM_K8, PIX>(P, grid, block, smem, s, pdl);
    case 9: return launch_one<Q_IMM_K9, PIX>(P, grid, block, smem, s, pdl);
    case 10: return launch_one<Q_IMM_K10, PIX>(P, grid, block, smem, s, pdl);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_tma_kmask(int k, int pix, const TmaParams &P, int grid, int block, size_t smem, cudaStream_t s, bool pdl)
{
    if (pix == DT_F32) return launch_k<DT_F32>(k, P, grid, block, smem, s, pdl);
    if (pix == DT_U8) return launch_k<DT_U8>(k, P, grid, block, smem, s, pdl);
    return cudaErrorInvalidValue;
}

} // namespace b200dct
