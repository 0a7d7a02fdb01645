// inst_direct_k.cu -- fused round trips of the direct family with the retained-coefficient mask
// (first k = 6..10 zig-zag coefficients, JPEG Q, Haweel's T) as a compile-time constant: the
// chains feeding dropped coefficients are never emitted and the inverse skips the known zeros
// (476 instead of 1408 FMAs per block at k = 10).
#include "dct_kernels.cuh"

namespace b200dct {

template <int QM, int PIX>
static cudaError_t launch_one(const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    return launch_kernel<k_direct<MODE_RT, TK_HAWEEL, QM, PIX>>(P, grid, block, P.zz_smem ? ZZ_SMEM_BYTES : 0, s, pdl, ctas_per_sm);
}

template <int PIX>
static cudaError_t launch_k(int k, const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    switch (k) {
    case 6: return launch_one<Q_IMM_K6, PIX>(P, grid, block, s, pdl, ctas_per_sm);
    case 7: return launch_one<Q_IMM_K7, PIX>(P, grid, block, s, pdl, ctas_per_sm);
    case 8: return launch_one<Q_IMM_K8, PIX>(P, grid, block, s, pdl, ctas_per_sm);
    case 9: return launch_one<Q_IMM_K9, PIX>(P, grid, block, s, pdl, ctas_per_sm);
    case 10: return launch_one<Q_IMM_K10, PIX>(P, grid, block, s, pdl, ctas_per_sm);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_direct_kmask(int k, int pix, const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    if (pix == DT_U8) return launch_k<DT_U8>(k, P, grid, block, s, pdl, ctas_per_sm);
    if (pix == DT_F32) return launch_k<DT_F32>(k, P, grid, block, s, pdl, ctas_per_sm);
    return cudaErrorInvalidValue;
}

} // namespace b200dct
