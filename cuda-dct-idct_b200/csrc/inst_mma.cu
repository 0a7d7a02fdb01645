// inst_mma.cu -- the tensor-core arm of the dense-T round trip (mma_kernels.cuh)
#include "mma_kernels.cuh"

namespace b200dct {

cudaError_t launch_mma(bool fastdiv, const MmaParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl)
{
    return fastdiv ? launch_kernel<k_mma<true>>(P, grid, block, 0, s, pdl) : launch_kernel<k_mma<false>>(P, grid, block, 0, s, pdl);
}

} // namespace b200dct
