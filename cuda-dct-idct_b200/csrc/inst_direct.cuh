// inst_direct.cuh -- instantiates k_direct for one (T family, quantiser) pair:
//   INST_SPARSE = 1/0, INST_Q = Q_IMM / Q_PARAM / Q_PARAM_DIV, INST_TAG = name suffix.
// One small translation unit per pair keeps the parallel build short.
#include "dct_kernels.cuh"

namespace b200dct {

#define B200_CAT_(a, b) a##b
#define B200_CAT(a, b) B200_CAT_(a, b)

#define B200_DIRECT_CASE(M, X, F, MET)                                              \
    if (mode == (M) && pix == (X) && finv == (F) && metrics == (MET))               \
        return launch_kernel<k_direct<M, INST_SPARSE, INST_Q, X, MET, F>>(P, grid, block, smem, s, pdl, ctas_per_sm);

// ctas_per_sm != NULL: no launch, only the occupancy of the kernel the arguments select
cudaError_t B200_CAT(launch_direct_, INST_TAG)(int mode, int pix, bool finv, bool metrics, const DirectParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl, int *ctas_per_sm)
{
    const size_t smem = P.zz_smem ? ZZ_SMEM_BYTES : 0;
    // finv: factored +-1 LSB inverse (Haweel's T, 8-bit pixel output only)
    B200_DIRECT_CASE(MODE_RT, DT_F32, false, false)
    B200_DIRECT_CASE(MODE_RT, DT_U8, false, false)
#if INST_SPARSE == 1
    B200_DIRECT_CASE(MODE_RT, DT_U8, true, false)
#endif
    B200_DIRECT_CASE(MODE_FWD, DT_F32, false, false)
    B200_DIRECT_CASE(MODE_FWD, DT_U8, false, false)
    B200_DIRECT_CASE(MODE_INV, DT_F32, false, false)
    B200_DIRECT_CASE(MODE_INV, DT_U8, false, false)
#if INST_SPARSE == 1
    B200_DIRECT_CASE(MODE_INV, DT_U8, true, false)
    B200_DIRECT_CASE(MODE_RT, DT_U8, true, true)
#endif
    B200_DIRECT_CASE(MODE_RT, DT_F32, false, true)
    B200_DIRECT_CASE(MODE_RT, DT_U8, false, true)
    return cudaErrorInvalidValue;
}

} // namespace b200dct
