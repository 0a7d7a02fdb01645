// inst_any.cuh -- instantiates the any-size round trips (any_kernels.cuh) for one pixel type: INST_PIX = DT_F32 (k_any)
// / DT_U8 (k_any_u8, word-packed, no shared-memory stage), INST_TAG = name suffix.  Every (T family, quantiser,
// factored inverse) that any_compiled() allows is compiled here.
#include "any_kernels.cuh"

namespace b200dct {

cudaError_t B200_CAT(launch_any_, INST_TAG)(int tk, int qm, bool finv, const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl)
{
    return pick<TK_DENSE, TK_HAWEEL, TK_DENSE_SYM>(tk, [&](auto t) {
        return pick<Q_IMM, Q_PARAM, Q_PARAM_DIV>(qm, [&](auto q) {
            return pick<false, true>(finv, [&](auto fi) {
                if constexpr (!any_compiled(IC(t), IC(q), MODE_RT, INST_PIX, IC(fi), false))
                    return cudaErrorInvalidValue;
                else if constexpr (INST_PIX == DT_U8)
                    return launch_kernel<k_any_u8<IC(t), IC(q), IC(fi)>>(P, grid, block, 0, s, pdl);
                else
                    return launch_kernel<k_any<IC(t), IC(q), INST_PIX, IC(fi)>>(P, grid, block, 0, s, pdl);
            });
        });
    });
}

} // namespace b200dct
