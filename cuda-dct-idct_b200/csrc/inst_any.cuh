// inst_any.cuh -- instantiates k_any (single-pass round trip for any image size and alignment)
// for one pixel type: INST_PIX = DT_F32 / DT_U8, INST_TAG = name suffix.
#include "any_kernels.cuh"

namespace b200dct {

#define B200_CAT_(a, b) a##b
#define B200_CAT(a, b) B200_CAT_(a, b)

template <int TK, int QM, int PIX, bool FINV = false>
static cudaError_t launch_one(const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl)
{
    if constexpr (PIX == DT_U8) return launch_kernel<k_any_u8<TK, QM, FINV>>(P, grid, block, 0, s, pdl); // word-packed, no shared-memory stage
    else return launch_kernel<k_any<TK, QM, PIX, FINV>>(P, grid, block, 0, s, pdl);
}

template <int PIX>
static cudaError_t launch_pix(int tk, int qm, bool finv, const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl)
{
    const bool sparse = tk == TK_HAWEEL;
    if (tk == TK_DENSE_SYM) {
        if (qm == Q_PARAM) return launch_one<TK_DENSE_SYM, Q_PARAM, PIX>(P, grid, block, s, pdl);
        return launch_one<TK_DENSE_SYM, Q_PARAM_DIV, PIX>(P, grid, block, s, pdl);
    }
    if constexpr (PIX == DT_U8) {
        if (sparse && finv) { // factored +-1 LSB inverse: 8-bit pixels only
            if (qm == Q_IMM) return launch_one<TK_HAWEEL, Q_IMM, PIX, true>(P, grid, block, s, pdl);
            if (qm == Q_PARAM) return launch_one<TK_HAWEEL, Q_PARAM, PIX, true>(P, grid, block, s, pdl);
            return launch_one<TK_HAWEEL, Q_PARAM_DIV, PIX, true>(P, grid, block, s, pdl);
        }
    }
    if (sparse) {
        if (qm == Q_IMM) return launch_one<TK_HAWEEL, Q_IMM, PIX>(P, grid, block, s, pdl);
        if (qm == Q_PARAM) return launch_one<TK_HAWEEL, Q_PARAM, PIX>(P, grid, block, s, pdl);
        return launch_one<TK_HAWEEL, Q_PARAM_DIV, PIX>(P, grid, block, s, pdl);
    }
    if (qm == Q_PARAM) return launch_one<TK_DENSE, Q_PARAM, PIX>(P, grid, block, s, pdl);
    return launch_one<TK_DENSE, Q_PARAM_DIV, PIX>(P, grid, block, s, pdl);
}

cudaError_t B200_CAT(launch_any_, INST_TAG)(int tk, int qm, bool finv, const AnyParams &P, dim3 grid, dim3 block, cudaStream_t s, bool pdl)
{
    return launch_pix<INST_PIX>(tk, qm, finv, P, grid, block, s, pdl);
}

} // namespace b200dct
