// Haweel's T with the retained-coefficient masks (first k = 6..10 zig-zag coefficients, JPEG Q) as compile-time
// constants (see inst_direct_k.cu).  Fused round trips only (tma_compiled).
#define INST_TK TK_HAWEEL
#define INST_Q Q_IMM_K6, Q_IMM_K7, Q_IMM_K8, Q_IMM_K9, Q_IMM_K10
#define INST_TAG k
#include "inst_tma.cuh"
