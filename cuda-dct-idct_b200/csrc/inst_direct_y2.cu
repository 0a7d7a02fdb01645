// dense T with symmetric even / antisymmetric odd rows (TK_DENSE_SYM), quantiser variant 2
#define INST_TK TK_DENSE_SYM
#define INST_Q Q_PARAM_DIV
#define INST_TAG y2
#include "inst_direct.cuh"
