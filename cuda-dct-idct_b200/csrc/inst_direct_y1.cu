// dense T with symmetric even / antisymmetric odd rows (TK_DENSE_SYM), quantiser variant 1
#define INST_TK TK_DENSE_SYM
#define INST_Q Q_PARAM
#define INST_TAG y1
#include "inst_direct.cuh"
