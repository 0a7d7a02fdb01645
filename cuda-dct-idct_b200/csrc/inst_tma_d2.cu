#define INST_TK TK_DENSE
#define INST_Q Q_PARAM_DIV
#define INST_TAG d2
#include "inst_tma.cuh"
