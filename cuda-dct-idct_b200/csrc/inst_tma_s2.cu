#define INST_TK TK_HAWEEL
#define INST_Q Q_PARAM_DIV
#define INST_TAG s2
#include "inst_tma.cuh"
