#define INST_TK TK_HAWEEL
#define INST_Q Q_IMM
#define INST_TAG s0
#include "inst_direct.cuh"
