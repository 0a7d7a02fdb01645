#define INST_TK TK_DENSE
#define INST_Q Q_PARAM
#define INST_TAG d1
#include "inst_direct.cuh"
