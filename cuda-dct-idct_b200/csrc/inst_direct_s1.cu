#define INST_TK TK_HAWEEL
#define INST_Q Q_PARAM
#define INST_TAG s1
#include "inst_direct.cuh"
