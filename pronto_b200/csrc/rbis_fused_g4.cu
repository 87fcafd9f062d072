// Warp-group kernels (rbis_group.cuh), 4 lanes per filter, decoupled and dense.
#define RBIS_TU_NAME g4
#define RBIS_TU_NS rbisk_g4
#define RBIS_TU_GROUP 4
#include "rbis_fused_tu.inc"
