// Warp-group kernels (rbis_group.cuh), 8 lanes per filter, decoupled and dense.
#define RBIS_TU_NAME g8
#define RBIS_TU_NS rbisk_g8
#define RBIS_TU_GROUP 8
#include "rbis_fused_tu.inc"
