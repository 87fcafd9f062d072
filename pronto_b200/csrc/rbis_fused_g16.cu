// Warp-group kernels (rbis_group.cuh), 16 lanes per filter, decoupled and dense.
#define RBIS_TU_NAME g16
#define RBIS_TU_NS rbisk_g16
#define RBIS_TU_GROUP 16
#include "rbis_fused_tu.inc"
