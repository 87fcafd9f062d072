// Warp-group kernels (rbis_group.cuh), 2 lanes per filter, decoupled and dense.
#define RBIS_TU_NAME g2
#define RBIS_TU_NS rbisk_g2
#define RBIS_TU_GROUP 2
#include "rbis_fused_tu.inc"
