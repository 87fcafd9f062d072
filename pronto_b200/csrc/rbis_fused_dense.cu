// Dense lane-per-filter kernels, 256 filters per CTA (2 warps per scheduler), all 231 covariance slots on chip: any
// covariance and any program, including those that the decoupled kernels cannot run.
#define RBIS_TU_NAME dense
#define RBIS_TU_NS rbisk_dense
#define RBIS_TU_DENSE
#define RBIS_TPB 256
#define RBIS_PLACEMENT 1
#include "rbis_fused_tu.inc"
