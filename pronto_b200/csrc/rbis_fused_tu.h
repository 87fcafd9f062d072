// rbis_fused_tu.h -- what a fused-kernel translation unit (rbis_fused_tu.inc) exports to the host code in rbis_batch.cu.
#ifndef RBIS_FUSED_TU_H_
#define RBIS_FUSED_TU_H_
#include <cuda_runtime.h>
#include <cstddef>
struct rbis_fused_tu_t {
  int lanes_per_filter;  // 1: lane-per-filter kernels; 2/4/8/16: warp-group kernels
  int threads, smem;     // lane-per-filter kernels: fixed launch shape
  int max_warps;         // warp-group kernels: warps per CTA at most
  int filters_per_warp;
  int smem_doubles_per_filter;  // warp-group kernels: (dense << 16) | decoupled
  size_t kparams_bytes;
  cudaError_t (*prepare)();
  // blocks_variant: the program has one-row / correlated chunks (lane-per-filter kernels: instantiation with those paths)
  // decoupled: which kernels of a warp-group unit (it holds both); a lane-per-filter unit holds either kind and ignores it
  // syn: the SYN instantiation (input rows drawn inside the kernel, KParams::syn); decoupled kernels without blocks_variant only
  // rec: 1 the REC instantiation (the program has RBIS_OP_RECORD ops, KParams::rec); 2 the REC instantiation with the
  //      innovation path (INNOV: a MEAS op of the program writes an innovation set, KParams::innov)
  // mask: 1 the MASK instantiation (a stream of the program has RBIS_STREAM_SKIP_NAN_ROWS, KParams::skip_nan_streams); 2 the MASK
  //       instantiation with the NIS gates (GATE: a stream has a gate or an innovation set asks for INNOV_APPLIED,
  //       KParams::gate_streams); not with syn
  cudaError_t (*launch)(int blocks_variant, int decoupled, int syn, int rec, int mask, unsigned grid, int threads, int smem, cudaStream_t st,
                        const void* kparams);
};
extern "C" {
extern const rbis_fused_tu_t rbis_fused_tu_dense, rbis_fused_tu_dc384, rbis_fused_tu_dc256, rbis_fused_tu_dc128;
extern const rbis_fused_tu_t rbis_fused_tu_g2, rbis_fused_tu_g4, rbis_fused_tu_g8, rbis_fused_tu_g16;
}
#endif
