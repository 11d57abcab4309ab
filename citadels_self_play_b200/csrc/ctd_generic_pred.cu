// ctd_generic_pred.cu -- one wave of cfr_pred (ctd_k_mccfr_pred) for any ruleset (see ctd_search.cuh), alone in its unit.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define CTD_DEVICE_ONLY 1
#define CTD_SEARCH_UNIT 1   /* every device function of this unit runs with the whole warp converged on the same scalar code (ctd_search.cuh) */
// measured (round 2 A/B, 4096 roots): node moves, fp64 division / exp and the byte shuffle inlined at their uses are 10 % faster
// than one out-of-line copy of each -- calls cost the search more (callee-saved registers through local memory on 32 lanes) than
// the extra 30 KB of image
#define CTD_NODE_MOVE_ATTR
#define CTD_MATH_ATTR
#define CTD_SHUFFLE_ATTR
#define CTD_NO_PLAYOUT_KERNEL 1
#define CTD_NO_TRAIN_KERNEL 1
#define CTD_MCCFR_KERNEL_NAME ctd_k_mccfr_unused
#define CTD_MCCFR_PRED_KERNEL_NAME ctd_k_mccfr_pred
#ifdef CTD_LAYOUT_HEADER   /* placement of the device functions by name order, see ctd_layout_classic.h / tools/layout_search.py */
#include CTD_LAYOUT_HEADER
#endif
#include "ctd_search.cuh"

cudaError_t ctd_mccfr_pred_generic_launch(const CtdPredArgs& p, int grid, cudaStream_t stream) {
  const size_t smem = p.fused ? CTD_PRED_FUSED_SMEM : 0;   // fused mode: per-warp activation buffers, more than 48 KB per block in all
  static bool opted = false;
  if (p.fused && !opted) {
    cudaError_t c = cudaFuncSetAttribute(ctd_k_mccfr_pred, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CTD_PRED_FUSED_SMEM);
    if (c != cudaSuccess) return c;
    opted = true;
  }
  ctd_k_mccfr_pred<<<grid, CTD_BLOCK, smem, stream>>>(p);
  return cudaGetLastError();
}
// fused != 0: occupancy with the fused mode's dynamic shared memory
cudaError_t ctd_mccfr_pred_generic_blocks_per_sm(int* per_sm, int fused) {
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_mccfr_pred, CTD_BLOCK, fused ? CTD_PRED_FUSED_SMEM : 0);
}
