// ctd_preset_search.cu -- cfr_train (ctd_k_mccfr) specialised for the preset ruleset (see ctd_search.cuh).  Device code only,
// one kernel per translation unit: out-of-line device functions are compiled once per unit, under the tightest register
// bound of the kernels that call them, so a kernel shares its unit only with itself.
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
#define CTD_FIXED_PRESET 1
#define CTD_NO_PLAYOUT_KERNEL 1
#define CTD_NO_PRED_KERNEL 1
#define CTD_MCCFR_KERNEL_NAME ctd_k_mccfr_preset
#define CTD_MCCFR_PRED_KERNEL_NAME ctd_k_mccfr_pred_preset_unused
#ifdef CTD_LAYOUT_HEADER   /* placement of the device functions by name order, see ctd_layout_classic.h / tools/layout_search.py */
#include CTD_LAYOUT_HEADER
#endif
#include "ctd_search.cuh"

cudaError_t ctd_mccfr_preset_launch(const CtdMccfrArgs& a, int grid, cudaStream_t stream) {
  ctd_k_mccfr_preset<<<grid, CTD_BLOCK, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t ctd_mccfr_preset_blocks_per_sm(int* per_sm) {
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_mccfr_preset, CTD_BLOCK, 0);
}
