// ctd_classic_playout.cu -- the fused playout kernel specialised for the classic eight (see ctd_playout.cuh,
// ctd_preset_playout.cu): Assassin, Thief, Magician, King, Bishop, Merchant, Architect, Warlord.  Device code only.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define CTD_DEVICE_ONLY 1
#define CTD_SMALL_CAPS 1   /* real games only: small containers, small working record (ctd_engine.cuh) */
#define CTD_WORK_LOCAL 1   /* every thread plays its own game in its own local memory (ctd_playout.cuh) */
#define CTD_FIXED_CLASSIC 1
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout_classic
// where ptxas puts the per-step functions (see the header): +9.7 % on the per-thread kernel (profiles/README.md, round 3)
#ifndef CTD_LAYOUT_HEADER
#define CTD_LAYOUT_HEADER "ctd_layout_classic.h"
#endif
#define CTD_CHOOSE_LINKAGE inline   /* ctd_lane_choose with an external name, as measured: its place in the name order follows from it */
#include CTD_LAYOUT_HEADER
#include "ctd_playout.cuh"

cudaError_t ctd_playout_classic_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream) {
  ctd_k_playout_classic<<<grid, CTD_BLOCK, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t ctd_playout_classic_blocks_per_sm(int* per_sm) {
  // the kernel keeps ~200 B of shared memory: what the carveout leaves over is the L1 that caches the threads' records
  cudaError_t c = cudaFuncSetAttribute(ctd_k_playout_classic, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
  if (c != cudaSuccess) return c;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_playout_classic, CTD_BLOCK, 0);
}
