// ctd_generic_playout.cu -- the fused playout kernel for any ruleset (see ctd_playout.cuh), alone in its translation unit
// like the specialised one (ctd_preset_playout.cu): device code only.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define CTD_DEVICE_ONLY 1
#define CTD_SMALL_CAPS 1   /* real games only: small containers, small working record (ctd_engine.cuh) */
#define CTD_WORK_LOCAL 1   /* every thread plays its own game in its own local memory (ctd_playout.cuh) */
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout
#include "ctd_playout.cuh"

cudaError_t ctd_playout_generic_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream) {
  ctd_k_playout<<<grid, CTD_BLOCK, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t ctd_playout_generic_blocks_per_sm(int* per_sm) {
  // the kernel keeps ~200 B of shared memory: what the carveout leaves over is the L1 that caches the threads' records
  cudaError_t c = cudaFuncSetAttribute(ctd_k_playout, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
  if (c != cudaSuccess) return c;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_playout, CTD_BLOCK, 0);
}
