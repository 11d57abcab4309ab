// ctd_preset_playout.cu -- the fused playout kernel specialised for the preset ruleset (see ctd_playout.cuh).  One kernel
// per translation unit on purpose: the kernel is sensitive to what else ptxas lays out next to it (1.02e9 env steps/s alone,
// 9.5e8 with the search kernels in the same unit).
// Device code only: CTD_DEVICE_ONLY keeps this translation unit from emitting host copies of the inline rules functions
// (ctd_kernels.cu owns those); the two units share nothing but the launch wrappers below.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define CTD_DEVICE_ONLY 1
#define CTD_SMALL_CAPS 1   /* real games only: small containers, small working record (ctd_engine.cuh) */
#define CTD_WORK_LOCAL 1   /* every thread plays its own game in its own local memory (ctd_playout.cuh) */
#define CTD_FIXED_PRESET 1
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout_preset
#define CTD_CHOOSE_LINKAGE inline   /* ctd_lane_choose with an external name, as measured: its place in the name order follows from it */
// placement of the device functions by name order (tools/layout_search.py): the functions' own names measured best for this
// kernel (profiles/README.md, round 3); the hook stays for the next search
#ifdef CTD_LAYOUT_HEADER
#include CTD_LAYOUT_HEADER
#endif
#include "ctd_playout.cuh"

cudaError_t ctd_playout_preset_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream) {
  ctd_k_playout_preset<<<grid, CTD_BLOCK, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t ctd_playout_preset_blocks_per_sm(int* per_sm) {
  // the kernel keeps ~200 B of shared memory: what the carveout leaves over is the L1 that caches the threads' records
  cudaError_t c = cudaFuncSetAttribute(ctd_k_playout_preset, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
  if (c != cudaSuccess) return c;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_playout_preset, CTD_BLOCK, 0);
}
