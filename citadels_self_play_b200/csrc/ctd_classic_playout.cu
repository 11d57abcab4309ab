// ctd_classic_playout.cu -- the fused playout kernel specialised for the classic eight (see ctd_playout.cuh,
// ctd_preset_playout.cu): Assassin, Thief, Magician, King, Bishop, Merchant, Architect, Warlord.  Device code only.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#define CTD_DEVICE_ONLY 1
#define CTD_SMALL_CAPS 1   /* real games only: small containers, small working record (ctd_engine.cuh) */
#define CTD_FIXED_CLASSIC 1
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout_classic
// where ptxas puts the per-step functions (see the header): worth a few per cent on an instruction-cache-bound kernel
#ifndef CTD_LAYOUT_HEADER
#define CTD_LAYOUT_HEADER "ctd_layout_classic.h"
#endif
#define CTD_CHOOSE_LINKAGE inline   /* external name: takes part in the ordering */
#include CTD_LAYOUT_HEADER
#include "ctd_playout.cuh"

cudaError_t ctd_playout_classic_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream) {
  ctd_k_playout_classic<<<grid, CTD_BLOCK, 0, stream>>>(a);
  return cudaGetLastError();
}
cudaError_t ctd_playout_classic_blocks_per_sm(int* per_sm) {
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ctd_k_playout_classic, CTD_BLOCK, 0);
}
