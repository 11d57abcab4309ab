// ctd_playout.cuh -- the fused random-playout kernel (run_utils.py:37-41 for a batch of games), shared by two translation
// units: ctd_kernels.cu instantiates it for any ruleset (ctd_k_playout), ctd_preset_playout.cu with CTD_FIXED_PRESET, where
// every option kind and character outside the preset eight (game/game.py:479-486) is marked unreachable
// (ctd_k_playout_preset: 7.9 k instead of 10.6 k instructions, +5 % env steps/s -- the kernel is instruction-fetch bound).
#pragma once
#include "ctd_engine.cuh"
#include "ctd_warp.cuh"

#ifndef CTD_WARPS_PER_BLOCK
#define CTD_WARPS_PER_BLOCK 8
#define CTD_BLOCK (CTD_WARPS_PER_BLOCK * 32)
#endif
#define CTD_PLAYOUT_MIN_BLOCKS 8
#ifndef CTD_FULL
#define CTD_FULL 0xFFFFFFFFu
#endif
#ifndef CTD_PLAYOUT_KERNEL_NAME
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout
#endif

// move one 256 B record between HBM and the warp's shared staging buffer: 32 lanes x 8 B
__device__ __forceinline__ void ctd_record_load(const ctd_state* g, ctd_state* s, int lane) {
  reinterpret_cast<uint64_t*>(s)[lane] = reinterpret_cast<const uint64_t*>(g)[lane];
  __syncwarp();
}
__device__ __forceinline__ void ctd_record_store(ctd_state* g, const ctd_state* s, int lane) {
  __syncwarp();
  reinterpret_cast<uint64_t*>(g)[lane] = reinterpret_cast<const uint64_t*>(s)[lane];
}

struct CtdPlayoutArgs {
  uint64_t n_games, seed, first_gid;
  int ruleset;
  uint32_t max_steps;
  int8_t* winner;    // [n] or null
  int8_t* points6;   // [n][6] or null
  uint16_t* steps;   // [n] or null
  ctd_playout_stats* stats;
  unsigned long long* counter;
  ctd_state* slots;  // non-null: continue from slots[0..n) instead of dealing new games
};

#ifndef CTD_NO_PLAYOUT_KERNEL
// Outcome statistics are accumulated per block in shared memory (one shared atomic per field and game) and flushed
// to HBM once per block.
__global__ void __launch_bounds__(CTD_BLOCK, CTD_PLAYOUT_MIN_BLOCKS) CTD_PLAYOUT_KERNEL_NAME(CtdPlayoutArgs a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  // the record staging area (game start / end) and the scalar chooser's option buffer (inside a step) are never live together;
  // shared memory is kept small because what is left of the 256 KB is the L1 that holds lane 0's stack
  __shared__ __align__(16) uint64_t scratch_u64[CTD_WARPS_PER_BLOCK][CTD_CHOOSE_BUF];
  static_assert(sizeof(ctd_state) <= CTD_CHOOSE_BUF * 8, "stage aliases the option buffer");
  __shared__ unsigned long long bst[sizeof(ctd_playout_stats) / 8];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  ctd_state* const stage = reinterpret_cast<ctd_state*>(scratch_u64[0]);   // stage[wib] == scratch_u64[wib]
  uint64_t (*choose_buf)[CTD_CHOOSE_BUF] = scratch_u64;
  CtdWork& w = works[wib];
  if (threadIdx.x < sizeof(ctd_playout_stats) / 8) bst[threadIdx.x] = 0;
  __syncthreads();
  ctd_playout_stats* bs = reinterpret_cast<ctd_playout_stats*>(bst);
  for (;;) {
    unsigned long long g = 0;
    if (lane == 0) g = atomicAdd(a.counter, 1ull);
    g = __shfl_sync(CTD_FULL, g, 0);
    if (g >= a.n_games) break;
    if (a.slots != nullptr) {
      ctd_record_load(&a.slots[g], &stage[wib], lane);
      if (lane == 0) {
        ctd_unpack(&stage[wib], w);
        w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
        w.stream = 0;
        w.tape = nullptr; w.tape_len = 0;
      }
      __syncwarp();
    } else {
      if (lane == 0) {
        ctd_chance_init(w, a.seed, a.first_gid + g, 0);
      }
      __syncwarp();
      if (lane == 0) {
        ctd_deal_preset(w, a.ruleset);
        ctd_setup_round<false>(w);
      }
      __syncwarp();
    }
    const uint32_t steps0 = w.steps;
    // ---- the hot loop: run_utils.py:37-41 ----
    for (;;) {
      bool stop = (w.gflags & 2) || w.err || (w.steps - steps0) >= a.max_steps;
      if (stop) break;
      uint64_t d = ctd_warp_choose(w, lane, choose_buf[wib]);
      if (lane == 0) {
        if (d == 0) w.err |= CTD_ERR_REF_RAISE;
        else ctd_apply<false>(w, d);
      }
      __syncwarp();
    }
    if (lane == 0 && !(w.gflags & 2) && !w.err) w.err |= CTD_ERR_MAXSTEPS;
    __syncwarp();
    const uint32_t ns = w.steps - steps0;
    if (lane < 6) {  // per-seat fields: one lane per seat
      const int pts = w.points[lane];
      if (a.points6) a.points6[g * 6 + lane] = (int8_t)(pts > 127 ? 127 : (pts < -128 ? -128 : pts));
      atomicAdd((unsigned long long*)&bs->points_sum[lane], (unsigned long long)(long long)pts);
      atomicAdd((unsigned long long*)&bs->points_sq[lane], (unsigned long long)(pts * pts));
      if (w.winner == lane) atomicAdd((unsigned long long*)&bs->wins[lane], 1ull);
    } else if (lane == 6) {
      if (a.winner) a.winner[g] = w.winner;
      if (a.steps) a.steps[g] = (uint16_t)ns;
      atomicAdd((unsigned long long*)&bs->games, 1ull);
      atomicAdd((unsigned long long*)&bs->steps, (unsigned long long)ns);
      atomicAdd((unsigned long long*)&bs->steps_sq, (unsigned long long)ns * ns);
      if (w.err) atomicAdd((unsigned long long*)&bs->errors, 1ull);
      atomicMax((unsigned long long*)&bs->max_steps, (unsigned long long)ns);
    }
    if (a.slots != nullptr) {
      if (lane == 0) ctd_pack(w, &stage[wib]);
      ctd_record_store(&a.slots[g], &stage[wib], lane);
    }
    __syncwarp();
  }
  __syncthreads();
  if (a.stats != nullptr && threadIdx.x < sizeof(ctd_playout_stats) / 8 && bst[threadIdx.x] != 0) {
    unsigned long long* gs = reinterpret_cast<unsigned long long*>(a.stats);
    const int maxi = offsetof(ctd_playout_stats, max_steps) / 8;
    if ((int)threadIdx.x == maxi) atomicMax(&gs[maxi], bst[threadIdx.x]);
    else atomicAdd(&gs[threadIdx.x], bst[threadIdx.x]);
  }
}
#endif  // CTD_NO_PLAYOUT_KERNEL
