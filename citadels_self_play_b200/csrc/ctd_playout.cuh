// ctd_playout.cuh -- the fused random-playout kernel (run_utils.py:37-41 for a batch of games), one translation unit per
// ruleset family: ctd_generic_playout.cu (any ruleset, ctd_k_playout), ctd_preset_playout.cu with CTD_FIXED_PRESET and
// ctd_classic_playout.cu with CTD_FIXED_CLASSIC, where every option kind and character outside the ruleset's eight is
// marked unreachable.  ctd_kernels.cu includes the header for the argument block, the record movers and the two passes
// of the choice (for its checker).
//
// One thread owns one game.  Its working record (CtdWork, 1.5 KB) is a local variable: local memory interleaves the
// lanes of a warp word by word, so the same field of the warp's 32 games is one 128-byte line, and one warp instruction
// advances every lane whose game is on that code path (DESIGN.md 3, 4).  A step is the scalar choice -- count the
// options, draw k, select the k-th -- followed by `ctd_apply`.
#pragma once
#include "ctd_engine.cuh"

#ifndef CTD_WARPS_PER_BLOCK
#define CTD_WARPS_PER_BLOCK 8
#define CTD_BLOCK (CTD_WARPS_PER_BLOCK * 32)
#endif
#ifndef CTD_PLAYOUT_MIN_BLOCKS   /* resident blocks per SM the registers are bounded for: 6 x 256 threads (profiles/README.md) */
#define CTD_PLAYOUT_MIN_BLOCKS 6
#endif
#ifndef CTD_PLAYOUT_KERNEL_NAME
#define CTD_PLAYOUT_KERNEL_NAME ctd_k_playout
#endif
#ifndef CTD_CHOOSE_LINKAGE
#define CTD_CHOOSE_LINKAGE static
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

// Enumeration visitor of the playout's choice: counts the options and keeps the `want`-th one, stores nothing.  CtdEmit with
// capacity 0 would do the same with one more compare per option, but as the playout's visitor it measured 17-18 % slower
// (preset 1.333e9 against 1.603e9 env steps/s, classic 1.416e9 against 1.718e9; profiles/README.md, round 3).
struct CtdPick {
  uint32_t n;
  uint32_t want;
  uint64_t got;
  __device__ void one(uint64_t d) {
    if (n == want) got = d;
    ++n;
  }
  __device__ void range(uint64_t base, uint32_t cnt) {   // cnt options that differ only in the ordinal field j
    if (want >= n && want - n < cnt) got = base | ctd_f_j(want - n);
    n += cnt;
  }
};
// the two passes of the choice (ctd_k_choose_check in ctd_kernels.cu tests them against the materialised list for every k)
__device__ __forceinline__ uint32_t ctd_lane_count(CtdWork& w) {
  CtdPick e{0, 0xFFFFFFFFu, 0};
  ctd_enumerate(w, e);
  return e.n;
}
__device__ __forceinline__ uint64_t ctd_lane_select(CtdWork& w, uint32_t k) {
  CtdPick e{0, k, 0};
  ctd_enumerate(w, e);
  return e.got;
}

#ifndef CTD_NO_PLAYOUT_KERNEL
// Agent.get_options, then a uniform draw among them: the counting pass, one draw, and a selecting pass over the same
// enumeration.  Returns the chosen descriptor, 0 when there is no option.
// The Seer's and the Scholar's enumerations are not pure (chance draws, a shrinking seven_drawn_cards): for those two
// states the selecting pass starts from what the counting pass started from, and the game goes on from where the
// counting pass and the draw left it.  Every other state restores nothing, so the draw's Philox block stays cached.
CTD_CHOOSE_LINKAGE __device__ __noinline__ uint64_t ctd_lane_choose(CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  if (w.state == 8 || w.state == 9) {
    CTD_NOT_PRESET(); CTD_NOT_CLASSIC();
    const uint32_t draws0 = w.draws, tape0 = w.tape_pos;
    const uint8_t n7 = w.n_seven;
    uint8_t s7[7];
    for (int i = 0; i < 7; ++i) s7[i] = w.seven[i];
    const uint32_t n = ctd_lane_count(w);
    if (n == 0) return 0;
    const uint32_t k = ctd_randbelow(w, n);
    const uint32_t draws1 = w.draws, tape1 = w.tape_pos;
    w.draws = draws0; w.tape_pos = tape0; w.n_seven = n7;
    for (int i = 0; i < 7; ++i) w.seven[i] = s7[i];
    const uint64_t d = ctd_lane_select(w, k);
    w.draws = draws1; w.tape_pos = tape1;
    return d;
  }
  const uint32_t n = ctd_lane_count(w);
  if (n == 0) return 0;
  return ctd_lane_select(w, ctd_randbelow(w, n));
}

// Every thread pulls game ids from a.counter and plays each game to its end.  The loop is flat -- one env step per trip,
// and a thread whose game has ended records it and starts the next one inside the trip -- so that a warp does not wait
// for its longest game before any lane starts a new one.  Outcome statistics are accumulated per block in shared memory
// (one shared atomic per field and game) and flushed to HBM once per block.
__global__ void __launch_bounds__(CTD_BLOCK, CTD_PLAYOUT_MIN_BLOCKS) CTD_PLAYOUT_KERNEL_NAME(CtdPlayoutArgs a) {
  __shared__ unsigned long long bst[sizeof(ctd_playout_stats) / 8];
  if (threadIdx.x < sizeof(ctd_playout_stats) / 8) bst[threadIdx.x] = 0;
  __syncthreads();
  ctd_playout_stats* bs = reinterpret_cast<ctd_playout_stats*>(bst);
  CtdWork w;
  unsigned long long g = 0;
  uint32_t steps0 = 0;
  bool live = false;
  for (;;) {
    if (!live || (w.gflags & 2) || w.err || (w.steps - steps0) >= a.max_steps) {
      if (live) {  // the game has ended: per-game outputs, block statistics, the record
        if (!(w.gflags & 2) && !w.err) w.err |= CTD_ERR_MAXSTEPS;
        const uint32_t ns = w.steps - steps0;
        for (int q = 0; q < 6; ++q) {
          const int pts = w.points[q];
          if (a.points6) a.points6[g * 6 + q] = (int8_t)(pts > 127 ? 127 : (pts < -128 ? -128 : pts));
          atomicAdd((unsigned long long*)&bs->points_sum[q], (unsigned long long)(long long)pts);
          atomicAdd((unsigned long long*)&bs->points_sq[q], (unsigned long long)(pts * pts));
        }
        if (w.winner >= 0 && w.winner < 6) atomicAdd((unsigned long long*)&bs->wins[w.winner], 1ull);
        if (a.winner) a.winner[g] = w.winner;
        if (a.steps) a.steps[g] = (uint16_t)ns;
        atomicAdd((unsigned long long*)&bs->games, 1ull);
        atomicAdd((unsigned long long*)&bs->steps, (unsigned long long)ns);
        atomicAdd((unsigned long long*)&bs->steps_sq, (unsigned long long)ns * ns);
        if (w.err) atomicAdd((unsigned long long*)&bs->errors, 1ull);
        atomicMax((unsigned long long*)&bs->max_steps, (unsigned long long)ns);
        if (a.slots != nullptr) ctd_pack(w, &a.slots[g]);
      }
      g = atomicAdd(a.counter, 1ull);
      if (g >= a.n_games) break;
      if (a.slots != nullptr) {
        ctd_unpack(&a.slots[g], w);
        w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
        w.stream = 0;
        w.tape = nullptr; w.tape_len = 0;
      } else {
        ctd_chance_init(w, a.seed, a.first_gid + g, 0);
        ctd_deal_preset(w, a.ruleset);
        ctd_setup_round<false>(w);
      }
      steps0 = w.steps;
      live = true;
      continue;  // a continued record may already have ended
    }
    // ---- the hot loop: run_utils.py:37-41 ----
    const uint64_t d = ctd_lane_choose(w);
    if (d == 0) w.err |= CTD_ERR_REF_RAISE;
    else ctd_apply<false>(w, d);
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
