// ctd_arena.cuh -- the device-resident arena (ctd_arena): compare_to_random.py:8-37 with a player per seat, every game in HBM
// from deal to end.  Between two searches ctd_k_arena_advance plays all random and forced moves of every game; a game whose
// player to move is a search seat with a real choice queues itself for its seat's search group, ctd_k_arena_gather copies the
// queued roots into the engine's root buffers, the ordinary search runs on them and ctd_k_arena_apply plays the decisions.
#pragma once
#include "ctd_playout.cuh"
#include "ctd_mccfr.cuh"

#define CTD_ARENA_STREAM 4u   // Philox counter word 1 of the random seats' choices (0 game chance, 1 trees, 2 root draws, 3 targets)
#define CTD_ARENA_GID_BITS 40 // facade.tree_gid: bits 40.. of a tree id carry the game's search number
#define CTD_REC_NONE 0xFFFFFFFFu  // recording: rec_off of a tree the dataset does not take

// what one game keeps between launches
struct CtdArenaGame {
  ctd_state rec;
  CtdKnow kn[6];          // what every seat has learnt (the root of a search is rec + kn[player] + used_cards)
  uint8_t used_cards[76];
  uint32_t searches;      // searches made so far: the next one runs on tree id tree_gid(gid, searches)
};

struct CtdArenaArgs {
  uint32_t n;
  uint64_t seed, first_gid;
  int ruleset;
  uint32_t max_steps;
  int8_t seat_group[6];   // search group of each seat, -1 for a random seat
  CtdArenaGame* games;
  uint32_t* queue;        // [groups][n] games waiting for a search of that group
  uint32_t* queued;       // [groups]
};

// u uniform over [0, n) for the move at step s of game gid: k = (u * n) >> 32, u = word s & 3 of Philox block (s >> 2, 4, gid).
// Keyed by the step rather than by a running counter, so forced and searched moves consume nothing.
CTD_HD inline uint32_t ctd_arena_pick(uint64_t seed, uint64_t gid, uint32_t s, uint32_t n) {
  uint32_t r[4];
  ctd_philox(s >> 2, CTD_ARENA_STREAM, (uint32_t)gid, (uint32_t)(gid >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
  return (uint32_t)(((uint64_t)r[s & 3] * n) >> 32);
}

// Play game `w` (all six observers' knowledge in kn6) from where it stands: every move of a random seat and every forced move,
// one enumeration per step as in run_utils.py:37-41.  Stops when the game is over (terminal, an error, max_steps) -> -1, or
// when the player to move belongs to a search group and has >= 2 options -> that group; the record then keeps what the
// enumeration did to it (Seer / Scholar), as the facade's get_options_from_state before run_mccfr does.
CTD_HD CTD_NI inline int ctd_arena_advance(CtdWork& w, CtdKnow* kn6, const int8_t* seat_group, uint64_t seed, uint32_t max_steps) {
  const CtdKnowSet ks{kn6, 6};
  const uint64_t gid = (uint64_t)w.g0 | ((uint64_t)w.g1 << 32);
  for (;;) {
    if ((w.gflags & 2) || w.err) return -1;
    if (w.steps >= max_steps) { w.err |= CTD_ERR_MAXSTEPS; return -1; }
    const uint32_t s = w.steps < 65535u ? w.steps : 65535u;   // the record's (saturating) steps field
    const CtdEnumSave sv = ctd_enum_save(w);
    CtdEmit e{nullptr, 0, 0, 0xFFFFFFFFu, 0};
    ctd_enumerate(w, e, kn6);
    if (e.n == 0) { w.err |= CTD_ERR_REF_RAISE; return -1; }
    const int g = w.player < 6 ? seat_group[w.player] : -1;
    if (g >= 0 && e.n >= 2) return g;
    const uint32_t k = e.n == 1 ? 0u : ctd_arena_pick(seed, gid, s, e.n);
    ctd_apply(w, ctd_enum_select(w, kn6, sv, k), ks);
    CTD_LOOP for (int o = 0; o < 6; ++o) w.err |= kn6[o].err;
  }
}

// a search's decision on its game (ctd_mccfr_result.live_option); a failed search ends the game with an error flag
CTD_HD CTD_NI inline void ctd_arena_decide(CtdWork& w, CtdKnow* kn6, uint32_t status, uint64_t live_option) {
  if (status != 0 || live_option == 0) {
    w.err |= (status & CTD_TREE_REF_RAISE) || status == 0 ? CTD_ERR_REF_RAISE : CTD_ERR_OVERFLOW;
    return;
  }
  ctd_apply(w, live_option, CtdKnowSet{kn6, 6});
  CTD_LOOP for (int o = 0; o < 6; ++o) w.err |= kn6[o].err;
}

#ifdef __CUDACC__
__device__ __forceinline__ void ctd_arena_know_copy(CtdKnow* dst, const CtdKnow* src, int lane) {
  for (int i = lane; i < (int)(6 * sizeof(CtdKnow) / 16); i += 32) ((uint4*)dst)[i] = ((const uint4*)src)[i];
}

// run_utils.create_game for every game, knowledge of all six observers tracked from the deal (ctd_k_one op 0)
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_arena_deal(CtdArenaArgs a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK][6];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t i = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (i >= a.n) return;
  CtdWork& w = works[wib];
  CtdKnow* kn = knows[wib];
  CtdArenaGame& G = a.games[i];
  if (lane == 0) {
    ctd_chance_init(w, a.seed, a.first_gid + i, 0);
    ctd_deal_preset(w, a.ruleset, G.used_cards);
    for (int o = 0; o < 6; ++o) ctd_kn_init(kn[o], o);
    ctd_setup_round(w, CtdKnowSet{kn, 6});
    ctd_pack(w, &stage[wib]);
    G.searches = 0;
  }
  __syncwarp();
  ctd_record_store(&G.rec, &stage[wib], lane);
  ctd_arena_know_copy(G.kn, kn, lane);
}

// one warp per game: play on until the game is over or a search seat has to decide (then queue the game for its group)
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_arena_advance(CtdArenaArgs a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK][6];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t i = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (i >= a.n) return;
  CtdWork& w = works[wib];
  CtdKnow* kn = knows[wib];
  CtdArenaGame& G = a.games[i];
  ctd_record_load(&G.rec, &stage[wib], lane);
  if ((stage[wib].gflags & 2) || stage[wib].err) return;   // over: nothing to do (the warp agrees, the staged record is shared)
  ctd_arena_know_copy(kn, G.kn, lane);
  __syncwarp();
  if (lane == 0) {
    ctd_unpack(&stage[wib], w);
    w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
    w.stream = 0; w.tape = nullptr; w.tape_len = 0;
    const int g = ctd_arena_advance(w, kn, a.seat_group, a.seed, a.max_steps);
    ctd_pack(w, &stage[wib]);
    if (g >= 0) a.queue[(size_t)g * a.n + atomicAdd(&a.queued[g], 1u)] = i;
  }
  __syncwarp();
  ctd_record_store(&G.rec, &stage[wib], lane);
  ctd_arena_know_copy(G.kn, kn, lane);
}

// roots [0, count) of a search: queue entries [first, first + count) of `list` -> the engine's root buffers
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_arena_gather(const CtdArenaGame* games, const uint32_t* list, uint32_t count,
                                                                ctd_state* roots, CtdKnow* knows, uint8_t* used_cards, uint64_t* gids) {
  const int lane = threadIdx.x & 31;
  const uint32_t j = blockIdx.x * CTD_WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (j >= count) return;
  const CtdArenaGame& G = games[list[j]];
  reinterpret_cast<uint64_t*>(&roots[j])[lane] = reinterpret_cast<const uint64_t*>(&G.rec)[lane];
  const int p = G.rec.player < 6 ? G.rec.player : 0;
  for (int k = lane; k < (int)(sizeof(CtdKnow) / 16); k += 32) ((uint4*)&knows[j])[k] = ((const uint4*)&G.kn[p])[k];
  for (int k = lane; k < 76; k += 32) used_cards[(size_t)j * 76 + k] = G.used_cards[k];
  if (lane == 0)
    gids[j] = (G.rec.gid & ((1ull << CTD_ARENA_GID_BITS) - 1)) | ((uint64_t)G.searches << CTD_ARENA_GID_BITS);
}

// the decisions of searches [0, count) on the games they came from
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_arena_apply(CtdArenaArgs a, const uint32_t* list, uint32_t count,
                                                               const ctd_mccfr_result* results) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK][6];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t j = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (j >= count) return;
  CtdWork& w = works[wib];
  CtdKnow* kn = knows[wib];
  CtdArenaGame& G = a.games[list[j]];
  ctd_record_load(&G.rec, &stage[wib], lane);
  ctd_arena_know_copy(kn, G.kn, lane);
  __syncwarp();
  if (lane == 0) {
    ctd_unpack(&stage[wib], w);
    w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
    w.stream = 0; w.tape = nullptr; w.tape_len = 0;
    ctd_arena_decide(w, kn, results[j].status, results[j].live_option);
    ctd_pack(w, &stage[wib]);
    G.searches += 1;
  }
  __syncwarp();
  ctd_record_store(&G.rec, &stage[wib], lane);
  ctd_arena_know_copy(G.kn, kn, lane);
}

// per-game outputs and the outcome statistics of the finished games (block totals in shared memory, as in the playout kernel)
__global__ void __launch_bounds__(256) ctd_k_arena_finish(const CtdArenaGame* games, uint32_t n, int8_t* winner, int8_t* points6,
                                                          uint16_t* steps, uint32_t* searches, ctd_playout_stats* stats) {
  __shared__ unsigned long long bst[sizeof(ctd_playout_stats) / 8];
  if (threadIdx.x < sizeof(ctd_playout_stats) / 8) bst[threadIdx.x] = 0;
  __syncthreads();
  ctd_playout_stats* bs = reinterpret_cast<ctd_playout_stats*>(bst);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const ctd_state& r = games[i].rec;
    const int8_t win = r.err ? (int8_t)-1 : r.winner;
    const unsigned long long ns = r.steps;
    winner[i] = win; steps[i] = r.steps; searches[i] = games[i].searches;
    for (int p = 0; p < 6; ++p) {
      const int pts = r.points[p];
      points6[(size_t)i * 6 + p] = r.points[p];
      atomicAdd((unsigned long long*)&bs->points_sum[p], (unsigned long long)(long long)pts);
      atomicAdd((unsigned long long*)&bs->points_sq[p], (unsigned long long)(pts * pts));
    }
    if (win >= 0) atomicAdd((unsigned long long*)&bs->wins[win], 1ull);
    atomicAdd((unsigned long long*)&bs->games, 1ull);
    atomicAdd((unsigned long long*)&bs->steps, ns);
    atomicAdd((unsigned long long*)&bs->steps_sq, ns * ns);
    if (r.err) atomicAdd((unsigned long long*)&bs->errors, 1ull);
    atomicMax((unsigned long long*)&bs->max_steps, ns);
  }
  __syncthreads();
  if (threadIdx.x < sizeof(ctd_playout_stats) / 8 && bst[threadIdx.x] != 0) {
    unsigned long long* gs = reinterpret_cast<unsigned long long*>(stats);
    const int maxi = offsetof(ctd_playout_stats, max_steps) / 8;
    if ((int)threadIdx.x == maxi) atomicMax(&gs[maxi], bst[threadIdx.x]);
    else atomicAdd(&gs[threadIdx.x], bst[threadIdx.x]);
  }
}

// ------------------------------------------------------------------------------------------ recording (ctd_arena_record)
// The dataset's cursors and drop counts live on the device, so a search's trees claim their rows without the host waiting.
struct CtdDatasetCtr {
  unsigned long long n_records, n_slots, dropped_trees, dropped_records;
  unsigned long long call_first;   // n_records when the current ctd_arena_record call began: its records are [call_first, n_records)
};

// Rows for the trees of one search: an exclusive scan of their record and option-slot counts in queue order, behind the dataset's
// cursors.  A tree is kept when all of its records and slots fit.  The scan runs over every tree, kept or not, and the offsets only
// grow, so the kept trees are the leading ones and their rows are consecutive.  rec_off[t] = CTD_REC_NONE for a tree not kept (or
// without records).  One block; tiles of its width in order, so the result does not depend on scheduling.
#define CTD_RESERVE_THREADS 1024
__global__ void __launch_bounds__(CTD_RESERVE_THREADS) ctd_k_record_reserve(uint32_t n, const uint32_t* nrec, const uint32_t* nopt,
                                                                           uint32_t* rec_off, uint32_t* opt_off, CtdDatasetCtr* ctr,
                                                                           uint32_t max_records, uint32_t max_slots) {
  __shared__ unsigned long long wr[32], wo[32];
  __shared__ unsigned long long base_r, base_o, keep_r, keep_o, drop_t, drop_r;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) { base_r = ctr->n_records; base_o = ctr->n_slots; keep_r = keep_o = drop_t = drop_r = 0; }
  __syncthreads();
  for (uint32_t first = 0; first < n; first += CTD_RESERVE_THREADS) {
    const uint32_t t = first + tid;
    const unsigned long long r = t < n ? nrec[t] : 0ull, o = t < n ? nopt[t] : 0ull;
    unsigned long long sr = r, so = o;   // inclusive scan within the warp
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long ur = __shfl_up_sync(0xFFFFFFFFu, sr, d), uo = __shfl_up_sync(0xFFFFFFFFu, so, d);
      if (lane >= d) { sr += ur; so += uo; }
    }
    if (lane == 31) { wr[wid] = sr; wo[wid] = so; }
    __syncthreads();
    if (wid == 0) {   // exclusive scan of the 32 warp totals
      const unsigned long long own_r = wr[lane], own_o = wo[lane];
      unsigned long long xr = own_r, xo = own_o;
      for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long ur = __shfl_up_sync(0xFFFFFFFFu, xr, d), uo = __shfl_up_sync(0xFFFFFFFFu, xo, d);
        if (lane >= d) { xr += ur; xo += uo; }
      }
      wr[lane] = xr - own_r; wo[lane] = xo - own_o;
    }
    __syncthreads();
    const unsigned long long off_r = base_r + wr[wid] + sr - r, off_o = base_o + wo[wid] + so - o;
    const bool keep = r != 0 && off_r + r <= max_records && off_o + o <= max_slots;
    if (t < n) { rec_off[t] = keep ? (uint32_t)off_r : CTD_REC_NONE; opt_off[t] = keep ? (uint32_t)off_o : 0u; }
    if (keep) { atomicAdd(&keep_r, r); atomicAdd(&keep_o, o); }
    else if (r != 0) { atomicAdd(&drop_t, 1ull); atomicAdd(&drop_r, r); }
    __syncthreads();
    if (tid == CTD_RESERVE_THREADS - 1) { base_r = off_r + r; base_o = off_o + o; }   // the tile's total, kept or not
    __syncthreads();
  }
  if (tid == 0) {
    ctr->n_records += keep_r; ctr->n_slots += keep_o;
    ctr->dropped_trees += drop_t; ctr->dropped_records += drop_r;
  }
}

// the outcome of every record of this call: its game's winner (-1 for an errored game) and points, once every game is over
__global__ void __launch_bounds__(256) ctd_k_record_outcome(const CtdArenaGame* games, const ctd_target_meta* meta, ctd_record_origin* origin,
                                                            const CtdDatasetCtr* ctr) {
  const unsigned long long end = ctr->n_records;
  for (unsigned long long r = ctr->call_first + blockIdx.x * blockDim.x + threadIdx.x; r < end; r += (unsigned long long)gridDim.x * blockDim.x) {
    const ctd_state& s = games[meta[r].tree].rec;
    origin[r].winner = s.err ? (int8_t)-1 : s.winner;
    for (int p = 0; p < 6; ++p) origin[r].points[p] = s.points[p];
  }
}

// ctd_dataset_append: n records and n_slots option slots were copied in past the cursors, where no read reaches.  Rebase their
// option_offset by the slot cursor, OR every malformed record into *bad (1 option span, 2 mover, 4 winner), and advance the
// cursors only when none is.  One block, so the commit comes after every check.
#define CTD_APPEND_THREADS 1024
__global__ void __launch_bounds__(CTD_APPEND_THREADS) ctd_k_dataset_append(ctd_target_meta* meta, const ctd_record_origin* origin,
                                                                           CtdDatasetCtr* ctr, uint32_t n, uint32_t n_slots, int* bad) {
  __shared__ int sbad;
  if (threadIdx.x == 0) sbad = 0;
  __syncthreads();
  const unsigned long long base = ctr->n_records, slots = ctr->n_slots;
  int b = 0;
  for (uint32_t i = threadIdx.x; i < n; i += CTD_APPEND_THREADS) {
    ctd_target_meta& m = meta[base + i];
    const ctd_record_origin& o = origin[base + i];
    if (m.n_options == 0 || (unsigned long long)m.option_offset + m.n_options > n_slots) b |= 1;
    if (o.mover > 5) b |= 2;
    if (o.winner < -1 || o.winner > 5) b |= 4;
    m.option_offset += (uint32_t)slots;
  }
  if (b) atomicOr(&sbad, b);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sbad == 0) { ctr->n_records = base + n; ctr->n_slots = slots + n_slots; }
    *bad = sbad;
  }
}
#endif  // __CUDACC__
