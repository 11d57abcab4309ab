// ctd_kernels.cu -- sm_100a kernels and the C ABI (include/citadels_b200.h) of the Citadels rollout engine.
//
// Layout of the data path:
//   HBM     ctd_state slots[capacity]          256 B records, 2 x 128 B lines each, one warp moves one
//                                              record as 32 x 8 B (coalesced)
//   smem    CtdWork per warp (1.3 KB)          the game of a step-wise / search / arena kernel
//   local   CtdWork per thread (1.5 KB)        the game of a fused playout for its whole life (~420 steps)
// One warp owns one game, except in the fused playout, where one thread owns one game (ctd_playout.cuh).  The playout
// kernel is persistent: threads pull game ids from a global counter so that the 244..632-step spread of game lengths
// does not leave SMs idle at the tail.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <initializer_list>
#include <memory>
#include <new>
#include <stddef.h>

// the playout and search kernels are compiled one per translation unit (ctd_generic_*.cu, ctd_preset_*.cu): out-of-line
// device functions are compiled once per unit under the tightest register bound of their callers
#define CTD_NO_PLAYOUT_KERNEL 1
#define CTD_NO_TRAIN_KERNEL 1
#define CTD_NO_PRED_KERNEL 1
#include "ctd_engine.cuh"
#include "ctd_playout.cuh"
#include "ctd_mccfr.cuh"
#include "ctd_search.cuh"
#include "ctd_arena.cuh"
#include "ctd_value_tc.cuh"
#include "ctd_train.cuh"


// ------------------------------------------------------------------------------------------ device helpers
// (ctd_record_load / ctd_record_store live in ctd_playout.cuh)

struct CtdTapes {
  const uint8_t* tape;
  const uint32_t* off;
  uint32_t n;
};
__device__ __forceinline__ void ctd_attach_tape(CtdWork& w, const CtdTapes& t, uint32_t slot) {
  if (t.tape != nullptr && slot < t.n) {
    w.tape = t.tape + t.off[slot];
    w.tape_len = t.off[slot + 1] - t.off[slot];
  } else {
    w.tape = nullptr;
    w.tape_len = 0;
  }
}

// ------------------------------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_reset(ctd_state* slots, uint32_t n, uint64_t seed, uint64_t first_gid,
                                                         int ruleset, CtdTapes tapes) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= n) return;
  CtdWork& w = works[wib];
  if (lane == 0) {
    ctd_chance_init(w, seed, first_gid + slot, 0);
    ctd_attach_tape(w, tapes, slot);
    ctd_deal_preset(w, ruleset);
    ctd_setup_round(w);
    ctd_pack(w, &stage[wib]);
  }
  ctd_record_store(&slots[slot], &stage[wib], lane);
}

// Enumeration is read-only except in two states of the deluxe characters: the Seer's give-back list is built with
// fresh shuffles (chance is consumed) and the Scholar's list shrinks game.seven_drawn_cards.  Those records are written to
// `shadow`; the host commits the shadow only when every list of the batch fitted (a caller that has to retry with a larger
// stride must find the slots untouched).
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_enumerate(const ctd_state* slots, uint32_t n, ctd_option* opts,
                                                             uint32_t* counts, uint32_t stride, uint8_t* errs, uint64_t seed,
                                                             CtdTapes tapes, ctd_state* shadow, uint32_t* any_dirty) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= n) return;
  CtdWork& w = works[wib];
  ctd_record_load(&slots[slot], &stage[wib], lane);
  if (lane == 0) {
    ctd_unpack(&stage[wib], w);
    w.k0 = (uint32_t)seed; w.k1 = (uint32_t)(seed >> 32);
    w.stream = 0;
    ctd_attach_tape(w, tapes, slot);
    const bool dirty = (w.state == 8 || w.state == 9) && !(w.gflags & 2);
    CtdEmit e{opts + (size_t)slot * stride, stride, 0, 0xFFFFFFFFu, 0};
    ctd_enumerate(w, e);
    counts[slot] = e.n;
    errs[slot] = w.err;
    if (dirty) { ctd_pack(w, &stage[wib]); atomicOr(any_dirty, 1u); }
  }
  __syncwarp();
  ctd_record_store(&shadow[slot], &stage[wib], lane);
}

__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_step(ctd_state* slots, uint32_t n, const ctd_option* chosen,
                                                        int8_t* winner, uint64_t seed, CtdTapes tapes) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= n) return;
  const ctd_option d = chosen[slot];
  if (d == 0) {  // role_pick by seat 0 always carries a rank field, so 0 is never a real option
    if (lane == 0) winner[slot] = -1;
    return;
  }
  CtdWork& w = works[wib];
  ctd_record_load(&slots[slot], &stage[wib], lane);
  if (lane == 0) {
    ctd_unpack(&stage[wib], w);
    w.k0 = (uint32_t)seed; w.k1 = (uint32_t)(seed >> 32);
    ctd_attach_tape(w, tapes, slot);
    bool won = ctd_apply(w, d);
    winner[slot] = won ? w.winner : (int8_t)-1;
    ctd_pack(w, &stage[wib]);
  }
  ctd_record_store(&slots[slot], &stage[wib], lane);
}

// Checker for the fused playout's choice (ctd_playout.cuh): for every slot, the counting pass (ctd_lane_count) and the
// selecting pass (ctd_lane_select) for every k must equal the scalar enumerator's materialised list.
// mismatches[slot] = number of differing entries (+1e6 if the counts differ).  Lane 0 of each warp checks its slot.
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_choose_check(const ctd_state* slots, uint32_t n, uint32_t* mismatches,
                                                                uint64_t* scratch_opts, uint32_t cap) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= n) return;
  CtdWork& w = works[wib];
  ctd_record_load(&slots[slot], &stage[wib], lane);
  if (lane != 0) return;
  ctd_unpack(&stage[wib], w);
  uint64_t* ref = scratch_opts + (size_t)slot * cap;
  CtdEmit e{ref, cap, 0, 0xFFFFFFFFu, 0};
  ctd_enumerate(w, e);
  const uint32_t nref = e.n;
  uint32_t bad = 0;
  // impure enumerations (the Seer's and the Scholar's) change the record: ctd_lane_choose restores it around its passes
  if (nref != 0 && w.state != 8 && w.state != 9) {
    if (ctd_lane_count(w) != nref) {
      bad = 1000000;
    } else {
      // discard_and_draw ordinals are reproduced too, so compare everything
      for (uint32_t k = 0; k < nref && k < cap; ++k)
        if (ctd_lane_select(w, k) != ref[k]) ++bad;
    }
  }
  mismatches[slot] = bad;
}

// the same kernel specialised for the preset eight, compiled in ctd_preset_playout.cu
cudaError_t ctd_playout_generic_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream);
cudaError_t ctd_playout_generic_blocks_per_sm(int* per_sm);
cudaError_t ctd_playout_classic_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream);
cudaError_t ctd_playout_classic_blocks_per_sm(int* per_sm);
cudaError_t ctd_playout_preset_launch(const CtdPlayoutArgs& a, int grid, cudaStream_t stream);
cudaError_t ctd_playout_preset_blocks_per_sm(int* per_sm);

// ------------------------------------------------------------------------------------------ CFR roots + MCCFR
// run_utils.create_a_close_to_finished_game / create_a_random_game (run_utils.py:29-72): play a preset game to
// terminal, step back `u` decisions (u uniform in [back_lo, back_hi], drawn from Philox stream word 2), then move
// forward until the player to move has a real choice.  The game is replayed from its (seed, gid) with the
// knowledge of all six observers tracked, so the root carries what its player to move has learnt so far.
struct CtdRootArgs {
  uint32_t n;
  uint64_t seed, first_gid;
  int ruleset;
  uint32_t back_lo, back_hi;
  int flavour;          // CTD_ROOTS_CLOSE_TO_FINISHED / CTD_ROOTS_RANDOM_GAME
  ctd_state* roots;
  CtdKnow* knows;
  uint8_t* used_cards;  // [n][76]
  uint64_t* gids;
  uint32_t* root_step;  // [n] index of the root in the game's step sequence
};

__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_make_roots(CtdRootArgs a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK][6];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= a.n) return;
  CtdWork& w = works[wib];
  CtdKnow* kn = knows[wib];
  if (lane == 0) {
    const uint64_t gid = a.first_gid + slot;
    uint32_t step = 0;
    const int viewer = ctd_make_root(w, kn, a.seed, gid, a.ruleset, a.back_lo, a.back_hi, a.flavour,
                                     a.used_cards + (size_t)slot * 76, &step);
    a.root_step[slot] = step;
    a.gids[slot] = gid;
    a.knows[slot] = kn[viewer];
    ctd_pack(w, &stage[wib]);
  }
  ctd_record_store(&a.roots[slot], &stage[wib], lane);
}

// (CtdMccfrArgs, ctd_tree_at, ctd_write_result, ctd_k_mccfr and ctd_k_mccfr_pred live in ctd_search.cuh)
// the same kernels specialised for the preset eight, compiled in ctd_preset_search.cu
cudaError_t ctd_mccfr_generic_launch(const CtdMccfrArgs& a, int grid, cudaStream_t stream);
cudaError_t ctd_mccfr_generic_blocks_per_sm(int* per_sm);
cudaError_t ctd_mccfr_pred_generic_launch(const CtdPredArgs& p, int grid, cudaStream_t stream);
cudaError_t ctd_mccfr_pred_generic_blocks_per_sm(int* per_sm, int fused);
cudaError_t ctd_mccfr_preset_launch(const CtdMccfrArgs& a, int grid, cudaStream_t stream);
cudaError_t ctd_mccfr_preset_blocks_per_sm(int* per_sm);
cudaError_t ctd_mccfr_pred_preset_launch(const CtdPredArgs& p, int grid, cudaStream_t stream);
cudaError_t ctd_mccfr_pred_preset_blocks_per_sm(int* per_sm, int fused);

// ------------------------------------------------------------------------------------------ training targets
// CFRNode.get_all_targets / build_train_targets (algorithms/deep_mccfr.py:258-274, :321-345): depth-first pre-order
// over the tree, one record per node that has children and node_value.sum() >= threshold.  Role-pick nodes are
// encoded from the viewpoint of a random seat i = randint(0, 5) (Philox stream 3 of the tree, one draw per emitted
// role-pick node) and export row i of their regret matrix.
struct CtdTargetArgs {
  uint32_t n_roots;
  CtdTreeHdr* hdrs;
  uint64_t seed;
  double threshold;
  int fill;                 // 0: count only; 1: write records
  uint32_t* n_targets;      // [n_roots]
  uint32_t* n_options;      // [n_roots] sum of K over the tree's targets
  const uint32_t* rec_off;  // [n_roots] (fill) first record of the tree
  const uint32_t* opt_off;  // [n_roots] (fill) first option slot of the tree
  float* feat;              // [records][CTD_FEATURES_PAD]
  ctd_target_meta* meta;    // [records]
  ctd_option* options;      // [option slots]
  double* regrets;          // [option slots]
  // recording (ctd_arena_record) only: tree t is the search of game list[t]
  const CtdArenaGame* games;
  const uint32_t* list;
  uint32_t seat_mask;       // trees whose mover (the searching seat) is not in the mask have no records
  int root_only;            // CTD_RECORD_ROOT: node 0 alone, threshold not applied
  ctd_record_origin* origin;   // [records]
};

// Rec: the recording form -- trees of unrecorded seats count nothing, rec_off[t] == CTD_REC_NONE skips a tree, meta.tree is the
// game index and every record also gets its origin.  Without Rec this is ctd_mccfr_targets' walk.
template <bool Rec>
__device__ __forceinline__ void ctd_targets_tree(const CtdTargetArgs& a, uint32_t t, CtdWork* work, CtdKnow* know, ctd_state* stage) {
  CtdTree T;
  T.w = work; T.kn = know; T.stage = stage; T.vnet = nullptr; T.act = nullptr;
  ctd_tree_attach(T, &a.hdrs[t], CtdArena{a.hdrs[t].arena, nullptr, 0});
  const CtdTreeHdr& h = *T.hdr;
  uint32_t nrec = 0, nopt = 0, rp_draws = 0;
  const CtdArenaGame* G = Rec ? &a.games[a.list[t]] : nullptr;
  bool take = true;
  if (Rec) take = ((a.seat_mask >> G->rec.player) & 1) && (!a.fill || a.rec_off[t] != CTD_REC_NONE);
  // trees that stopped early (arena exhausted, engine limit, the reference raises) are not training data
  if (take && h.n_nodes != 0 && h.status == CTD_TREE_OK) {
    // Where node_value counts backpropagations (cfr_train, and cfr_pred in training mode: every backprop adds a reward that sums
    // to one to each node on its path) a child never has more than its parent, so nothing below a node under the threshold
    // qualifies and the walk does not go there: a 2000-iteration tree has ~3800 nodes and a handful over 200 backprops.
    const bool prune = h.training || !h.has_model;
    int cur = 0;
    for (;;) {
      const CtdNode& n = ctd_node(T, cur);
      const uint32_t K = n.n_children;
      double vs = 0.0;
      for (int i = 0; i < 6; ++i) vs += n.V[i];
      if (K != 0 && (vs >= a.threshold || (Rec && a.root_only))) {
        const bool rp = n.flags & CTD_NF_ROLE_PICK;
        uint32_t seat = n.player;
        if (rp) {
          uint32_t r[4];
          ctd_philox(rp_draws >> 2, 3u, (uint32_t)h.gid, (uint32_t)(h.gid >> 32), (uint32_t)a.seed, (uint32_t)(a.seed >> 32), r);
          seat = (uint32_t)(((uint64_t)r[rp_draws & 3] * 6) >> 32);
          ++rp_draws;
        }
        if (a.fill) {
          const uint32_t rec = a.rec_off[t] + nrec, ko = a.opt_off[t] + nopt;
          ctd_node_load(T, n);
          ctd_encode_game(*T.w, *T.kn, (int)seat, a.feat + (size_t)rec * CTD_FEATURES_PAD);
          ctd_target_meta& m = a.meta[rec];
          m.tree = Rec ? a.list[t] : t; m.node = (uint32_t)cur; m.n_options = K; m.option_offset = ko; m.seat = seat; m.role_pick = rp ? 1 : 0;
          for (int i = 0; i < 6; ++i) m.node_value[i] = n.V[i];
          if (Rec) {
            ctd_record_origin& o = a.origin[rec];
            o.gid = G->rec.gid; o.search = G->searches; o.step = G->rec.steps; o.mover = G->rec.player; o.winner = -1;
            for (int i = 0; i < 6; ++i) o.points[i] = 0;
            o.pad[0] = o.pad[1] = 0;
          }
          const double* R = ctd_R(T, n) + (rp ? seat * 10 : 0);
          const CtdChild* kids = ctd_kids(T, n);
          double rs = 0.0;
          for (uint32_t i = 0; i < K; ++i) rs += R[i];
          for (uint32_t i = 0; i < K; ++i) {
            a.options[ko + i] = kids[i].desc;
            a.regrets[ko + i] = rs == 0.0 ? 1.0 : R[i];   // all-zero regrets are exported as ones (:333-334, :342-343)
          }
        }
        ++nrec;
        nopt += K;
      }
      if (Rec && a.root_only) break;
      // pre-order successor: first child, else next sibling of the nearest ancestor that has one
      if (K != 0 && !(prune && vs < a.threshold)) { cur = (int)ctd_kids(T, n)[0].node; continue; }
      int c = cur;
      for (;;) {
        const int par = ctd_node(T, c).parent;
        if (par < 0) { c = -1; break; }
        const CtdNode& pn = ctd_node(T, par);
        const CtdChild* pk = ctd_kids(T, pn);
        uint32_t i = 0;
        while (i < pn.n_children && (int)pk[i].node != c) ++i;
        if (i + 1 < pn.n_children) { c = (int)pk[i + 1].node; break; }
        c = par;
      }
      if (c < 0) break;
      cur = c;
    }
  }
  if (!a.fill) { a.n_targets[t] = nrec; a.n_options[t] = nopt; }
}

template <bool Rec>
__device__ __forceinline__ void ctd_targets_warp(const CtdTargetArgs& a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK];
  __shared__ __align__(16) ctd_state tstage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t t = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (t >= a.n_roots || lane != 0) return;
  ctd_targets_tree<Rec>(a, t, &works[wib], &knows[wib], &tstage[wib]);
}
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_targets(CtdTargetArgs a) { ctd_targets_warp<false>(a); }
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_record_targets(CtdTargetArgs a) { ctd_targets_warp<true>(a); }

// ------------------------------------------------------------------------------------------ single-game entry points
// The facade's Game object owns its record and the knowledge of all six observers on the host; these kernels run
// one warp on device copies of them (op 0: new game, 1: enumerate, 2: step).
struct CtdOneArgs {
  int op;
  uint64_t seed, gid;
  int ruleset;
  ctd_state* state;
  CtdKnow* know6;        // may be null
  uint8_t* used_cards;   // op 0
  ctd_option* opts;      // op 1
  uint32_t cap;
  uint32_t* count;
  ctd_option chosen;     // op 2
  int8_t* winner;
  int viewer, role_sample;  // op 3
};
__global__ void __launch_bounds__(32) ctd_k_one(CtdOneArgs a) {
  __shared__ CtdWork w;
  __shared__ CtdKnow kn[6];
  __shared__ ctd_state stage;
  __shared__ __align__(16) uint8_t sscratch[CTD_TREE_SCRATCH];
  const int lane = threadIdx.x;
  if (a.op != 0) ctd_record_load(a.state, &stage, lane);
  if (a.know6 != nullptr && a.op != 0)
    for (int i = lane; i < (int)(6 * sizeof(CtdKnow) / 4); i += 32) ((uint32_t*)kn)[i] = ((const uint32_t*)a.know6)[i];
  __syncwarp();
  if (lane == 0) {
    CtdKnowSet ks{a.know6 ? kn : nullptr, a.know6 ? 6 : 0};
    if (a.op == 0) {
      ctd_chance_init(w, a.seed, a.gid, 0);
      ctd_deal_preset(w, a.ruleset, a.used_cards);
      for (int o = 0; o < 6; ++o) ctd_kn_init(kn[o], o);
      ctd_setup_round(w, ks);
      ctd_pack(w, &stage);
    } else if (a.op == 1) {
      ctd_unpack(&stage, w);
      w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
      w.stream = 0; w.tape = nullptr; w.tape_len = 0;
      CtdEmit e{a.opts, a.cap, 0, 0xFFFFFFFFu, 0};
      ctd_enumerate(w, e, a.know6 ? &kn[0] : nullptr);
      *a.count = e.n;
      if (e.n <= a.cap) ctd_pack(w, &stage);   // Seer / Scholar enumerations change the record (a list that does not fit is asked for again)
    } else if (a.op == 3) {   // Game.sample_private_information (game/game.py:215-242) from seat a.viewer's knowledge
      ctd_unpack(&stage, w);
      w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
      w.stream = 0; w.tape = nullptr; w.tape_len = 0;
      ctd_stage_used(sscratch + 256, a.used_cards);
      ctd_sample_private(w, kn[a.viewer], sscratch + 256, a.role_sample != 0, sscratch);
      w.err |= kn[a.viewer].err;
      ctd_pack(w, &stage);
    } else {
      ctd_unpack(&stage, w);
      w.k0 = (uint32_t)a.seed; w.k1 = (uint32_t)(a.seed >> 32);
      w.stream = 0; w.tape = nullptr; w.tape_len = 0;
      bool won = ctd_apply(w, a.chosen, ks);
      *a.winner = won ? w.winner : (int8_t)-1;
      for (int o = 0; o < ks.n; ++o) w.err |= kn[o].err;
      ctd_pack(w, &stage);
    }
  }
  __syncwarp();
  ctd_record_store(a.state, &stage, lane);
  if (a.op != 1) {
    if (a.know6 != nullptr)
      for (int i = lane; i < (int)(6 * sizeof(CtdKnow) / 4); i += 32) ((uint32_t*)a.know6)[i] = ((const uint32_t*)kn)[i];
  }
}

// ------------------------------------------------------------------------------------------ deep MCCFR
// export pass: every tree as a compact block (ctd_tree_export), one warp per tree, only when trees are copied out
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_export_trees(CtdTreeHdr* hdrs, uint32_t first, uint32_t n, const uint64_t* out_off,
                                                                uint8_t* out) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ __align__(16) ctd_state tstage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t t = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (t >= n || lane != 0) return;
  CtdTree T;
  T.w = &works[wib]; T.stage = &tstage[wib];
  ctd_tree_attach(T, &hdrs[first + t], CtdArena{hdrs[first + t].arena, nullptr, 0});
  ctd_tree_export(T, out + out_off[t]);
}

// root arrays of one tree beyond what a result record holds (ctd_mccfr_root_children)
__global__ void ctd_k_root_children(CtdTreeHdr* hdrs, uint32_t tree, uint32_t first, uint32_t count, ctd_option* options, double* R,
                                    double* S, double* C) {
  CtdTree T;
  ctd_tree_attach(T, &hdrs[tree], CtdArena{hdrs[tree].arena, nullptr, 0});
  if (T.hdr->n_nodes == 0) return;
  const CtdNode& n = ctd_node(T, 0);
  const CtdChild* kids = ctd_kids(T, n);
  const double *r = ctd_R(T, n), *s = ctd_S(T, n), *c = ctd_C(T, n);
  const bool rp = n.flags & CTD_NF_ROLE_PICK;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const uint32_t k = first + i;
    options[i] = k < n.n_children ? kids[k].desc : 0;
    if (!rp) { R[i] = k < n.n_children ? r[k] : 0.0; S[i] = k < n.n_children ? s[k] : 0.0; C[i] = k < n.n_children ? c[k] : 0.0; }
  }
}

// ValueOnlyNN.forward in eval mode (algorithms/models.py:17-23) with BatchNorm folded into fc1/fc2, then
// model_reward_weights * square_and_normalize (train_utils.py:143-145).  fp32 CUDA-core version: a tile of 16 rows per
// CTA, activations k-major in shared memory, weights transposed [in][out] so every warp reads a contiguous row.
struct CtdValueModel {
  const float *w1t, *b1, *w2t, *b2, *w3t, *b3, *w4t, *b4;  // w1t [448][512], w2t [512][256], w3t [256][128], w4t [128][6]
};
#define CTD_MLP_ROWS 16
__global__ void __launch_bounds__(256) ctd_k_value_mlp(const float* __restrict__ feat, const uint8_t* __restrict__ pending,
                                                       uint32_t n, CtdValueModel m, float* __restrict__ pred, float weight) {
  extern __shared__ float sm[];
  float* X = sm;                                   // [448][16]
  float* H1 = X + CTD_FEATURES_PAD * CTD_MLP_ROWS;  // [512][16]
  float* H2 = H1 + 512 * CTD_MLP_ROWS;             // [256][16]
  float* H3 = H2 + 256 * CTD_MLP_ROWS;             // [128][16]
  __shared__ int any;
  const int t = threadIdx.x;
  const uint32_t row0 = blockIdx.x * CTD_MLP_ROWS;
  if (t == 0) any = 0;
  __syncthreads();
  if (t < CTD_MLP_ROWS && row0 + t < n && (pending == nullptr || pending[row0 + t])) any = 1;
  __syncthreads();
  if (!any) return;
  for (int i = t; i < CTD_FEATURES_PAD * CTD_MLP_ROWS; i += 256) {
    int r = i / CTD_FEATURES_PAD, k = i % CTD_FEATURES_PAD;
    X[k * CTD_MLP_ROWS + r] = row0 + r < n ? feat[(size_t)(row0 + r) * CTD_FEATURES_PAD + k] : 0.f;
  }
  __syncthreads();
  {  // fc1 + bn1 + relu: 512 outputs, thread t -> outputs t and t+256
    float a0[CTD_MLP_ROWS], a1[CTD_MLP_ROWS];
#pragma unroll
    for (int r = 0; r < CTD_MLP_ROWS; ++r) { a0[r] = 0.f; a1[r] = 0.f; }
    for (int k = 0; k < CTD_FEATURES_PAD; ++k) {
      const float w0 = m.w1t[k * 512 + t], w1 = m.w1t[k * 512 + t + 256];
      const float4* x4 = reinterpret_cast<const float4*>(X + k * CTD_MLP_ROWS);
#pragma unroll
      for (int q = 0; q < CTD_MLP_ROWS / 4; ++q) {
        float4 x = x4[q];
        a0[4 * q + 0] = fmaf(w0, x.x, a0[4 * q + 0]); a0[4 * q + 1] = fmaf(w0, x.y, a0[4 * q + 1]);
        a0[4 * q + 2] = fmaf(w0, x.z, a0[4 * q + 2]); a0[4 * q + 3] = fmaf(w0, x.w, a0[4 * q + 3]);
        a1[4 * q + 0] = fmaf(w1, x.x, a1[4 * q + 0]); a1[4 * q + 1] = fmaf(w1, x.y, a1[4 * q + 1]);
        a1[4 * q + 2] = fmaf(w1, x.z, a1[4 * q + 2]); a1[4 * q + 3] = fmaf(w1, x.w, a1[4 * q + 3]);
      }
    }
    const float c0 = m.b1[t], c1 = m.b1[t + 256];
#pragma unroll
    for (int r = 0; r < CTD_MLP_ROWS; ++r) {
      H1[t * CTD_MLP_ROWS + r] = fmaxf(a0[r] + c0, 0.f);
      H1[(t + 256) * CTD_MLP_ROWS + r] = fmaxf(a1[r] + c1, 0.f);
    }
  }
  __syncthreads();
  {  // fc2 + bn2 + relu: 256 outputs
    float a0[CTD_MLP_ROWS];
#pragma unroll
    for (int r = 0; r < CTD_MLP_ROWS; ++r) a0[r] = 0.f;
    for (int k = 0; k < 512; ++k) {
      const float w0 = m.w2t[k * 256 + t];
      const float4* x4 = reinterpret_cast<const float4*>(H1 + k * CTD_MLP_ROWS);
#pragma unroll
      for (int q = 0; q < CTD_MLP_ROWS / 4; ++q) {
        float4 x = x4[q];
        a0[4 * q + 0] = fmaf(w0, x.x, a0[4 * q + 0]); a0[4 * q + 1] = fmaf(w0, x.y, a0[4 * q + 1]);
        a0[4 * q + 2] = fmaf(w0, x.z, a0[4 * q + 2]); a0[4 * q + 3] = fmaf(w0, x.w, a0[4 * q + 3]);
      }
    }
    const float c0 = m.b2[t];
#pragma unroll
    for (int r = 0; r < CTD_MLP_ROWS; ++r) H2[t * CTD_MLP_ROWS + r] = fmaxf(a0[r] + c0, 0.f);
  }
  __syncthreads();
  {  // fc3 + relu: 128 outputs x 16 rows, thread t -> output t & 127, rows (t >> 7) * 8 ..
    const int o = t & 127, rb = (t >> 7) * 8;
    float a0[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) a0[r] = 0.f;
    for (int k = 0; k < 256; ++k) {
      const float w0 = m.w3t[k * 128 + o];
      const float4* x4 = reinterpret_cast<const float4*>(H2 + k * CTD_MLP_ROWS + rb);
      float4 x = x4[0], y = x4[1];
      a0[0] = fmaf(w0, x.x, a0[0]); a0[1] = fmaf(w0, x.y, a0[1]); a0[2] = fmaf(w0, x.z, a0[2]); a0[3] = fmaf(w0, x.w, a0[3]);
      a0[4] = fmaf(w0, y.x, a0[4]); a0[5] = fmaf(w0, y.y, a0[5]); a0[6] = fmaf(w0, y.z, a0[6]); a0[7] = fmaf(w0, y.w, a0[7]);
    }
    const float c0 = m.b3[o];
#pragma unroll
    for (int r = 0; r < 8; ++r) H3[o * CTD_MLP_ROWS + rb + r] = fmaxf(a0[r] + c0, 0.f);
  }
  __syncthreads();
  // fc4: 6 outputs x 16 rows; then weight * y^2 / sum(y^2)
  float* Y = X;  // reuse: [16][8]
  if (t < 6 * CTD_MLP_ROWS) {
    const int o = t % 6, r = t / 6;
    float acc = 0.f;
    for (int k = 0; k < 128; ++k) acc = fmaf(m.w4t[k * 6 + o], H3[k * CTD_MLP_ROWS + r], acc);
    Y[r * 8 + o] = acc + m.b4[o];
  }
  __syncthreads();
  if (t < CTD_MLP_ROWS && row0 + t < n && (pending == nullptr || pending[row0 + t])) {
    float s = 0.f, y[6];
#pragma unroll
    for (int o = 0; o < 6; ++o) { y[o] = Y[t * 8 + o]; y[o] *= y[o]; s += y[o]; }
#pragma unroll
    for (int o = 0; o < 6; ++o) pred[(size_t)(row0 + t) * 8 + o] = weight * (y[o] / s);
  }
}
#define CTD_MLP_SMEM ((CTD_FEATURES_PAD + 512 + 256 + 128) * CTD_MLP_ROWS * sizeof(float))

// features of the games in slots [0,n) as their player to move sees them (role-pick states: player 5)
__global__ void __launch_bounds__(CTD_BLOCK) ctd_k_encode(const ctd_state* slots, const CtdKnow* knows, uint32_t n, float* feat,
                                                          int cfr_role_pick) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ ctd_state stage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const uint32_t slot = blockIdx.x * CTD_WARPS_PER_BLOCK + wib;
  if (slot >= n) return;
  ctd_record_load(&slots[slot], &stage[wib], lane);
  if (lane == 0) {
    CtdWork& w = works[wib];
    ctd_unpack(&stage[wib], w);
    ctd_encode_game(w, knows[slot], (w.state == 0 && cfr_role_pick) ? 5 : w.player, feat + (size_t)slot * CTD_FEATURES_PAD);
  }
}

// ------------------------------------------------------------------------------------------ host side / C ABI
// Device memory (page-locked host memory with Pinned) owned by one holder and freed with it.  grow() reallocates only when
// asked for more than it holds, freeing the old block first; the size is recorded once the new block exists.
template <class T, bool Pinned = false>
struct CtdBuf {
  T* p = nullptr;
  size_t bytes = 0;
  CtdBuf() = default;
  CtdBuf(const CtdBuf&) = delete;
  CtdBuf& operator=(const CtdBuf&) = delete;
  CtdBuf(CtdBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  CtdBuf& operator=(CtdBuf&& o) noexcept {
    if (this != &o) { reset(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; }
    return *this;
  }
  ~CtdBuf() { reset(); }
  operator T*() const { return p; }
  T* get() const { return p; }
  cudaError_t reset() {
    const cudaError_t c = p == nullptr ? cudaSuccess : Pinned ? cudaFreeHost(p) : cudaFree(p);
    p = nullptr; bytes = 0;
    return c;
  }
  cudaError_t grow(size_t n) {
    if (n <= bytes) return cudaSuccess;
    cudaError_t c = reset();
    if (c == cudaSuccess) c = Pinned ? cudaHostAlloc((void**)&p, n, cudaHostAllocDefault) : cudaMalloc((void**)&p, n);
    if (c == cudaSuccess) bytes = n;
    else p = nullptr;
    return c;
  }
};

// value-network training (algorithms/train.py:13-86, train_node_value_only) on the device; kernels in ctd_train.cuh.  Every
// buffer starts zeroed (ctd_train_begin).
struct CtdTrainer {
  uint32_t n_train, n_val, batch, bp;   // bp: batch rounded up to a multiple of 32 (the K extent of the weight-gradient products)
  uint32_t step;                        // optimiser steps taken (Adam bias correction, dropout mask counter)
  CtdBuf<float> feat_tr, feat_va;
  CtdBuf<double> val_tr, val_va;
  CtdBuf<uint32_t> perm;
  CtdBuf<float> P, G, M, V;             // CtdTrainLayout
  CtdBuf<float> rm1, rv1, rm2, rv2;     // BatchNorm running statistics
  CtdBuf<float> X, XT, Z1, H1, H1T, Z2, H2, H2T, H3, dY, dZ3, dZ3T, dH2, dZ2T, dH1, dZ1T, W2T, W3T, inv1, inv2, zero;
  CtdBuf<double> T, loss;
};

// one value model as the engine holds it (ctd_set_value_model_slot): the fused search and the fp32 kernel read the BN-folded
// [in][out] weights, the tcgen05 kernels, by TMA, their split TF32 terms
struct CtdValueSlot {
  bool ready;              // the last load completed
  CtdBuf<float> d_model;   // BN folded, transposed
  CtdValueModel model;
  // the weights pre-split into their three TF32 terms, [3][N][K] per layer, and their tensor maps (TMA loads of the B operand)
  CtdBuf<float> d_wsplit;
  CUtensorMap tmap[3];
};

#define CTD_MAX_ARENAS 6
struct ctd_engine {
  int device;
  uint32_t slots_rs_n;      // slots [0, slots_rs_n) are known to hold games of ruleset slots_rs (ctd_reset / ctd_load_states):
  int slots_rs;             // lets ctd_playout_slots pick a specialised kernel
  uint32_t capacity;
  CtdBuf<ctd_state> d_slots;
  cudaStream_t stream;
  cudaStream_t stream2;            // second stream of the deep-MCCFR wave pipeline (created on first use)
  CtdBuf<unsigned long long> d_counter2;
  CtdBuf<uint32_t> d_n_pending2;
  cudaEvent_t ev_join;
  CtdBuf<uint32_t, true> h_np;     // pinned host words the waves report into
  bool own_stream;
  uint64_t seed;
  uint64_t launches;
  // replay tapes
  CtdBuf<uint8_t> d_tape;
  CtdBuf<uint32_t> d_tape_off;
  uint32_t n_tapes;
  // scratch
  CtdBuf<uint8_t> d_scratch;
  CtdBuf<unsigned long long> d_counter;
  CtdBuf<ctd_playout_stats> d_stats;
  cudaEvent_t ev0, ev1;
  int sm_count;
  // CFR roots (device): parallel to slots
  CtdBuf<CtdKnow> d_knows;
  CtdBuf<uint8_t> d_used_cards;
  CtdBuf<uint64_t> d_gids;
  CtdBuf<uint32_t> d_root_step;
  // MCCFR trees: one 256-byte header per root + arenas the trees allocate from (arena 0: the whole batch; 1..: retries of
  // trees that found an arena exhausted, each with a larger budget per tree)
  CtdBuf<CtdTreeHdr> d_hdrs;
  CtdBuf<uint8_t> d_arena[CTD_MAX_ARENAS];
  CtdBuf<unsigned long long> d_arena_used;   // [CTD_MAX_ARENAS]
  uint32_t trees_n;                          // roots searched by the last ctd_mccfr / ctd_mccfr_pred call
  CtdBuf<ctd_mccfr_result> d_results;
  CtdBuf<uint32_t> d_list;                   // retry lists
  CtdBuf<uint64_t> d_opts_scratch;
  // value models (slot 0: ctd_set_value_model) and deep-MCCFR batch buffers
  CtdValueSlot vm[CTD_MAX_VALUE_MODELS];
  CtdBuf<float> d_feat;
  CtdBuf<float> d_pred;
  CtdBuf<uint8_t> d_pending;
  CtdBuf<uint32_t> d_n_pending;
  CtdBuf<uint32_t> d_n_epool;   // [1] trees that found their arena exhausted in the passes since it was last cleared
  // tensor-core path of the value model: activations between layers, error flag
  CtdBuf<float> d_h1, d_h2, d_h3;
  CtdBuf<int> d_tc_err;
  int value_backend;  // batched evaluations: 0 = fp32 CUDA cores (ctd_k_value_mlp), 1 = tcgen05 split-TF32 (ctd_k_linear_tc_tma)
  int fused;          // deep MCCFR: 1 = one launch, every warp evaluates its own leaves (ctd_value_inline); 0 = waves + batched evaluation
  CtdBuf<uint8_t, true> h_pinned;        // pinned host staging for result copies
  std::unique_ptr<CtdTrainer> trainer;   // value-network training (ctd_train_*), created on first use
  CtdBuf<uint8_t> d_one;  // single-game staging: state | know6 | used_cards | count | winner | opts
  // self-play dataset (ctd_dataset_*, ctd_arena_record): rows of CTD_FEATURES_PAD floats, metas and origins; option slots
  uint32_t ds_max_records, ds_max_slots;   // 0: not reserved
  CtdBuf<float> ds_feat;
  CtdBuf<ctd_target_meta> ds_meta;
  CtdBuf<ctd_record_origin> ds_origin;
  CtdBuf<ctd_option> ds_opt;
  CtdBuf<double> ds_reg;
  CtdBuf<CtdDatasetCtr> ds_ctr;
  char err[256];
};

static ctd_status ctd_fail(ctd_engine* e, cudaError_t c, const char* where) {
  snprintf(e->err, sizeof(e->err), "%s: %s", where, cudaGetErrorString(c));
  return CTD_ECUDA;
}
#define CTD_CUDA(e, call)                                   \
  do {                                                      \
    cudaError_t _c = (call);                                \
    if (_c != cudaSuccess) return ctd_fail(e, _c, #call);   \
  } while (0)

static CtdTapes ctd_tapes(const ctd_engine* e) { return CtdTapes{e->d_tape, e->d_tape_off, e->n_tapes}; }
static inline uint32_t ctd_blocks(uint32_t n) { return (n + CTD_WARPS_PER_BLOCK - 1) / CTD_WARPS_PER_BLOCK; }

// A persistent kernel as compiled in its own unit (DESIGN.md 3): its launch and how many of its blocks one SM holds.
template <class Args>
struct CtdPersistent {
  int sm_count;
  int per_sm;
  cudaError_t (*launch)(const Args&, int grid, cudaStream_t);
  int per_block = CTD_WARPS_PER_BLOCK;   // items one block works on at once: one per warp, or one per thread (the playouts)
  // enough blocks to fill every SM at the kernel's occupancy, fewer when `n` items need fewer (at least one)
  int grid(uint64_t n) const {
    const uint64_t want = (uint64_t)sm_count * (per_sm < 1 ? 1 : per_sm), need = (n + per_block - 1) / per_block;
    return need == 0 ? 1 : (int)(need < want ? need : want);
  }
};
// the specialised kernel of each family for games of ruleset `rs` (any other value: the generic one)
static cudaError_t ctd_playout_kernel(int rs, CtdPersistent<CtdPlayoutArgs>& k) {
  k.per_block = CTD_BLOCK;   // one game per thread (ctd_playout.cuh)
  if (rs == CTD_RULESET_PRESET) { k.launch = ctd_playout_preset_launch; return ctd_playout_preset_blocks_per_sm(&k.per_sm); }
  if (rs == CTD_RULESET_CLASSIC) { k.launch = ctd_playout_classic_launch; return ctd_playout_classic_blocks_per_sm(&k.per_sm); }
  k.launch = ctd_playout_generic_launch;
  return ctd_playout_generic_blocks_per_sm(&k.per_sm);
}
static cudaError_t ctd_mccfr_kernel(int rs, CtdPersistent<CtdMccfrArgs>& k) {
  if (rs == CTD_RULESET_PRESET) { k.launch = ctd_mccfr_preset_launch; return ctd_mccfr_preset_blocks_per_sm(&k.per_sm); }
  k.launch = ctd_mccfr_generic_launch;
  return ctd_mccfr_generic_blocks_per_sm(&k.per_sm);
}
// fused != 0: the fused mode's occupancy (its dynamic shared memory)
static cudaError_t ctd_pred_kernel(int rs, int fused, CtdPersistent<CtdPredArgs>& k) {
  if (rs == CTD_RULESET_PRESET) { k.launch = ctd_mccfr_pred_preset_launch; return ctd_mccfr_pred_preset_blocks_per_sm(&k.per_sm, fused); }
  k.launch = ctd_mccfr_pred_generic_launch;
  return ctd_mccfr_pred_generic_blocks_per_sm(&k.per_sm, fused);
}

extern "C" {

ctd_status ctd_create(int device, uint32_t capacity, ctd_engine** out) {
  if (!out || capacity == 0) return CTD_EARG;
  ctd_engine* e = new (std::nothrow) ctd_engine();
  if (!e) return CTD_ENOMEM;
  e->device = device;
  e->capacity = capacity;
  e->value_backend = 1;  // batched evaluations: dense layers on the tensor cores
  e->fused = 1;          // deep MCCFR: fused (measured 1.27x the wave scheduler at 4096 roots)
  *out = e;
  CTD_CUDA(e, cudaSetDevice(device));
  CTD_CUDA(e, cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  e->own_stream = true;
  CTD_CUDA(e, e->d_slots.grow((size_t)capacity * sizeof(ctd_state)));
  CTD_CUDA(e, cudaMemsetAsync(e->d_slots, 0, (size_t)capacity * sizeof(ctd_state), e->stream));
  CTD_CUDA(e, e->d_counter.grow(sizeof(unsigned long long)));
  CTD_CUDA(e, e->d_n_epool.grow(sizeof(uint32_t)));
  CTD_CUDA(e, e->d_stats.grow(sizeof(ctd_playout_stats)));
  CTD_CUDA(e, cudaEventCreate(&e->ev0));
  CTD_CUDA(e, cudaEventCreate(&e->ev1));
  CTD_CUDA(e, cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, device));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

void ctd_destroy(ctd_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  if (e->stream2) cudaStreamDestroy(e->stream2);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
  delete e;   // the buffers and the trainer free themselves
}

const char* ctd_last_error(const ctd_engine* e) { return e ? e->err : "null engine"; }
// sizes of the records that cross the boundary (binding self-check): 0 ctd_state, 1 ctd_mccfr_result, 2 ctd_target_meta,
// 3 knowledge block, 4 exported tree header, 5 exported node, 6 child entry, 7 ctd_playout_stats, 8 ctd_arena_seat, 9 ctd_record_origin
uint32_t ctd_sizeof(int what) {
  switch (what) {
    case 0: return (uint32_t)sizeof(ctd_state);
    case 1: return (uint32_t)sizeof(ctd_mccfr_result);
    case 2: return (uint32_t)sizeof(ctd_target_meta);
    case 3: return (uint32_t)sizeof(CtdKnow);
    case 4: return (uint32_t)sizeof(CtdTreeHdrOut);
    case 5: return (uint32_t)sizeof(CtdNodeOut);
    case 6: return (uint32_t)sizeof(CtdChild);
    case 7: return (uint32_t)sizeof(ctd_playout_stats);
    case 8: return (uint32_t)sizeof(ctd_arena_seat);
    case 9: return (uint32_t)sizeof(ctd_record_origin);
    default: return 0;
  }
}
uint64_t ctd_launch_count(const ctd_engine* e) { return e ? e->launches : 0; }

ctd_status ctd_sync(ctd_engine* e) {
  if (!e) return CTD_EARG;
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_set_stream(ctd_engine* e, void* cuda_stream) {
  if (!e) return CTD_EARG;
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (e->own_stream) CTD_CUDA(e, cudaStreamDestroy(e->stream));
  e->stream = (cudaStream_t)cuda_stream;
  e->own_stream = false;
  return CTD_OK;
}

ctd_status ctd_set_seed(ctd_engine* e, uint64_t seed) {
  if (!e) return CTD_EARG;
  e->seed = seed;
  return CTD_OK;
}

ctd_status ctd_reset(ctd_engine* e, uint32_t n, uint64_t seed, uint64_t first_gid, int ruleset) {
  if (!e || n > e->capacity || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  e->seed = seed;
  e->slots_rs = ruleset; e->slots_rs_n = n;
  ctd_k_reset<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_slots, n, seed, first_gid, ruleset, ctd_tapes(e));
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  return CTD_OK;
}

ctd_status ctd_load_states(ctd_engine* e, uint32_t first_slot, uint32_t n, const ctd_state* states) {
  if (!e || !states || (uint64_t)first_slot + n > e->capacity) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  if (n != 0) {  // keep track of the leading run of slots known to hold games of one ruleset (picks a specialised playout kernel)
    const int rs = states[0].ruleset;
    bool uniform = true;
    for (uint32_t i = 1; i < n && uniform; ++i) uniform = states[i].ruleset == rs;
    if (uniform && first_slot == 0 && n >= e->slots_rs_n) {
      e->slots_rs = rs; e->slots_rs_n = n;                         // the run is replaced
    } else if (uniform && rs == e->slots_rs && first_slot <= e->slots_rs_n) {
      if (first_slot + n > e->slots_rs_n) e->slots_rs_n = first_slot + n;   // the run is extended
    } else if (first_slot < e->slots_rs_n) {
      e->slots_rs_n = first_slot;                                  // the run is cut where foreign records begin
    }
  }
  CTD_CUDA(e, cudaMemcpyAsync(e->d_slots + first_slot, states, (size_t)n * sizeof(ctd_state), cudaMemcpyHostToDevice,
                              e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_store_states(ctd_engine* e, uint32_t first_slot, uint32_t n, ctd_state* states) {
  if (!e || !states || (uint64_t)first_slot + n > e->capacity) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, cudaMemcpyAsync(states, e->d_slots + first_slot, (size_t)n * sizeof(ctd_state), cudaMemcpyDeviceToHost,
                              e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_states_dev(ctd_engine* e, void** dev_ptr) {
  if (!e || !dev_ptr) return CTD_EARG;
  e->slots_rs_n = 0;   // the caller may write the slots behind the engine's back
  *dev_ptr = e->d_slots;
  return CTD_OK;
}

ctd_status ctd_set_tapes(ctd_engine* e, uint32_t n, const uint8_t* tape, const uint32_t* tape_off) {
  if (!e || n > e->capacity) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  CTD_CUDA(e, e->d_tape.reset());
  CTD_CUDA(e, e->d_tape_off.reset());
  e->n_tapes = 0;
  if (n == 0) return CTD_OK;
  if (!tape || !tape_off) return CTD_EARG;
  size_t bytes = tape_off[n];
  CTD_CUDA(e, e->d_tape.grow(bytes ? bytes : 1));
  CTD_CUDA(e, e->d_tape_off.grow((size_t)(n + 1) * sizeof(uint32_t)));
  CTD_CUDA(e, cudaMemcpy(e->d_tape, tape, bytes, cudaMemcpyHostToDevice));
  CTD_CUDA(e, cudaMemcpy(e->d_tape_off, tape_off, (size_t)(n + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice));
  e->n_tapes = n;
  return CTD_OK;
}

ctd_status ctd_enumerate(ctd_engine* e, uint32_t n, ctd_option* opts, uint32_t* counts, uint32_t stride) {
  if (!e || !opts || !counts || n > e->capacity || stride == 0) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  size_t ob = (size_t)n * stride * sizeof(ctd_option), cb = (size_t)n * sizeof(uint32_t);
  size_t cb_al = (cb + 255) & ~(size_t)255, eb_al = ((size_t)n + 255) & ~(size_t)255;
  CTD_CUDA(e, e->d_scratch.grow(ob + cb_al + eb_al + 256 + (size_t)n * sizeof(ctd_state)));
  ctd_option* d_opts = (ctd_option*)e->d_scratch.get();
  uint32_t* d_counts = (uint32_t*)(e->d_scratch + ob);
  uint8_t* d_errs = e->d_scratch + ob + cb_al;
  uint32_t* d_dirty = (uint32_t*)(e->d_scratch + ob + cb_al + eb_al);
  ctd_state* d_shadow = (ctd_state*)(e->d_scratch + ob + cb_al + eb_al + 256);
  CTD_CUDA(e, cudaMemsetAsync(d_dirty, 0, 4, e->stream));
  ctd_k_enumerate<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_slots, n, d_opts, d_counts, stride, d_errs, e->seed, ctd_tapes(e),
                                                              d_shadow, d_dirty);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  uint32_t dirty = 0;
  CTD_CUDA(e, cudaMemcpyAsync(counts, d_counts, cb, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(&dirty, d_dirty, 4, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(opts, d_opts, ob, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  for (uint32_t i = 0; i < n; ++i)
    if (counts[i] > stride) return CTD_ECAP;
  if (dirty) {  // Seer / Scholar enumerations changed their records: commit
    CTD_CUDA(e, cudaMemcpyAsync(e->d_slots, d_shadow, (size_t)n * sizeof(ctd_state), cudaMemcpyDeviceToDevice, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  }
  return CTD_OK;
}

ctd_status ctd_choose_check(ctd_engine* e, uint32_t n, uint32_t* mismatches) {
  if (!e || !mismatches || n > e->capacity) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  const uint32_t cap = 4096;
  size_t ob = (size_t)n * cap * sizeof(ctd_option);
  CTD_CUDA(e, e->d_scratch.grow(ob + (size_t)n * 4));
  uint32_t* d_mis = (uint32_t*)(e->d_scratch + ob);
  ctd_k_choose_check<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_slots, n, d_mis, (uint64_t*)e->d_scratch.get(), cap);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaMemcpyAsync(mismatches, d_mis, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_step(ctd_engine* e, uint32_t n, const ctd_option* chosen, int8_t* winner) {
  if (!e || !chosen || n > e->capacity) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  size_t ob = (size_t)n * sizeof(ctd_option);
  CTD_CUDA(e, e->d_scratch.grow(ob + n));
  ctd_option* d_chosen = (ctd_option*)e->d_scratch.get();
  int8_t* d_winner = (int8_t*)e->d_scratch.get() + ob;
  CTD_CUDA(e, cudaMemcpyAsync(d_chosen, chosen, ob, cudaMemcpyHostToDevice, e->stream));
  ctd_k_step<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_slots, n, d_chosen, d_winner, e->seed, ctd_tapes(e));
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  if (winner) CTD_CUDA(e, cudaMemcpyAsync(winner, d_winner, n, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

static ctd_status ctd_playout_launch(ctd_engine* e, CtdPlayoutArgs& a, ctd_playout_stats* stats, float* elapsed_ms) {
  // every game of this launch is known to play the preset eight: the specialised kernel (ctd_preset_playout.cu)
  const int rs = a.slots == nullptr ? a.ruleset : (a.n_games <= e->slots_rs_n ? e->slots_rs : -1);
  CtdPersistent<CtdPlayoutArgs> k{e->sm_count, 0, nullptr};
  CTD_CUDA(e, ctd_playout_kernel(rs, k));
  CTD_CUDA(e, cudaMemsetAsync(e->d_counter, 0, sizeof(unsigned long long), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(e->d_stats, 0, sizeof(ctd_playout_stats), e->stream));
  a.counter = e->d_counter;
  a.stats = e->d_stats;
  CTD_CUDA(e, cudaEventRecord(e->ev0, e->stream));
  CTD_CUDA(e, k.launch(a, k.grid(a.n_games), e->stream));
  e->launches++;
  CTD_CUDA(e, cudaEventRecord(e->ev1, e->stream));
  if (stats) CTD_CUDA(e, cudaMemcpyAsync(stats, e->d_stats, sizeof(ctd_playout_stats), cudaMemcpyDeviceToHost, e->stream));
  (void)elapsed_ms;
  return CTD_OK;
}

ctd_status ctd_playout_dev(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                           uint32_t max_steps, ctd_playout_stats* stats, float* elapsed_ms) {
  if (!e || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdPlayoutArgs a;
  memset(&a, 0, sizeof(a));
  a.n_games = n_games; a.seed = seed; a.first_gid = first_gid; a.ruleset = ruleset; a.max_steps = max_steps;
  ctd_status s = ctd_playout_launch(e, a, stats, elapsed_ms);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (elapsed_ms) CTD_CUDA(e, cudaEventElapsedTime(elapsed_ms, e->ev0, e->ev1));
  return CTD_OK;
}

ctd_status ctd_playout(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                       uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps, ctd_playout_stats* stats) {
  if (!e || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  if (n_games == 0) { if (stats) memset(stats, 0, sizeof(*stats)); return CTD_OK; }
  CTD_CUDA(e, cudaSetDevice(e->device));
  size_t wb = (n_games + 255) & ~(size_t)255, pb = (n_games * 6 + 255) & ~(size_t)255, sb = n_games * 2;
  CTD_CUDA(e, e->d_scratch.grow(wb + pb + sb));
  CtdPlayoutArgs a;
  memset(&a, 0, sizeof(a));
  a.n_games = n_games; a.seed = seed; a.first_gid = first_gid; a.ruleset = ruleset; a.max_steps = max_steps;
  a.winner = (int8_t*)e->d_scratch.get();
  a.points6 = (int8_t*)e->d_scratch.get() + wb;
  a.steps = (uint16_t*)(e->d_scratch + wb + pb);
  CTD_CUDA(e, e->h_pinned.grow(wb + pb + sb));   // results come back through pinned host memory in one DMA
  ctd_status s = ctd_playout_launch(e, a, stats, nullptr);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaMemcpyAsync(e->h_pinned, e->d_scratch, wb + pb + sb, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (winner) memcpy(winner, e->h_pinned, n_games);
  if (points6) memcpy(points6, e->h_pinned + wb, n_games * 6);
  if (steps) memcpy(steps, e->h_pinned + wb + pb, sb);
  return CTD_OK;
}

ctd_status ctd_playout_slots(ctd_engine* e, uint32_t n, uint32_t max_steps, int8_t* winner, uint16_t* steps) {
  if (!e || n > e->capacity) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  size_t wb = ((size_t)n + 255) & ~(size_t)255, sb = (size_t)n * 2;
  CTD_CUDA(e, e->d_scratch.grow(wb + sb));
  CtdPlayoutArgs a;
  memset(&a, 0, sizeof(a));
  a.n_games = n; a.seed = e->seed; a.max_steps = max_steps; a.slots = e->d_slots;
  a.winner = (int8_t*)e->d_scratch.get();
  a.steps = (uint16_t*)(e->d_scratch + wb);
  ctd_status s = ctd_playout_launch(e, a, nullptr, nullptr);
  if (s != CTD_OK) return s;
  if (winner) CTD_CUDA(e, cudaMemcpyAsync(winner, a.winner, n, cudaMemcpyDeviceToHost, e->stream));
  if (steps) CTD_CUDA(e, cudaMemcpyAsync(steps, a.steps, sb, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// d_knows stands for the whole group: it is handed to the engine only once every buffer is allocated and cleared, so a
// failure part way leaves the group absent and the next call tries again
static ctd_status ctd_root_buffers(ctd_engine* e) {
  if (e->d_knows) return CTD_OK;
  const size_t n = e->capacity;
  CtdBuf<CtdKnow> knows;
  CTD_CUDA(e, knows.grow(n * sizeof(CtdKnow)));
  CTD_CUDA(e, e->d_used_cards.grow(n * 76));
  CTD_CUDA(e, e->d_gids.grow(n * sizeof(uint64_t)));
  CTD_CUDA(e, e->d_root_step.grow(n * sizeof(uint32_t)));
  CTD_CUDA(e, cudaMemsetAsync(knows, 0, n * sizeof(CtdKnow), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(e->d_used_cards, 0, n * 76, e->stream));
  CTD_CUDA(e, cudaMemsetAsync(e->d_gids, 0, n * sizeof(uint64_t), e->stream));
  e->d_knows = std::move(knows);
  return CTD_OK;
}

ctd_status ctd_make_roots(ctd_engine* e, uint32_t n, uint64_t seed, uint64_t first_gid, int ruleset, uint32_t back_lo,
                          uint32_t back_hi, int flavour, uint32_t* root_step) {
  if (!e || n > e->capacity || back_hi < back_lo || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM) ||
      (flavour != CTD_ROOTS_CLOSE_TO_FINISHED && flavour != CTD_ROOTS_RANDOM_GAME))
    return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_root_buffers(e);
  if (s != CTD_OK) return s;
  e->slots_rs_n = 0;
  e->seed = seed;
  CtdRootArgs a{n, seed, first_gid, ruleset, back_lo, back_hi, flavour, e->d_slots, e->d_knows, e->d_used_cards, e->d_gids,
                e->d_root_step};
  ctd_k_make_roots<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(a);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  if (root_step)
    CTD_CUDA(e, cudaMemcpyAsync(root_step, e->d_root_step, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_load_roots(ctd_engine* e, uint32_t n, const ctd_state* roots, const void* knows, const uint8_t* used_cards,
                          const uint64_t* gids) {
  if (!e || n > e->capacity || !roots || !knows || !used_cards || !gids) return CTD_EARG;
  e->slots_rs_n = 0;
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_root_buffers(e);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaMemcpyAsync(e->d_slots, roots, (size_t)n * sizeof(ctd_state), cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(e->d_knows, knows, (size_t)n * sizeof(CtdKnow), cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(e->d_used_cards, used_cards, (size_t)n * 76, cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(e->d_gids, gids, (size_t)n * sizeof(uint64_t), cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_store_roots(ctd_engine* e, uint32_t n, ctd_state* roots, void* knows, uint8_t* used_cards, uint64_t* gids) {
  if (!e || n > e->capacity || !e->d_knows) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  if (roots) CTD_CUDA(e, cudaMemcpyAsync(roots, e->d_slots, (size_t)n * sizeof(ctd_state), cudaMemcpyDeviceToHost, e->stream));
  if (knows) CTD_CUDA(e, cudaMemcpyAsync(knows, e->d_knows, (size_t)n * sizeof(CtdKnow), cudaMemcpyDeviceToHost, e->stream));
  if (used_cards) CTD_CUDA(e, cudaMemcpyAsync(used_cards, e->d_used_cards, (size_t)n * 76, cudaMemcpyDeviceToHost, e->stream));
  if (gids) CTD_CUDA(e, cudaMemcpyAsync(gids, e->d_gids, (size_t)n * sizeof(uint64_t), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// ---- memory plan of a search
// chunk 0 of a tree: the smallest power of two >= 2 x iterations (measured on the reference: 1.7 nodes per iteration on average,
// <= 3.6 for 99 % of preset trees), at least 64
static uint32_t ctd_n0_log2(uint32_t iterations) {
  uint32_t k = 6;
  while (k < 20 && (1ull << k) < 2ull * iterations) ++k;
  return k;
}
// arena bytes budgeted per tree: chunk 0 plus one and a half times as much again for the trees that outgrow it (2000-iteration
// trees from create_a_random_game roots: 1.9 nodes per iteration, 40 % of them take a second chunk; a budget of 1.5 chunks ran
// the shared arena dry at the very end of such a batch and sent the slowest trees through a second search), the node arrays,
// slab slack.
// The classic Magician expands ~1600 children at once and the Cardinal of the random rulesets thousands, more than once per tree:
// those rulesets get a larger share.  A budget is an average, not a limit: trees borrow from each other, and a tree that finds
// the arena exhausted is searched again from a larger one (ctd_search below).
static uint64_t ctd_tree_budget(uint32_t iterations, int ruleset) {
  const uint64_t n0 = 1ull << ctd_n0_log2(iterations);
  uint64_t b = n0 * sizeof(CtdNode) * 5 / 2 + (uint64_t)iterations * 30 * 40 + 4 * CTD_SLAB_UNITS * CTD_ARENA_UNIT;
  if (ruleset == CTD_RULESET_CLASSIC) b *= 4;
  if (ruleset == CTD_RULESET_RANDOM) b *= 8;
  return b;
}
void ctd_mccfr_tree_shape(uint32_t iterations, int ruleset, uint32_t n_roots, uint32_t* first_chunk_nodes, uint32_t* node_bytes,
                          uint64_t* arena_bytes) {
  if (first_chunk_nodes) *first_chunk_nodes = 1u << ctd_n0_log2(iterations);
  if (node_bytes) *node_bytes = (uint32_t)sizeof(CtdNode);
  if (arena_bytes) *arena_bytes = ctd_tree_budget(iterations, ruleset) * n_roots + (64ull << 20);
}

static ctd_status ctd_ensure_arena(ctd_engine* e, int idx, size_t bytes) {
  CTD_CUDA(e, e->d_arena_used.grow(CTD_MAX_ARENAS * sizeof(unsigned long long)));
  if (!e->d_hdrs) {
    CTD_CUDA(e, e->d_hdrs.grow((size_t)e->capacity * sizeof(CtdTreeHdr)));
    CTD_CUDA(e, cudaMemsetAsync(e->d_hdrs, 0, (size_t)e->capacity * sizeof(CtdTreeHdr), e->stream));
  }
  CtdBuf<uint8_t>& arena = e->d_arena[idx];
  if (bytes > arena.bytes) {
    if (arena) CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    CTD_CUDA(e, arena.reset());
    size_t free_b = 0, total_b = 0;
    CTD_CUDA(e, cudaMemGetInfo(&free_b, &total_b));
    if (bytes > free_b - free_b / 8) bytes = free_b - free_b / 8;   // leave an eighth of what is free to everybody else
    bytes &= ~(size_t)255;
    cudaError_t c = arena.grow(bytes);
    if (c != cudaSuccess) { (void)cudaGetLastError(); snprintf(e->err, sizeof(e->err), "tree arena of %zu bytes: %s", bytes, cudaGetErrorString(c)); return CTD_ENOMEM; }
  }
  const unsigned long long one = 1;   // offset 0 means "none"
  CTD_CUDA(e, cudaMemcpyAsync(e->d_arena_used + idx, &one, sizeof(one), cudaMemcpyHostToDevice, e->stream));
  return CTD_OK;
}
static CtdArena ctd_arena_of(ctd_engine* e, int idx) {
  return CtdArena{e->d_arena[idx], e->d_arena_used + idx, (unsigned long long)(e->d_arena[idx].bytes / CTD_ARENA_UNIT)};
}

// what one search call asks for
struct CtdSearch {
  uint32_t n_roots;
  uint64_t seed;
  uint32_t iterations;
  int ruleset;
  bool deep;
  uint32_t max_depth;
  float weight;
  bool resume;      // pure MCCFR only: continue the trees of the previous call for `iterations` more
  int model;        // deep MCCFR: the value-model slot that evaluates the leaves
};
static ctd_status ctd_value_forward(ctd_engine* e, const CtdValueSlot& vm, uint32_t n, const uint8_t* pending, float weight, uint32_t row0,
                                    cudaStream_t st);
static ctd_status ctd_pred_buffers(ctd_engine* e);

// one pass of pure MCCFR over `n` trees (d_list: their root indices, or null for roots [0, n)) allocating from arena `ai`
static ctd_status ctd_pure_pass(ctd_engine* e, const CtdSearch& sp, const uint32_t* d_list, uint32_t n, int ai) {
  CtdPersistent<CtdMccfrArgs> k{e->sm_count, 0, nullptr};   // the roots were made / loaded for this ruleset: its kernel
  CTD_CUDA(e, ctd_mccfr_kernel(sp.ruleset, k));
  const int grid = k.grid(n);
  CTD_CUDA(e, e->d_opts_scratch.grow((size_t)grid * CTD_WARPS_PER_BLOCK * CTD_MCCFR_OPT_CAP * sizeof(uint64_t)));
  CtdMccfrArgs a;
  memset(&a, 0, sizeof(a));
  a.n_roots = n; a.tree_list = d_list; a.roots = e->d_slots; a.knows = e->d_knows; a.used_cards = e->d_used_cards; a.gids = e->d_gids;
  a.seed = sp.seed; a.iterations = sp.iterations; a.n0_log2 = ctd_n0_log2(sp.iterations); a.hdrs = e->d_hdrs; a.arena = ctd_arena_of(e, ai);
  a.results = e->d_results; a.counter = e->d_counter; a.opts_scratch = e->d_opts_scratch; a.resume = sp.resume ? 1 : 0;
  a.n_epool = e->d_n_epool;
  CTD_CUDA(e, cudaMemsetAsync(e->d_counter, 0, sizeof(unsigned long long), e->stream));
  CTD_CUDA(e, k.launch(a, grid, e->stream));
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  return CTD_OK;
}

// one pass of deep MCCFR over `n` trees.  Trees advance in waves: every tree walks until it needs a leaf value (or has spent
// its wave budget), the value model runs on the batch of all waiting leaves, the trees resume.
static ctd_status ctd_deep_pass(ctd_engine* e, const CtdSearch& sp, const uint32_t* d_list, uint32_t n, int ai, uint32_t* waves_out) {
  CtdPredArgs p;
  memset(&p, 0, sizeof(p));
  CtdMccfrArgs& a = p.m;
  a.roots = e->d_slots; a.knows = e->d_knows; a.used_cards = e->d_used_cards; a.gids = e->d_gids;
  a.seed = sp.seed; a.iterations = sp.iterations; a.n0_log2 = ctd_n0_log2(sp.iterations); a.hdrs = e->d_hdrs; a.arena = ctd_arena_of(e, ai);
  a.results = e->d_results; a.n_epool = e->d_n_epool;
  // wave budget: trees that never reach the depth limit would otherwise walk all their iterations in the first wave
  const uint32_t wave_budget = 20;   // measured best at 4096 roots x 200 iterations (8: 8.4e6, 20: 1.12e7, 64: 8.9e6, unbounded: 7.3e6 it/s)
  p.budget = wave_budget;
  p.max_depth = sp.max_depth; p.feat = e->d_feat; p.pred = e->d_pred; p.pending = e->d_pending;
  CtdPersistent<CtdPredArgs> k{e->sm_count, 0, nullptr};
  CTD_CUDA(e, ctd_pred_kernel(sp.ruleset, e->fused, k));
  if (e->fused) {
    // fused: one launch; every warp walks its tree to the end and evaluates the leaves it meets itself (ctd_value_inline)
    p.fused = 1; p.budget = 0xFFFFFFFFu; p.first = 1;
    const CtdValueModel& m = e->vm[sp.model].model;
    p.net = CtdValueNet{m.w1t, m.b1, m.w2t, m.b2, m.w3t, m.b3, m.w4t, m.b4, sp.weight};
    const int grid = k.grid(n);
    CTD_CUDA(e, e->d_opts_scratch.grow((size_t)grid * CTD_WARPS_PER_BLOCK * CTD_MCCFR_OPT_CAP * sizeof(uint64_t)));
    a.tree_list = d_list; a.first_root = 0; a.n_roots = n; a.counter = e->d_counter; a.opts_scratch = e->d_opts_scratch;
    p.n_pending = e->d_n_pending;
    CTD_CUDA(e, cudaMemsetAsync(e->d_counter, 0, sizeof(unsigned long long), e->stream));
    CTD_CUDA(e, cudaMemsetAsync(e->d_n_pending, 0, 2 * sizeof(uint32_t), e->stream));
    CTD_CUDA(e, k.launch(p, grid, e->stream));
    e->launches++;
    CTD_CUDA(e, cudaGetLastError());
    if (waves_out) *waves_out = 1;
    return CTD_OK;
  }
  // Two groups of trees take turns: each group's waves (walk kernel -> batched leaf evaluation -> walk kernel ...) run on
  // their own stream, so the tail of one group's wave -- a few trees with expensive expansions -- overlaps with the other
  // group's kernel instead of idling the GPU.  Trees are independent, results do not depend on the grouping.
  // A retry pass (d_list) runs as one group: its rows are indexed by root, so two groups would evaluate each other's rows.
  const int G = n >= 1024 && !d_list ? 2 : 1;
  if (G == 2 && !e->ev_join) {   // the join event comes last: a failure part way is completed by the next call
    if (!e->stream2) CTD_CUDA(e, cudaStreamCreateWithFlags(&e->stream2, cudaStreamNonBlocking));
    CTD_CUDA(e, e->d_counter2.grow(sizeof(unsigned long long)));
    CTD_CUDA(e, e->d_n_pending2.grow(2 * sizeof(uint32_t)));
    CTD_CUDA(e, cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
  }
  const uint32_t split = G == 2 ? ((n / 2 + 7) & ~7u) : n;
  const uint32_t g_first[2] = {0, split}, g_n[2] = {split, n - split};
  cudaStream_t g_stream[2] = {e->stream, G == 2 ? e->stream2 : e->stream};
  unsigned long long* g_counter[2] = {e->d_counter, e->d_counter2};
  uint32_t* g_pending[2] = {e->d_n_pending, e->d_n_pending2};
  int g_grid[2];
  size_t g_opts_off[2] = {0, 0}, warps = 0;
  for (int g = 0; g < G; ++g) {
    g_grid[g] = k.grid(g_n[g]);
    g_opts_off[g] = warps * CTD_MCCFR_OPT_CAP;
    warps += (size_t)g_grid[g] * CTD_WARPS_PER_BLOCK;
  }
  CTD_CUDA(e, e->d_opts_scratch.grow(warps * CTD_MCCFR_OPT_CAP * sizeof(uint64_t)));
  ctd_status s = CTD_OK;
  if (G == 2) {
    CTD_CUDA(e, cudaEventRecord(e->ev_join, e->stream));
    CTD_CUDA(e, cudaStreamWaitEvent(e->stream2, e->ev_join, 0));
  }
  uint32_t g_waves[2] = {0, 0};
  bool g_done[2] = {false, G == 1};
  uint32_t* h_np = e->h_np;   // pinned: [group][2]
  auto launch_wave = [&](int g) -> ctd_status {
    CtdPredArgs q = p;
    q.m.tree_list = d_list ? d_list + g_first[g] : nullptr;
    q.m.first_root = d_list ? 0 : g_first[g]; q.m.n_roots = g_n[g]; q.m.counter = g_counter[g]; q.n_pending = g_pending[g];
    q.m.opts_scratch = e->d_opts_scratch + g_opts_off[g];
    q.first = g_waves[g] == 0;
    CTD_CUDA(e, cudaMemsetAsync(g_counter[g], 0, sizeof(unsigned long long), g_stream[g]));
    CTD_CUDA(e, cudaMemsetAsync(g_pending[g], 0, 2 * sizeof(uint32_t), g_stream[g]));
    CTD_CUDA(e, k.launch(q, g_grid[g], g_stream[g]));
    e->launches++;
    CTD_CUDA(e, cudaMemcpyAsync(h_np + 2 * g, g_pending[g], 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, g_stream[g]));
    ++g_waves[g];
    return CTD_OK;
  };
  for (int g = 0; g < G; ++g) { s = launch_wave(g); if (s != CTD_OK) return s; }
  while (!(g_done[0] && g_done[1])) {
    for (int g = 0; g < G; ++g) {
      if (g_done[g]) continue;
      CTD_CUDA(e, cudaStreamSynchronize(g_stream[g]));
      const uint32_t waiting = h_np[2 * g], yielded = h_np[2 * g + 1];
      if (waiting == 0 && yielded == 0) { g_done[g] = true; continue; }
      if (g_waves[g] > 2 * sp.iterations + 4) { snprintf(e->err, sizeof(e->err), "ctd_mccfr_pred: wave limit"); return CTD_ECAP; }
      if (waiting != 0) {
        // the feature / pending rows are indexed by root: with a retry list the model runs over every row of the call and the
        // pending mask picks the waiting ones
        const uint32_t row0 = d_list ? 0 : g_first[g], rows = d_list ? sp.n_roots : g_n[g];
        s = ctd_value_forward(e, e->vm[sp.model], rows, e->d_pending + row0, sp.weight, row0, g_stream[g]);
        if (s != CTD_OK) return s;
      }
      s = launch_wave(g);
      if (s != CTD_OK) return s;
    }
  }
  if (G == 2) {   // join: the engine's stream continues after both groups
    CTD_CUDA(e, cudaEventRecord(e->ev_join, e->stream2));
    CTD_CUDA(e, cudaStreamWaitEvent(e->stream, e->ev_join, 0));
  }
  if (waves_out) *waves_out = g_waves[0] > g_waves[1] ? g_waves[0] : g_waves[1];
  if (e->value_backend == 1 && !e->fused) {   // a tcgen05 kernel that timed out on an mbarrier skips its stores: never hand such values to the trees silently
    int terr = 0;
    CTD_CUDA(e, cudaMemcpyAsync(&terr, e->d_tc_err, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    if (terr) {
      CTD_CUDA(e, cudaMemsetAsync(e->d_tc_err, 0, sizeof(int), e->stream));
      snprintf(e->err, sizeof(e->err), "tcgen05 value kernel: mbarrier wait timed out");
      return CTD_ECUDA;
    }
  }
  return CTD_OK;
}

// The search proper.  The reference never refuses a root, so neither does this: all trees share arena 0; trees that found it
// exhausted (status CTD_TREE_EPOOL) are searched again from scratch, by themselves, from a further arena with 16x the budget per
// tree, and so on (a tree is a pure function of (seed, root, gid), so the second search is the same search).
static ctd_status ctd_search(ctd_engine* e, const CtdSearch& sp, ctd_mccfr_result* results, float* elapsed_ms, uint32_t* waves_out) {
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, e->d_results.grow((size_t)sp.n_roots * sizeof(ctd_mccfr_result)));
  // a record's arrays are written up to the root's children only: the rest of the record must not keep an earlier call's tree
  CTD_CUDA(e, cudaMemsetAsync(e->d_results, 0, (size_t)sp.n_roots * sizeof(ctd_mccfr_result), e->stream));
  ctd_status s = CTD_OK;
  if (sp.deep) { s = ctd_pred_buffers(e); if (s != CTD_OK) return s; }
  if (sp.resume) {   // the trees stay where they are (arena 0 keeps its bump pointer); trees that run out of arena now keep status 2
    if (!e->d_hdrs || sp.n_roots > e->trees_n || sp.deep) return CTD_EARG;
    CTD_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    s = ctd_pure_pass(e, sp, nullptr, sp.n_roots, 0);
    if (s != CTD_OK) return s;
    CTD_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    if (results) CTD_CUDA(e, cudaMemcpyAsync(results, e->d_results, (size_t)sp.n_roots * sizeof(ctd_mccfr_result), cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    if (elapsed_ms) CTD_CUDA(e, cudaEventElapsedTime(elapsed_ms, e->ev0, e->ev1));
    return CTD_OK;
  }
  uint64_t budget = ctd_tree_budget(sp.iterations, sp.ruleset);
  size_t arena0 = (size_t)(budget * sp.n_roots + (64ull << 20));
  if (const char* env = getenv("CTD_ARENA0_BYTES")) {   // test hook: a squeezed first arena exercises the retry path
    arena0 = (size_t)strtoull(env, nullptr, 10);
    if (e->d_arena[0] && e->d_arena[0].bytes != arena0) { CTD_CUDA(e, cudaStreamSynchronize(e->stream)); CTD_CUDA(e, e->d_arena[0].reset()); }
  }
  s = ctd_ensure_arena(e, 0, arena0);
  if (s != CTD_OK) return s;
  e->trees_n = sp.n_roots;
  CTD_CUDA(e, cudaMemsetAsync(e->d_n_epool, 0, sizeof(uint32_t), e->stream));
  CTD_CUDA(e, cudaEventRecord(e->ev0, e->stream));
  s = sp.deep ? ctd_deep_pass(e, sp, nullptr, sp.n_roots, 0, waves_out) : ctd_pure_pass(e, sp, nullptr, sp.n_roots, 0);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaEventRecord(e->ev1, e->stream));
  // which trees ran out of arena?  (status word of every header: 256-byte stride, 4 bytes each)
  std::unique_ptr<uint32_t[]> st(new (std::nothrow) uint32_t[sp.n_roots]);
  if (!st) return CTD_ENOMEM;
  for (int ai = 1; ai < CTD_MAX_ARENAS; ++ai) {
    uint32_t any = 0;   // one word first: the strided read-back of every header's status costs a DMA descriptor per tree
    CTD_CUDA(e, cudaMemcpyAsync(&any, e->d_n_epool, sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    if (any == 0) break;
    CTD_CUDA(e, cudaMemsetAsync(e->d_n_epool, 0, sizeof(uint32_t), e->stream));
    CTD_CUDA(e, cudaMemcpy2DAsync(st.get(), sizeof(uint32_t), (const uint8_t*)e->d_hdrs.get() + offsetof(CtdTreeHdr, status),
                                  sizeof(CtdTreeHdr), sizeof(uint32_t), sp.n_roots, cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    uint32_t nf = 0;
    for (uint32_t t = 0; t < sp.n_roots; ++t) if (st[t] & CTD_TREE_EPOOL) st[nf++] = t;
    if (nf == 0) break;
    CTD_CUDA(e, e->d_list.grow((size_t)nf * sizeof(uint32_t)));
    CTD_CUDA(e, cudaMemcpyAsync(e->d_list, st.get(), (size_t)nf * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
    budget *= 16;
    s = ctd_ensure_arena(e, ai, (size_t)(budget * nf + (64ull << 20)));
    if (s != CTD_OK) return s;
    s = sp.deep ? ctd_deep_pass(e, sp, e->d_list, nf, ai, nullptr) : ctd_pure_pass(e, sp, e->d_list, nf, ai);
    if (s != CTD_OK) return s;
    CTD_CUDA(e, cudaEventRecord(e->ev1, e->stream));   // the reported kernel time covers every pass
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));     // `st` is reused as the upload source
  }
  if (results) CTD_CUDA(e, cudaMemcpyAsync(results, e->d_results, (size_t)sp.n_roots * sizeof(ctd_mccfr_result), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (elapsed_ms) CTD_CUDA(e, cudaEventElapsedTime(elapsed_ms, e->ev0, e->ev1));
  return CTD_OK;
}

ctd_status ctd_mccfr(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, int ruleset,
                     ctd_mccfr_result* results, float* elapsed_ms) {
  if (!e || n_roots > e->capacity || !e->d_knows || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  if (n_roots == 0) return CTD_OK;
  CtdSearch sp{n_roots, seed, iterations, ruleset, false, 0, 0.f, false};
  return ctd_search(e, sp, results, elapsed_ms, nullptr);
}

// ---- root-parallel mode (labelled: NOT the reference's algorithm, see DESIGN.md 6) ----
// more iterations on the trees the last ctd_mccfr call grew (same n_roots, seed, ruleset), from where their walks stood
ctd_status ctd_mccfr_continue(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t more_iterations, int ruleset,
                              ctd_mccfr_result* results, float* elapsed_ms) {
  if (!e || !e->d_knows || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  if (n_roots == 0) return CTD_OK;
  CtdSearch sp{n_roots, seed, more_iterations, ruleset, false, 0, 0.f, true};
  return ctd_search(e, sp, results, elapsed_ms, nullptr);
}

__global__ void ctd_k_root_set(CtdTreeHdr* hdrs, uint32_t n, uint32_t stride, const double* R, const double* C, const double* V) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  CtdTree T;
  ctd_tree_attach(T, &hdrs[t], CtdArena{hdrs[t].arena, nullptr, 0});
  if (T.hdr->n_nodes == 0 || (T.hdr->status & ~CTD_TREE_TERMINAL_ROOT)) return;
  CtdNode& n0 = ctd_node(T, 0);
  for (int i = 0; i < 6; ++i) n0.V[i] = V[(size_t)t * 6 + i];
  double vs = 0.0;
  for (int i = 0; i < 6; ++i) vs += n0.V[i];
  if (vs != 0.0) for (int i = 0; i < 6; ++i) n0.P[i] = n0.V[i] / vs;
  if (n0.n_children == 0) return;
  const uint32_t na = (n0.flags & CTD_NF_ROLE_PICK) ? 60u : n0.n_children;
  if (na > stride) return;
  double *r = ctd_R(T, n0), *c = ctd_C(T, n0);
  for (uint32_t i = 0; i < na; ++i) { r[i] = R[(size_t)t * stride + i]; c[i] = C[(size_t)t * stride + i]; }
}
// overwrite node_value, cumulative_regrets and cumulative_strategy of the roots of trees [0, n_roots) (rows of `stride` doubles;
// trees whose arrays are longer than a row keep theirs)
ctd_status ctd_mccfr_root_set(ctd_engine* e, uint32_t n_roots, uint32_t stride, const double* cumulative_regrets,
                              const double* cumulative_strategy, const double* node_value) {
  if (!e || !e->d_hdrs || n_roots > e->trees_n || !cumulative_regrets || !cumulative_strategy || !node_value || stride == 0) return CTD_EARG;
  if (n_roots == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  const size_t ab = (size_t)n_roots * stride * sizeof(double), vb = (size_t)n_roots * 6 * sizeof(double);
  CTD_CUDA(e, e->d_scratch.grow(2 * ab + vb));
  double* d = (double*)e->d_scratch.get();
  CTD_CUDA(e, cudaMemcpyAsync(d, cumulative_regrets, ab, cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(d + (size_t)n_roots * stride, cumulative_strategy, ab, cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(d + 2 * (size_t)n_roots * stride, node_value, vb, cudaMemcpyHostToDevice, e->stream));
  ctd_k_root_set<<<(n_roots + 127) / 128, 128, 0, e->stream>>>(e->d_hdrs, n_roots, stride, d, d + (size_t)n_roots * stride, d + 2 * (size_t)n_roots * stride);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// trees of the last search, roots [first, first + n), as compact blocks (ctd_tree_export in csrc/ctd_mccfr.cuh)
ctd_status ctd_mccfr_export(ctd_engine* e, uint32_t first, uint32_t n, uint64_t* sizes, void* buf, uint64_t buf_bytes) {
  if (!e || !sizes || !e->d_hdrs || (uint64_t)first + n > e->trees_n) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  std::unique_ptr<CtdTreeHdr[]> hh(new (std::nothrow) CtdTreeHdr[n]);
  std::unique_ptr<uint64_t[]> off(new (std::nothrow) uint64_t[n]);
  if (!hh || !off) return CTD_ENOMEM;
  CTD_CUDA(e, cudaMemcpyAsync(hh.get(), e->d_hdrs + first, (size_t)n * sizeof(CtdTreeHdr), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  uint64_t total = 0;
  for (uint32_t i = 0; i < n; ++i) {
    sizes[i] = (ctd_tree_export_bytes(hh[i].n_nodes, hh[i].child_used, hh[i].arr_used) + 15) & ~(uint64_t)15;
    off[i] = total;
    total += sizes[i];
  }
  if (!buf) return CTD_OK;
  if (buf_bytes < total) return CTD_ECAP;
  CtdBuf<uint8_t> d_out;
  CtdBuf<uint64_t> d_off;
  CTD_CUDA(e, d_out.grow(total));
  CTD_CUDA(e, d_off.grow((size_t)n * sizeof(uint64_t)));
  CTD_CUDA(e, cudaMemcpyAsync(d_off, off.get(), (size_t)n * sizeof(uint64_t), cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemsetAsync(d_out, 0, total, e->stream));
  ctd_k_export_trees<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_hdrs, first, n, d_off, d_out);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaMemcpyAsync(buf, d_out, total, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// children [first, first + count) of the root of tree `tree`: descriptors and, for vector nodes, regrets / strategy / cumulative
// strategy (a result record holds the first CTD_MCCFR_MAX_RESULT; the Cardinal expands thousands)
ctd_status ctd_mccfr_root_children(ctd_engine* e, uint32_t tree, uint32_t first, uint32_t count, ctd_option* options, double* R,
                                   double* S, double* C) {
  if (!e || !e->d_hdrs || tree >= e->trees_n || !options || !R || !S || !C) return CTD_EARG;
  if (count == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  const size_t ob = (size_t)count * sizeof(ctd_option), db = (size_t)count * sizeof(double);
  CTD_CUDA(e, e->d_scratch.grow(ob + 3 * db));
  ctd_option* d_o = (ctd_option*)e->d_scratch.get();
  double* d_r = (double*)(e->d_scratch + ob);
  CTD_CUDA(e, cudaMemsetAsync(e->d_scratch, 0, ob + 3 * db, e->stream));
  ctd_k_root_children<<<(count + 255) / 256 < 64 ? (count + 255) / 256 : 64, 256, 0, e->stream>>>(e->d_hdrs, tree, first, count, d_o, d_r, d_r + count, d_r + 2 * count);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaMemcpyAsync(options, d_o, ob, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(R, d_r, db, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(S, d_r + count, db, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(C, d_r + 2 * count, db, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

#define CTD_ONE_OPTS 16384 /* the Cardinal's lists reach ~8000 options */
#define CTD_ONE_KNOW_OFF 256
#define CTD_ONE_KNOW6 (6 * CTD_KNOW_BYTES)
#define CTD_ONE_USED_OFF (256 + CTD_ONE_KNOW6)
#define CTD_ONE_COUNT_OFF (256 + CTD_ONE_KNOW6 + 80)
#define CTD_ONE_WINNER_OFF (CTD_ONE_COUNT_OFF + 4)
#define CTD_ONE_OPTS_OFF (CTD_ONE_COUNT_OFF + 8)
#define CTD_ONE_BYTES (CTD_ONE_OPTS_OFF + CTD_ONE_OPTS * 8)
// a block of the staging buffer (offset, bytes) and the host memory it is copied from or to (null: not copied)
struct CtdOneCopy {
  const void* host;
  size_t off, bytes;
};
// one ctd_k_one op on the staging buffer: upload `up`, run `a` (its op fields set by the caller; know: with the knowledge
// block), download `down`, synchronise
static ctd_status ctd_game_op(ctd_engine* e, CtdOneArgs a, bool know, std::initializer_list<CtdOneCopy> up,
                              std::initializer_list<CtdOneCopy> down) {
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, e->d_one.grow(CTD_ONE_BYTES));
  uint8_t* one = e->d_one;
  for (const CtdOneCopy& c : up)
    if (c.host) CTD_CUDA(e, cudaMemcpyAsync(one + c.off, c.host, c.bytes, cudaMemcpyHostToDevice, e->stream));
  a.state = (ctd_state*)one;
  a.know6 = know ? (CtdKnow*)(one + CTD_ONE_KNOW_OFF) : nullptr;
  a.used_cards = one + CTD_ONE_USED_OFF;
  a.count = (uint32_t*)(one + CTD_ONE_COUNT_OFF);
  a.winner = (int8_t*)(one + CTD_ONE_WINNER_OFF);
  a.opts = (ctd_option*)(one + CTD_ONE_OPTS_OFF);
  ctd_k_one<<<1, 32, 0, e->stream>>>(a);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  for (const CtdOneCopy& c : down)
    if (c.host) CTD_CUDA(e, cudaMemcpyAsync((void*)c.host, one + c.off, c.bytes, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_game_new(ctd_engine* e, uint64_t seed, uint64_t gid, int ruleset, ctd_state* state, void* know6, uint8_t* used_cards) {
  if (!e || !state || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  CtdOneArgs a{};
  a.op = 0; a.seed = seed; a.gid = gid; a.ruleset = ruleset;
  return ctd_game_op(e, a, true, {},
                     {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}, {used_cards, CTD_ONE_USED_OFF, 76}});
}

ctd_status ctd_game_options(ctd_engine* e, uint64_t seed, ctd_state* state, const void* know6, ctd_option* opts, uint32_t cap,
                            uint32_t* count) {
  if (!e || !state || !opts || !count) return CTD_EARG;
  CtdOneArgs a{};
  a.op = 1; a.seed = seed;
  a.cap = cap < CTD_ONE_OPTS ? cap : CTD_ONE_OPTS;   // a list the caller cannot take leaves the record untouched
  ctd_status s = ctd_game_op(e, a, know6 != nullptr, {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}},
                             {{count, CTD_ONE_COUNT_OFF, sizeof(uint32_t)}, {state, 0, sizeof(ctd_state)}});
  if (s != CTD_OK) return s;
  uint32_t n = *count < cap ? *count : cap;
  if (n > CTD_ONE_OPTS) n = CTD_ONE_OPTS;
  CTD_CUDA(e, cudaMemcpyAsync(opts, e->d_one + CTD_ONE_OPTS_OFF, (size_t)n * sizeof(ctd_option), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return *count > cap || *count > CTD_ONE_OPTS ? CTD_ECAP : CTD_OK;
}

ctd_status ctd_game_step(ctd_engine* e, uint64_t seed, ctd_state* state, void* know6, ctd_option chosen, int8_t* winner) {
  if (!e || !state || !winner) return CTD_EARG;
  CtdOneArgs a{};
  a.op = 2; a.seed = seed; a.chosen = chosen;
  return ctd_game_op(e, a, know6 != nullptr, {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}},
                     {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}, {winner, CTD_ONE_WINNER_OFF, 1}});
}

ctd_status ctd_game_sample(ctd_engine* e, uint64_t seed, ctd_state* state, void* know6, const uint8_t* used_cards, int viewer,
                           int role_sample) {
  if (!e || !state || !know6 || !used_cards || viewer < 0 || viewer > 5) return CTD_EARG;
  CtdOneArgs a{};
  a.op = 3; a.seed = seed; a.viewer = viewer; a.role_sample = role_sample;
  return ctd_game_op(e, a, true,
                     {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}, {used_cards, CTD_ONE_USED_OFF, 76}},
                     {{state, 0, sizeof(ctd_state)}, {know6, CTD_ONE_KNOW_OFF, CTD_ONE_KNOW6}});
}

// CFRNode.get_all_targets over the trees of the last ctd_mccfr / ctd_mccfr_pred call (they stay on the device).
// Call once with all output pointers NULL to size the buffers (*n_records, *n_option_slots), then again to fill.
ctd_status ctd_mccfr_targets(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, int ruleset, double threshold,
                             uint32_t* n_records, uint32_t* n_option_slots, float* features, ctd_target_meta* meta,
                             ctd_option* options, double* regrets) {
  if (!e || !n_records || !n_option_slots || n_roots > e->trees_n || !e->d_hdrs) return CTD_EARG;
  (void)iterations; (void)ruleset;   // the trees on the device know their own shape
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_pred_buffers(e);
  if (s != CTD_OK) return s;
  // counts
  size_t cb = (size_t)n_roots * sizeof(uint32_t);
  CtdBuf<uint32_t> d_cnt;
  CTD_CUDA(e, d_cnt.grow(4 * cb));
  CtdTargetArgs a;
  memset(&a, 0, sizeof(a));
  a.n_roots = n_roots; a.hdrs = e->d_hdrs; a.seed = seed;
  a.threshold = threshold; a.n_targets = d_cnt; a.n_options = d_cnt + n_roots;
  ctd_k_targets<<<ctd_blocks(n_roots), CTD_BLOCK, 0, e->stream>>>(a);
  e->launches++;
  std::unique_ptr<uint32_t[]> h_cnt(new (std::nothrow) uint32_t[4 * (size_t)n_roots]);
  if (!h_cnt) return CTD_ENOMEM;
  CTD_CUDA(e, cudaMemcpyAsync(h_cnt.get(), d_cnt, 2 * cb, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  uint32_t nrec = 0, nopt = 0;
  for (uint32_t t = 0; t < n_roots; ++t) {
    h_cnt[2 * n_roots + t] = nrec; h_cnt[3 * n_roots + t] = nopt;
    nrec += h_cnt[t]; nopt += h_cnt[n_roots + t];
  }
  const bool fill = features && meta && options && regrets;
  if (fill && (nrec > *n_records || nopt > *n_option_slots)) return CTD_ECAP;
  *n_records = nrec; *n_option_slots = nopt;
  if (!fill || nrec == 0) return CTD_OK;
  CtdBuf<float> d_feat;
  CtdBuf<ctd_target_meta> d_meta;
  CtdBuf<ctd_option> d_opt;
  CtdBuf<double> d_reg;
  CTD_CUDA(e, cudaMemcpyAsync(d_cnt + 2 * n_roots, h_cnt.get() + 2 * n_roots, 2 * cb, cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, d_feat.grow((size_t)nrec * CTD_FEATURES_PAD * sizeof(float)));
  CTD_CUDA(e, d_meta.grow((size_t)nrec * sizeof(ctd_target_meta)));
  CTD_CUDA(e, d_opt.grow((size_t)(nopt + 1) * sizeof(ctd_option)));
  CTD_CUDA(e, d_reg.grow((size_t)(nopt + 1) * sizeof(double)));
  a.fill = 1; a.rec_off = d_cnt + 2 * n_roots; a.opt_off = d_cnt + 3 * n_roots;
  a.feat = d_feat; a.meta = d_meta; a.options = d_opt; a.regrets = d_reg;
  ctd_k_targets<<<ctd_blocks(n_roots), CTD_BLOCK, 0, e->stream>>>(a);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaMemcpyAsync(features, d_feat, (size_t)nrec * CTD_FEATURES_PAD * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(meta, d_meta, (size_t)nrec * sizeof(ctd_target_meta), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(options, d_opt, (size_t)nopt * sizeof(ctd_option), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(regrets, d_reg, (size_t)nopt * sizeof(double), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// d_feat stands for the whole group, as d_knows does for the root buffers (ctd_root_buffers)
static ctd_status ctd_pred_buffers(ctd_engine* e) {
  if (e->d_feat) return CTD_OK;
  const size_t n = e->capacity;
  CtdBuf<float> feat;
  CTD_CUDA(e, feat.grow(n * CTD_FEATURES_PAD * sizeof(float)));
  CTD_CUDA(e, e->d_pred.grow(n * 8 * sizeof(float)));
  CTD_CUDA(e, e->d_pending.grow(n));
  CTD_CUDA(e, e->d_n_pending.grow(2 * sizeof(uint32_t)));
  CTD_CUDA(e, e->h_np.grow(4 * sizeof(uint32_t)));
  CTD_CUDA(e, cudaMemsetAsync(feat, 0, n * CTD_FEATURES_PAD * sizeof(float), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(e->d_pred, 0, n * 8 * sizeof(float), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(e->d_pending, 0, n, e->stream));
  CTD_CUDA(e, cudaFuncSetAttribute(ctd_k_value_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CTD_MLP_SMEM));
  CTD_CUDA(e, cudaFuncSetAttribute(ctd_k_linear_tc_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CTD_TC_SMEM));
  CTD_CUDA(e, e->d_h1.grow(n * 512 * sizeof(float)));
  CTD_CUDA(e, e->d_h2.grow(n * 256 * sizeof(float)));
  CTD_CUDA(e, e->d_h3.grow(n * 128 * sizeof(float)));
  CTD_CUDA(e, e->d_tc_err.grow(sizeof(int)));   // ctd_train_begin may have made it already
  CTD_CUDA(e, cudaMemsetAsync(e->d_tc_err, 0, sizeof(int), e->stream));
  e->d_feat = std::move(feat);
  return CTD_OK;
}

// the value model `vm` on rows [row0, row0 + n) of d_feat -> d_pred (`pending` is the mask of those rows; rows with pending == 0
// may be skipped), on `st`
static ctd_status ctd_value_forward(ctd_engine* e, const CtdValueSlot& vm, uint32_t n, const uint8_t* pending, float weight, uint32_t row0,
                                    cudaStream_t st) {
  if (st == nullptr) st = e->stream;
  const float* feat = e->d_feat + (size_t)row0 * CTD_FEATURES_PAD;
  float* pred = e->d_pred + (size_t)row0 * 8;
  const CtdValueModel& m = vm.model;
  if (e->value_backend == 0) {
    ctd_k_value_mlp<<<(n + CTD_MLP_ROWS - 1) / CTD_MLP_ROWS, 256, CTD_MLP_SMEM, st>>>(feat, pending, n, m, pred, weight);
    e->launches++;
    CTD_CUDA(e, cudaGetLastError());
    return CTD_OK;
  }
  float *h1 = e->d_h1 + (size_t)row0 * 512, *h2 = e->d_h2 + (size_t)row0 * 256, *h3 = e->d_h3 + (size_t)row0 * 128;
  const int M = (int)n, gm = (M + CTD_TC_BM - 1) / CTD_TC_BM;
  // weight operand by TMA from the pre-split terms
  ctd_k_linear_tc_tma<<<dim3(gm, 512 / CTD_TC_BN), 128, CTD_TC_SMEM, st>>>(feat, CTD_FEATURES_PAD, vm.tmap[0], m.b1, h1, 512, M, CTD_FEATURES_PAD, 1, e->d_tc_err);
  ctd_k_linear_tc_tma<<<dim3(gm, 256 / CTD_TC_BN), 128, CTD_TC_SMEM, st>>>(h1, 512, vm.tmap[1], m.b2, h2, 256, M, 512, 1, e->d_tc_err);
  ctd_k_linear_tc_tma<<<dim3(gm, 128 / CTD_TC_BN), 128, CTD_TC_SMEM, st>>>(h2, 256, vm.tmap[2], m.b3, h3, 128, M, 256, 1, e->d_tc_err);
  ctd_k_value_head<<<(n + 127) / 128, 128, 0, st>>>(h3, m.w4t, m.b4, pending, n, pred, weight);
  e->launches += 4;
  CTD_CUDA(e, cudaGetLastError());
  return CTD_OK;
}

// 3-D tensor map (K, N, term) over a [3][N][K] fp32 tensor, box = 16 bytes of K x 128 rows x one term, no swizzle.  The encoder
// lives in the driver (cuTensorMapEncodeTiled): fetched through the runtime, so the library does not link libcuda.
typedef CUresult (*ctd_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static bool ctd_make_weight_map(CUtensorMap* map, float* base, int N, int K) {
  static ctd_encode_tiled_fn encode = nullptr;
  if (!encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
      (void)cudaGetLastError();
      return false;
    }
    encode = (ctd_encode_tiled_fn)fn;
  }
  const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)N, 3};
  const cuuint64_t strides[2] = {(cuuint64_t)K * 4, (cuuint64_t)N * K * 4};
  const cuuint32_t box[3] = {4, 128, 1}, estr[3] = {1, 1, 1};
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

ctd_status ctd_set_value_backend(ctd_engine* e, int backend) {
  if (!e || backend < 0 || backend > 2) return CTD_EARG;
  e->fused = backend == 2;
  e->value_backend = backend == 0 ? 0 : 1;
  return CTD_OK;
}

ctd_status ctd_set_value_model_slot(ctd_engine* e, int slot, const float* w1t, const float* b1, const float* w2t, const float* b2,
                                    const float* w3t, const float* b3, const float* w4t, const float* b4) {
  if (!e || slot < 0 || slot >= CTD_MAX_VALUE_MODELS || !w1t || !b1 || !w2t || !b2 || !w3t || !b3 || !w4t || !b4) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdValueSlot& v = e->vm[slot];
  v.ready = false;   // until the whole load below has completed
  const size_t n1 = (size_t)CTD_FEATURES_PAD * 512, n2 = 512 * 256, n3 = 256 * 128, n4 = 128 * 6 + 2;
  const size_t total = n1 + 512 + n2 + 256 + n3 + 128 + n4 + 8;
  CTD_CUDA(e, v.d_model.grow(total * sizeof(float)));
  float* p = v.d_model;
  CtdValueModel& m = v.model;
  const float* src[8] = {w1t, b1, w2t, b2, w3t, b3, w4t, b4};
  const size_t cnt[8] = {n1, 512, n2, 256, n3, 128, 128 * 6, 6};
  const size_t pad[8] = {n1, 512, n2, 256, n3, 128, n4, 8};
  const float** dst[8] = {&m.w1t, &m.b1, &m.w2t, &m.b2, &m.w3t, &m.b3, &m.w4t, &m.b4};
  for (int i = 0; i < 8; ++i) {
    CTD_CUDA(e, cudaMemcpyAsync(p, src[i], cnt[i] * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    *dst[i] = p;
    p += pad[i];
  }
  {  // tensor-core layout: the static weights split into their TF32 terms once, and described to the TMA engine
    const size_t t1 = (size_t)512 * CTD_FEATURES_PAD, t2 = (size_t)256 * 512, t3 = (size_t)128 * 256;
    CTD_CUDA(e, v.d_wsplit.grow(3 * (t1 + t2 + t3) * sizeof(float)));
    float* sp[3] = {v.d_wsplit, v.d_wsplit + 3 * t1, v.d_wsplit + 3 * (t1 + t2)};
    const size_t cnt[3] = {t1, t2, t3};
    const int Ns[3] = {512, 256, 128}, Ks[3] = {CTD_FEATURES_PAD, 512, 256};
    for (int l = 0; l < 3; ++l)
      if (!ctd_make_weight_map(&v.tmap[l], sp[l], Ns[l], Ks[l])) {
        snprintf(e->err, sizeof(e->err), "ctd_set_value_model: cannot build the TMA tensor maps of the weights (cuTensorMapEncodeTiled)");
        return CTD_ECUDA;
      }
    // the split's source: [out][in] (the reference's own nn.Linear layout), BN already folded
    std::unique_ptr<float[]> h(new (std::nothrow) float[t1 + t2 + t3]);
    if (!h) return CTD_ENOMEM;
    for (int o = 0; o < 512; ++o) for (int k = 0; k < CTD_FEATURES_PAD; ++k) h[(size_t)o * CTD_FEATURES_PAD + k] = w1t[(size_t)k * 512 + o];
    for (int o = 0; o < 256; ++o) for (int k = 0; k < 512; ++k) h[t1 + (size_t)o * 512 + k] = w2t[(size_t)k * 256 + o];
    for (int o = 0; o < 128; ++o) for (int k = 0; k < 256; ++k) h[t1 + t2 + (size_t)o * 256 + k] = w3t[(size_t)k * 128 + o];
    CtdBuf<float> d_oi;
    CTD_CUDA(e, d_oi.grow((t1 + t2 + t3) * sizeof(float)));
    CTD_CUDA(e, cudaMemcpy(d_oi, h.get(), (t1 + t2 + t3) * sizeof(float), cudaMemcpyHostToDevice));
    const float* src[3] = {d_oi, d_oi + t1, d_oi + t1 + t2};
    for (int l = 0; l < 3; ++l) {
      ctd_k_split3<<<(unsigned)((cnt[l] + 255) / 256), 256, 0, e->stream>>>(src[l], sp[l], cnt[l]);
      e->launches++;
    }
    CTD_CUDA(e, cudaGetLastError());
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));   // the split has read d_oi before it is freed
  }
  v.ready = true;
  return CTD_OK;
}

ctd_status ctd_set_value_model(ctd_engine* e, const float* w1t, const float* b1, const float* w2t, const float* b2,
                               const float* w3t, const float* b3, const float* w4t, const float* b4) {
  return ctd_set_value_model_slot(e, 0, w1t, b1, w2t, b2, w3t, b3, w4t, b4);
}

ctd_status ctd_value_eval(ctd_engine* e, uint32_t n, const float* features, float weight, float* out6) {
  if (!e || !features || !out6 || n > e->capacity || !e->vm[0].ready) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_pred_buffers(e);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaMemcpyAsync(e->d_feat, features, (size_t)n * CTD_FEATURES_PAD * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  s = ctd_value_forward(e, e->vm[0], n, nullptr, weight, 0, nullptr);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaMemcpy2DAsync(out6, 6 * sizeof(float), e->d_pred, 8 * sizeof(float), 6 * sizeof(float), n, cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (e->value_backend == 1) {
    int terr = 0;
    CTD_CUDA(e, cudaMemcpy(&terr, e->d_tc_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (terr) { snprintf(e->err, sizeof(e->err), "tcgen05 value kernel: mbarrier wait timed out"); return CTD_ECUDA; }
  }
  return CTD_OK;
}

ctd_status ctd_encode(ctd_engine* e, uint32_t n, int cfr_role_pick, float* features) {
  if (!e || !features || n > e->capacity || !e->d_knows) return CTD_EARG;
  if (n == 0) return CTD_OK;
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_pred_buffers(e);
  if (s != CTD_OK) return s;
  ctd_k_encode<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(e->d_slots, e->d_knows, n, e->d_feat, cfr_role_pick);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaMemcpyAsync(features, e->d_feat, (size_t)n * CTD_FEATURES_PAD * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_mccfr_pred(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, uint32_t max_depth, int ruleset,
                          float reward_weight, ctd_mccfr_result* results, float* elapsed_ms, uint32_t* waves_out) {
  if (!e || n_roots > e->capacity || !e->d_knows || !e->vm[0].ready || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM)) return CTD_EARG;
  if (n_roots == 0) return CTD_OK;
  CtdSearch sp{n_roots, seed, iterations, ruleset, true, max_depth, reward_weight, false, 0};
  return ctd_search(e, sp, results, elapsed_ms, waves_out);
}

// ------------------------------------------------------------------------------------------ arena (ctd_arena.cuh)
// Record the trees of one arena search (roots [0, cnt), game list[t]), still in e->d_hdrs -- ctd_search leaves every tree there
// from its final pass, retried trees included.  Three launches between the event pair: count, reserve rows on the device, fill.
// rcnt: 4 * capacity words.  Nothing is waited for.
static ctd_status ctd_record_search(ctd_engine* e, const ctd_record_opts& rec, const CtdArenaGame* games, const uint32_t* list, uint32_t cnt,
                                    uint64_t seed, uint32_t* rcnt, cudaEvent_t ev0, cudaEvent_t ev1) {
  CtdTargetArgs a;
  memset(&a, 0, sizeof(a));
  a.n_roots = cnt; a.hdrs = e->d_hdrs; a.seed = seed; a.threshold = rec.threshold;
  a.n_targets = rcnt; a.n_options = rcnt + e->capacity; a.rec_off = rcnt + 2 * e->capacity; a.opt_off = rcnt + 3 * e->capacity;
  a.games = games; a.list = list; a.seat_mask = rec.seat_mask; a.root_only = rec.mode == CTD_RECORD_ROOT;
  a.feat = e->ds_feat; a.meta = e->ds_meta; a.options = e->ds_opt; a.regrets = e->ds_reg; a.origin = e->ds_origin;
  CTD_CUDA(e, cudaEventRecord(ev0, e->stream));
  ctd_k_record_targets<<<ctd_blocks(cnt), CTD_BLOCK, 0, e->stream>>>(a);
  ctd_k_record_reserve<<<1, CTD_RESERVE_THREADS, 0, e->stream>>>(cnt, a.n_targets, a.n_options, rcnt + 2 * e->capacity, rcnt + 3 * e->capacity,
                                                                  e->ds_ctr, e->ds_max_records, e->ds_max_slots);
  a.fill = 1;
  ctd_k_record_targets<<<ctd_blocks(cnt), CTD_BLOCK, 0, e->stream>>>(a);
  e->launches += 3;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaEventRecord(ev1, e->stream));
  return CTD_OK;
}

// the phase-timing events of one ctd_arena call, destroyed on every way out (ev[4], ev[5]: recording only)
struct CtdArenaEvents {
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  ~CtdArenaEvents() {
    for (cudaEvent_t v : ev) if (v) cudaEventDestroy(v);
  }
};

// ctd_arena, and with `rec` ctd_arena_record: elapsed_ms then takes a fourth time, the recording's
static ctd_status ctd_arena_run(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset, const ctd_arena_seat seats[6],
                                uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps, uint32_t* searches,
                                ctd_playout_stats* stats, const ctd_record_opts* rec, float* elapsed_ms) {
  // max_steps: the record's steps field saturates at 65535, a larger limit would never be reached
  if (!e || !seats || n_games > 0xFFFFFFFFull || max_steps > 65535u || (ruleset < CTD_RULESET_PRESET || ruleset > CTD_RULESET_RANDOM))
    return CTD_EARG;
  CtdArenaArgs a;
  memset(&a, 0, sizeof(a));
  // seats with the same player (kind, value-model slot included, and parameters) share a search group: one batch of roots per
  // group and decision round
  CtdSearch groups[6];
  int n_groups = 0;
  for (int s = 0; s < 6; ++s) {
    const ctd_arena_seat& p = seats[s];
    a.seat_group[s] = -1;
    const uint32_t kind = (uint32_t)p.kind & 0xFFu, slot = ((uint32_t)p.kind >> 8) & 0xFFu;   // CTD_SEAT_DEEP_MODEL(slot)
    if (((uint32_t)p.kind >> 16) != 0 || (slot != 0 && kind != CTD_SEAT_DEEP)) return CTD_EARG;
    if (kind == CTD_SEAT_RANDOM) continue;
    if ((kind != CTD_SEAT_PURE && kind != CTD_SEAT_DEEP) || p.iterations == 0 ||
        (kind == CTD_SEAT_DEEP && (slot >= CTD_MAX_VALUE_MODELS || !e->vm[slot].ready)))
      return CTD_EARG;
    for (int t = 0; t < s && a.seat_group[s] < 0; ++t)
      if (a.seat_group[t] >= 0 && seats[t].kind == p.kind && seats[t].iterations == p.iterations && seats[t].max_depth == p.max_depth &&
          seats[t].reward_weight == p.reward_weight)
        a.seat_group[s] = a.seat_group[t];
    if (a.seat_group[s] < 0) {
      groups[n_groups] = CtdSearch{0, seed, p.iterations, ruleset, kind == CTD_SEAT_DEEP, p.max_depth, p.reward_weight, false, (int)slot};
      a.seat_group[s] = (int8_t)n_groups++;
    }
  }
  // a group is recorded when one of its seats is in the mask
  bool recorded[6] = {false, false, false, false, false, false};
  if (rec)
    for (int s = 0; s < 6; ++s)
      if (a.seat_group[s] >= 0 && ((rec->seat_mask >> s) & 1)) recorded[a.seat_group[s]] = true;
  float ms[4] = {0.f, 0.f, 0.f, 0.f};
  const size_t ms_bytes = (rec ? 4 : 3) * sizeof(float);
  if (n_games == 0) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (elapsed_ms) memcpy(elapsed_ms, ms, ms_bytes);
    return CTD_OK;
  }
  const uint32_t n = (uint32_t)n_games;
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_status s = ctd_root_buffers(e);
  if (s != CTD_OK) return s;
  CtdBuf<CtdArenaGame> games;
  CtdBuf<uint32_t> queue;
  CtdBuf<int8_t> out;
  CtdArenaEvents run;
  const size_t wb = ((size_t)n + 255) & ~(size_t)255, pb = ((size_t)n * 6 + 255) & ~(size_t)255, sb = ((size_t)n * 2 + 255) & ~(size_t)255,
               cb = (size_t)n * 4;
  CTD_CUDA(e, games.grow((size_t)n * sizeof(CtdArenaGame)));
  CTD_CUDA(e, queue.grow(256 + (size_t)n_groups * n * sizeof(uint32_t)));
  CTD_CUDA(e, out.grow(wb + pb + sb + ((cb + 255) & ~(size_t)255) + sizeof(ctd_playout_stats)));
  for (int k = 0; k < (rec ? 6 : 4); ++k) CTD_CUDA(e, cudaEventCreate(&run.ev[k]));
  CtdBuf<uint32_t> rcnt;   // recording: per tree of a search, records, option slots, first row, first slot
  if (rec) CTD_CUDA(e, rcnt.grow((size_t)4 * e->capacity * sizeof(uint32_t)));
  int8_t* d_winner = out;
  int8_t* d_points = d_winner + wb;
  uint16_t* d_steps = (uint16_t*)(d_winner + wb + pb);
  uint32_t* d_searches = (uint32_t*)(d_winner + wb + pb + sb);
  ctd_playout_stats* d_stats = (ctd_playout_stats*)(d_winner + wb + pb + sb + ((cb + 255) & ~(size_t)255));
  a.n = n; a.seed = seed; a.first_gid = first_gid; a.ruleset = ruleset; a.max_steps = max_steps;
  a.games = games;
  a.queued = queue;
  a.queue = a.queued + 64;
  e->slots_rs_n = 0;
  // Phase times.  The advance and the search phases end where the host waits anyway (the queue counts, the search's own
  // read-backs); an apply launch is not waited for: its event pair (ev[2], ev[3]) is read at the next of those waits.
  // The recording's pair (ev[4], ev[5]) is read the same way.
  bool apply_pending = false, record_pending = false;
  auto timed = [&](int phase) -> ctd_status {
    CTD_CUDA(e, cudaEventRecord(run.ev[1], e->stream));
    CTD_CUDA(e, cudaEventSynchronize(run.ev[1]));
    float t = 0.f;
    CTD_CUDA(e, cudaEventElapsedTime(&t, run.ev[0], run.ev[1]));
    ms[phase] += t;
    if (apply_pending) {
      CTD_CUDA(e, cudaEventElapsedTime(&t, run.ev[2], run.ev[3]));
      ms[2] += t;
      apply_pending = false;
    }
    if (record_pending) {
      CTD_CUDA(e, cudaEventElapsedTime(&t, run.ev[4], run.ev[5]));
      ms[3] += t;
      record_pending = false;
    }
    return CTD_OK;
  };
  CTD_CUDA(e, cudaEventRecord(run.ev[0], e->stream));
  ctd_k_arena_deal<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(a);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  if (rec)   // this call's records start where the dataset stands now
    CTD_CUDA(e, cudaMemcpyAsync(&e->ds_ctr.get()->call_first, &e->ds_ctr.get()->n_records, sizeof(unsigned long long),
                                cudaMemcpyDeviceToDevice, e->stream));
  uint32_t queued[6];
  for (;;) {   // one decision round: every live game plays on to its next search (or its end), then each group searches
    CTD_CUDA(e, cudaMemsetAsync(a.queued, 0, sizeof(queued), e->stream));
    ctd_k_arena_advance<<<ctd_blocks(n), CTD_BLOCK, 0, e->stream>>>(a);
    e->launches++;
    CTD_CUDA(e, cudaGetLastError());
    CTD_CUDA(e, cudaMemcpyAsync(queued, a.queued, sizeof(queued), cudaMemcpyDeviceToHost, e->stream));
    if ((s = timed(0)) != CTD_OK) return s;
    uint32_t total = 0;
    for (int g = 0; g < n_groups; ++g) total += queued[g];
    if (total == 0) break;
    for (int g = 0; g < n_groups; ++g) {
      for (uint32_t first = 0; first < queued[g]; first += e->capacity) {   // roots go through the engine's slots, capacity at a time
        const uint32_t cnt = queued[g] - first < e->capacity ? queued[g] - first : e->capacity;
        const uint32_t* list = a.queue + (size_t)g * n + first;
        CTD_CUDA(e, cudaEventRecord(run.ev[0], e->stream));
        ctd_k_arena_gather<<<ctd_blocks(cnt), CTD_BLOCK, 0, e->stream>>>(a.games, list, cnt, e->d_slots, e->d_knows, e->d_used_cards, e->d_gids);
        e->launches++;
        CTD_CUDA(e, cudaGetLastError());
        CtdSearch sp = groups[g];
        sp.n_roots = cnt;
        if ((s = ctd_search(e, sp, nullptr, nullptr, nullptr)) != CTD_OK) return s;   // results stay in d_results
        if ((s = timed(1)) != CTD_OK) return s;
        if (recorded[g]) {   // the trees of this search, before its decisions are applied (the games still stand at the roots)
          if ((s = ctd_record_search(e, *rec, a.games, list, cnt, seed, rcnt, run.ev[4], run.ev[5])) != CTD_OK) return s;
          record_pending = true;
        }
        CTD_CUDA(e, cudaEventRecord(run.ev[2], e->stream));
        ctd_k_arena_apply<<<ctd_blocks(cnt), CTD_BLOCK, 0, e->stream>>>(a, list, cnt, e->d_results);
        e->launches++;
        CTD_CUDA(e, cudaGetLastError());
        CTD_CUDA(e, cudaEventRecord(run.ev[3], e->stream));
        apply_pending = true;
      }
    }
    CTD_CUDA(e, cudaEventRecord(run.ev[0], e->stream));
  }
  CTD_CUDA(e, cudaEventRecord(run.ev[0], e->stream));
  CTD_CUDA(e, cudaMemsetAsync(d_stats, 0, sizeof(ctd_playout_stats), e->stream));
  ctd_k_arena_finish<<<(n + 255) / 256, 256, 0, e->stream>>>(a.games, n, d_winner, d_points, d_steps, d_searches, d_stats);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  CTD_CUDA(e, cudaEventRecord(run.ev[1], e->stream));
  if (rec) {   // every game is over: the outcome of each record this call appended
    CTD_CUDA(e, cudaEventRecord(run.ev[4], e->stream));
    ctd_k_record_outcome<<<(unsigned)e->sm_count * 4, 256, 0, e->stream>>>(a.games, e->ds_meta, e->ds_origin, e->ds_ctr);
    e->launches++;
    CTD_CUDA(e, cudaGetLastError());
    CTD_CUDA(e, cudaEventRecord(run.ev[5], e->stream));
  }
  // the final records of the first games stay readable through ctd_store_states
  const uint32_t keep = n < e->capacity ? n : e->capacity;
  CTD_CUDA(e, cudaMemcpy2DAsync(e->d_slots, sizeof(ctd_state), &a.games[0].rec, sizeof(CtdArenaGame), sizeof(ctd_state), keep,
                                cudaMemcpyDeviceToDevice, e->stream));
  if (winner) CTD_CUDA(e, cudaMemcpyAsync(winner, d_winner, n, cudaMemcpyDeviceToHost, e->stream));
  if (points6) CTD_CUDA(e, cudaMemcpyAsync(points6, d_points, (size_t)n * 6, cudaMemcpyDeviceToHost, e->stream));
  if (steps) CTD_CUDA(e, cudaMemcpyAsync(steps, d_steps, (size_t)n * 2, cudaMemcpyDeviceToHost, e->stream));
  if (searches) CTD_CUDA(e, cudaMemcpyAsync(searches, d_searches, cb, cudaMemcpyDeviceToHost, e->stream));
  if (stats) CTD_CUDA(e, cudaMemcpyAsync(stats, d_stats, sizeof(ctd_playout_stats), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  float t = 0.f;
  CTD_CUDA(e, cudaEventElapsedTime(&t, run.ev[0], run.ev[1]));   // the final kernel
  ms[0] += t;
  if (rec) {
    CTD_CUDA(e, cudaEventElapsedTime(&t, run.ev[4], run.ev[5]));
    ms[3] += t;
  }
  if (elapsed_ms) memcpy(elapsed_ms, ms, ms_bytes);
  return CTD_OK;
}

ctd_status ctd_arena(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset, const ctd_arena_seat seats[6],
                     uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps, uint32_t* searches,
                     ctd_playout_stats* stats, float* elapsed_ms) {
  return ctd_arena_run(e, n_games, seed, first_gid, ruleset, seats, max_steps, winner, points6, steps, searches, stats, nullptr, elapsed_ms);
}

ctd_status ctd_arena_record(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset, const ctd_arena_seat seats[6],
                            uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps, uint32_t* searches,
                            ctd_playout_stats* stats, const ctd_record_opts* rec, float* elapsed_ms) {
  if (!e || !rec || (rec->seat_mask >> 6) != 0 || (rec->mode != CTD_RECORD_TREE && rec->mode != CTD_RECORD_ROOT) ||
      !(rec->threshold >= 0.0) || e->ds_max_records == 0)
    return CTD_EARG;
  return ctd_arena_run(e, n_games, seed, first_gid, ruleset, seats, max_steps, winner, points6, steps, searches, stats, rec, elapsed_ms);
}

// ------------------------------------------------------------------------------------------ self-play dataset
ctd_status ctd_dataset_reserve(ctd_engine* e, uint32_t max_records, uint32_t max_option_slots) {
  if (!e || max_records == 0 || max_option_slots == 0) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));   // no recording may still write into the old buffers
  e->ds_max_records = e->ds_max_slots = 0;         // not reserved until every buffer exists
  CTD_CUDA(e, e->ds_feat.grow((size_t)max_records * CTD_FEATURES_PAD * sizeof(float)));
  CTD_CUDA(e, e->ds_meta.grow((size_t)max_records * sizeof(ctd_target_meta)));
  CTD_CUDA(e, e->ds_origin.grow((size_t)max_records * sizeof(ctd_record_origin)));
  CTD_CUDA(e, e->ds_opt.grow((size_t)max_option_slots * sizeof(ctd_option)));
  CTD_CUDA(e, e->ds_reg.grow((size_t)max_option_slots * sizeof(double)));
  CTD_CUDA(e, e->ds_ctr.grow(sizeof(CtdDatasetCtr)));
  CTD_CUDA(e, cudaMemsetAsync(e->ds_ctr, 0, sizeof(CtdDatasetCtr), e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  e->ds_max_records = max_records; e->ds_max_slots = max_option_slots;
  return CTD_OK;
}

ctd_status ctd_dataset_clear(ctd_engine* e) {
  if (!e || e->ds_max_records == 0) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, cudaMemsetAsync(e->ds_ctr, 0, sizeof(CtdDatasetCtr), e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

static ctd_status ctd_dataset_counts(ctd_engine* e, CtdDatasetCtr* c) {
  if (!e || e->ds_max_records == 0) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CTD_CUDA(e, cudaMemcpyAsync(c, e->ds_ctr, sizeof(CtdDatasetCtr), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_dataset_info(ctd_engine* e, uint32_t* n_records, uint32_t* n_option_slots, uint64_t* dropped_trees, uint64_t* dropped_records) {
  CtdDatasetCtr c;
  const ctd_status s = ctd_dataset_counts(e, &c);
  if (s != CTD_OK) return s;
  if (n_records) *n_records = (uint32_t)c.n_records;
  if (n_option_slots) *n_option_slots = (uint32_t)c.n_slots;
  if (dropped_trees) *dropped_trees = c.dropped_trees;
  if (dropped_records) *dropped_records = c.dropped_records;
  return CTD_OK;
}

ctd_status ctd_dataset_read(ctd_engine* e, uint32_t first, uint32_t n, float* features, ctd_target_meta* meta, ctd_record_origin* origin) {
  CtdDatasetCtr c;
  const ctd_status s = ctd_dataset_counts(e, &c);
  if (s != CTD_OK) return s;
  if ((uint64_t)first + n > c.n_records) return CTD_EARG;
  if (n == 0) return CTD_OK;
  // cudaMemcpyDefault: the outputs may be host memory or device memory on any GPU
  if (features) CTD_CUDA(e, cudaMemcpyAsync(features, e->ds_feat + (size_t)first * CTD_FEATURES_PAD, (size_t)n * CTD_FEATURES_PAD * sizeof(float),
                                            cudaMemcpyDefault, e->stream));
  if (meta) CTD_CUDA(e, cudaMemcpyAsync(meta, e->ds_meta + first, (size_t)n * sizeof(ctd_target_meta), cudaMemcpyDefault, e->stream));
  if (origin) CTD_CUDA(e, cudaMemcpyAsync(origin, e->ds_origin + first, (size_t)n * sizeof(ctd_record_origin), cudaMemcpyDefault, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

ctd_status ctd_dataset_read_options(ctd_engine* e, uint32_t first_slot, uint32_t n, ctd_option* options, double* regrets) {
  CtdDatasetCtr c;
  const ctd_status s = ctd_dataset_counts(e, &c);
  if (s != CTD_OK) return s;
  if ((uint64_t)first_slot + n > c.n_slots) return CTD_EARG;
  if (n == 0) return CTD_OK;
  if (options) CTD_CUDA(e, cudaMemcpyAsync(options, e->ds_opt + first_slot, (size_t)n * sizeof(ctd_option), cudaMemcpyDefault, e->stream));
  if (regrets) CTD_CUDA(e, cudaMemcpyAsync(regrets, e->ds_reg + first_slot, (size_t)n * sizeof(double), cudaMemcpyDefault, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// The incoming records are copied past the cursors, where no read reaches them, and ctd_k_dataset_append checks them, rebases their
// option offsets and only then moves the cursors: a rejected append leaves the dataset as it was.
ctd_status ctd_dataset_append(ctd_engine* e, uint32_t n_records, uint32_t n_option_slots, const float* features, const ctd_target_meta* meta,
                              const ctd_record_origin* origin, const ctd_option* options, const double* regrets) {
  if (!e || e->ds_max_records == 0 || (n_records && (!features || !meta || !origin)) || (n_option_slots && (!options || !regrets)))
    return CTD_EARG;
  if (n_records == 0 && n_option_slots == 0) return CTD_OK;
  CtdDatasetCtr c;
  ctd_status s = ctd_dataset_counts(e, &c);   // waits for every recording in flight
  if (s != CTD_OK) return s;
  if (c.n_records + n_records > e->ds_max_records || c.n_slots + n_option_slots > e->ds_max_slots) {
    snprintf(e->err, sizeof(e->err), "ctd_dataset_append: %llu + %u records / %llu + %u option slots exceed the reservation (%u / %u)",
             c.n_records, n_records, c.n_slots, n_option_slots, e->ds_max_records, e->ds_max_slots);
    return CTD_ECAP;
  }
  CtdBuf<int> d_bad;
  CTD_CUDA(e, d_bad.grow(sizeof(int)));
  if (n_records) {
    CTD_CUDA(e, cudaMemcpyAsync(e->ds_feat + (size_t)c.n_records * CTD_FEATURES_PAD, features, (size_t)n_records * CTD_FEATURES_PAD * sizeof(float),
                                cudaMemcpyDefault, e->stream));
    CTD_CUDA(e, cudaMemcpyAsync(e->ds_meta + c.n_records, meta, (size_t)n_records * sizeof(ctd_target_meta), cudaMemcpyDefault, e->stream));
    CTD_CUDA(e, cudaMemcpyAsync(e->ds_origin + c.n_records, origin, (size_t)n_records * sizeof(ctd_record_origin), cudaMemcpyDefault, e->stream));
  }
  if (n_option_slots) {
    CTD_CUDA(e, cudaMemcpyAsync(e->ds_opt + c.n_slots, options, (size_t)n_option_slots * sizeof(ctd_option), cudaMemcpyDefault, e->stream));
    CTD_CUDA(e, cudaMemcpyAsync(e->ds_reg + c.n_slots, regrets, (size_t)n_option_slots * sizeof(double), cudaMemcpyDefault, e->stream));
  }
  ctd_k_dataset_append<<<1, CTD_APPEND_THREADS, 0, e->stream>>>(e->ds_meta, e->ds_origin, e->ds_ctr, n_records, n_option_slots, d_bad);
  e->launches++;
  CTD_CUDA(e, cudaGetLastError());
  int bad = 0;
  CTD_CUDA(e, cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (bad) {
    snprintf(e->err, sizeof(e->err), "ctd_dataset_append: %s", bad & 1 ? "a record's option span is empty or outside the incoming slots"
                                                                : bad & 2 ? "an origin's mover is not a seat" : "an origin's winner is not -1 or a seat");
    return CTD_EARG;
  }
  return CTD_OK;
}


// ------------------------------------------------------------------------------------------ value-network training
void ctd_train_end(ctd_engine* e) {
  if (!e || !e->trainer) return;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  e->trainer.reset();
}

// a new trainer for n_train / n_val rows: every buffer allocated and zeroed (the previous trainer is gone)
static ctd_status ctd_train_alloc(ctd_engine* e, uint32_t n_train, uint32_t n_val, uint32_t batch_size, std::unique_ptr<CtdTrainer>& out) {
  CTD_CUDA(e, cudaSetDevice(e->device));
  ctd_train_end(e);
  std::unique_ptr<CtdTrainer> t(new (std::nothrow) CtdTrainer());
  if (!t) return CTD_ENOMEM;
  t->n_train = n_train; t->n_val = n_val; t->batch = batch_size; t->bp = (batch_size + 31) & ~31u;
  const size_t bp = t->bp;
  cudaError_t c = cudaSuccess;
  auto zeroed = [&](auto& buf, size_t count) {   // allocate and clear, until the first failure
    const size_t bytes = count * sizeof(*buf.get());
    if (c == cudaSuccess) c = buf.grow(bytes);
    if (c == cudaSuccess) c = cudaMemsetAsync(buf, 0, bytes, e->stream);
  };
  zeroed(t->feat_tr, (size_t)n_train * 418); zeroed(t->val_tr, (size_t)n_train * 6);
  zeroed(t->feat_va, (size_t)(n_val ? n_val : 1) * 418); zeroed(t->val_va, (size_t)(n_val ? n_val : 1) * 6);
  zeroed(t->perm, n_train);
  zeroed(t->P, CtdTrainLayout::total); zeroed(t->G, CtdTrainLayout::total); zeroed(t->M, CtdTrainLayout::total); zeroed(t->V, CtdTrainLayout::total);
  zeroed(t->rm1, CTD_TR_H1); zeroed(t->rv1, CTD_TR_H1); zeroed(t->rm2, CTD_TR_H2); zeroed(t->rv2, CTD_TR_H2);
  zeroed(t->X, bp * CTD_TR_IN); zeroed(t->XT, bp * CTD_TR_IN);
  zeroed(t->Z1, bp * CTD_TR_H1); zeroed(t->H1, bp * CTD_TR_H1); zeroed(t->H1T, bp * CTD_TR_H1);
  zeroed(t->Z2, bp * CTD_TR_H2); zeroed(t->H2, bp * CTD_TR_H2); zeroed(t->H2T, bp * CTD_TR_H2);
  zeroed(t->H3, bp * CTD_TR_H3); zeroed(t->dY, bp * 8); zeroed(t->dZ3, bp * CTD_TR_H3); zeroed(t->dZ3T, bp * CTD_TR_H3);
  zeroed(t->dH2, bp * CTD_TR_H2); zeroed(t->dZ2T, bp * CTD_TR_H2); zeroed(t->dH1, bp * CTD_TR_H1); zeroed(t->dZ1T, bp * CTD_TR_H1);
  zeroed(t->W2T, (size_t)CTD_TR_H1 * CTD_TR_H2); zeroed(t->W3T, (size_t)CTD_TR_H2 * CTD_TR_H3);
  zeroed(t->inv1, CTD_TR_H1); zeroed(t->inv2, CTD_TR_H2); zeroed(t->zero, 512);
  zeroed(t->T, bp * 6); zeroed(t->loss, 2);
  if (c != cudaSuccess) return ctd_fail(e, c, "training buffers");
  out = std::move(t);
  return CTD_OK;
}

// the rows are in place: the GEMM's set-up, then the trainer becomes the engine's
static ctd_status ctd_train_install(ctd_engine* e, std::unique_ptr<CtdTrainer>& t) {
  CTD_CUDA(e, cudaFuncSetAttribute(ctd_k_linear_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CTD_TC_SMEM));
  if (!e->d_tc_err) {
    CTD_CUDA(e, e->d_tc_err.grow(sizeof(int)));
    CTD_CUDA(e, cudaMemsetAsync(e->d_tc_err, 0, sizeof(int), e->stream));
  }
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  e->trainer = std::move(t);
  return CTD_OK;
}

ctd_status ctd_train_begin(ctd_engine* e, uint32_t n_train, const float* features, const double* node_values, uint32_t n_val,
                           const float* val_features, const double* val_node_values, uint32_t batch_size) {
  if (!e || !features || !node_values || n_train == 0 || batch_size == 0 || batch_size > 65536 || (n_val != 0 && (!val_features || !val_node_values)))
    return CTD_EARG;
  std::unique_ptr<CtdTrainer> t;
  ctd_status s = ctd_train_alloc(e, n_train, n_val, batch_size, t);
  if (s != CTD_OK) return s;
  CTD_CUDA(e, cudaMemcpyAsync(t->feat_tr, features, (size_t)n_train * 418 * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(t->val_tr, node_values, (size_t)n_train * 6 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
  if (n_val) {
    CTD_CUDA(e, cudaMemcpyAsync(t->feat_va, val_features, (size_t)n_val * 418 * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    CTD_CUDA(e, cudaMemcpyAsync(t->val_va, val_node_values, (size_t)n_val * 6 * sizeof(double), cudaMemcpyHostToDevice, e->stream));
  }
  return ctd_train_install(e, t);
}

// rows idx[0, n) of the dataset -> X [n][418] and labels V [n][6]; bad |= 1 for an index past the records, 2 for a winner label on
// an errored game.  One block per row.
__global__ void __launch_bounds__(128) ctd_k_dataset_rows(const float* feat, const ctd_target_meta* meta, const ctd_record_origin* origin,
                                                          const CtdDatasetCtr* ctr, const uint32_t* idx, uint32_t n, int label, float* X,
                                                          double* V, int* bad) {
  const uint32_t r = blockIdx.x;
  if (r >= n) return;
  const uint32_t i = idx[r];
  if (i >= ctr->n_records) {
    if (threadIdx.x == 0) atomicOr(bad, 1);
    return;
  }
  for (int c = threadIdx.x; c < 418; c += blockDim.x) X[(size_t)r * 418 + c] = feat[(size_t)i * CTD_FEATURES_PAD + c];
  if (threadIdx.x < 6) {
    double v = meta[i].node_value[threadIdx.x];
    if (label == CTD_LABEL_WINNER) {
      const int w = origin[i].winner;
      if (w < 0 && threadIdx.x == 0) atomicOr(bad, 2);
      v = (int)threadIdx.x == w ? 1.0 : 0.0;
    }
    V[(size_t)r * 6 + threadIdx.x] = v;
  }
}

ctd_status ctd_train_begin_dataset(ctd_engine* e, uint32_t n_train, const uint32_t* train_idx, uint32_t n_val, const uint32_t* val_idx,
                                   int label, uint32_t batch_size) {
  if (!e || !train_idx || n_train == 0 || batch_size == 0 || batch_size > 65536 || (n_val != 0 && !val_idx) || e->ds_max_records == 0 ||
      (label != CTD_LABEL_NODE_VALUE && label != CTD_LABEL_WINNER))
    return CTD_EARG;
  std::unique_ptr<CtdTrainer> t;
  ctd_status s = ctd_train_alloc(e, n_train, n_val, batch_size, t);
  if (s != CTD_OK) return s;
  CtdBuf<uint32_t> d_idx;
  CtdBuf<int> d_bad;
  CTD_CUDA(e, d_idx.grow(((size_t)n_train + n_val) * sizeof(uint32_t)));
  CTD_CUDA(e, d_bad.grow(sizeof(int)));
  CTD_CUDA(e, cudaMemsetAsync(d_bad, 0, sizeof(int), e->stream));
  CTD_CUDA(e, cudaMemcpyAsync(d_idx, train_idx, (size_t)n_train * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  if (n_val) CTD_CUDA(e, cudaMemcpyAsync(d_idx + n_train, val_idx, (size_t)n_val * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  ctd_k_dataset_rows<<<n_train, 128, 0, e->stream>>>(e->ds_feat, e->ds_meta, e->ds_origin, e->ds_ctr, d_idx, n_train, label, t->feat_tr,
                                                      t->val_tr, d_bad);
  e->launches++;
  if (n_val) {
    ctd_k_dataset_rows<<<n_val, 128, 0, e->stream>>>(e->ds_feat, e->ds_meta, e->ds_origin, e->ds_ctr, d_idx + n_train, n_val, label,
                                                      t->feat_va, t->val_va, d_bad);
    e->launches++;
  }
  CTD_CUDA(e, cudaGetLastError());
  int bad = 0;
  CTD_CUDA(e, cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  if (bad) {
    snprintf(e->err, sizeof(e->err), "ctd_train_begin_dataset: %s", bad & 1 ? "an index past the dataset's records" : "a winner label on an errored game");
    return CTD_EARG;
  }
  return ctd_train_install(e, t);
}

// the 16 tensors of ValueOnlyNN(418, 512).state_dict() in its own order (num_batches_tracked aside):
// fc1.weight [512][418] fc1.bias bn1.weight bn1.bias bn1.running_mean bn1.running_var fc2.weight [256][512] fc2.bias bn2.weight
// bn2.bias bn2.running_mean bn2.running_var fc3.weight [128][256] fc3.bias fc4.weight [6][128] fc4.bias
static const size_t ctd_tr_count[16] = {512 * 418, 512, 512, 512, 512, 512, 256 * 512, 256, 256, 256, 256, 256, 128 * 256, 128, 6 * 128, 6};
static float* ctd_tr_slot(CtdTrainer* t, int i) {
  typedef CtdTrainLayout L;
  float* P = t->P;
  float* slots[16] = {P + L::w1, P + L::b1, P + L::g1, P + L::be1, t->rm1, t->rv1, P + L::w2, P + L::b2, P + L::g2, P + L::be2, t->rm2, t->rv2,
                      P + L::w3, P + L::b3, P + L::w4, P + L::b4};
  return slots[i];
}
ctd_status ctd_train_set_state(ctd_engine* e, const float* const* tensors16) {
  if (!e || !e->trainer || !tensors16) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdTrainer* t = e->trainer.get();
  CTD_CUDA(e, cudaMemsetAsync(t->P, 0, CtdTrainLayout::total * sizeof(float), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(t->M, 0, CtdTrainLayout::total * sizeof(float), e->stream));
  CTD_CUDA(e, cudaMemsetAsync(t->V, 0, CtdTrainLayout::total * sizeof(float), e->stream));
  for (int i = 0; i < 16; ++i) {
    if (!tensors16[i]) return CTD_EARG;
    if (i == 0)   // fc1.weight: rows of 418 into rows of 512
      CTD_CUDA(e, cudaMemcpy2DAsync(ctd_tr_slot(t, 0), CTD_TR_IN * sizeof(float), tensors16[0], 418 * sizeof(float), 418 * sizeof(float), 512, cudaMemcpyHostToDevice, e->stream));
    else
      CTD_CUDA(e, cudaMemcpyAsync(ctd_tr_slot(t, i), tensors16[i], ctd_tr_count[i] * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  }
  t->step = 0;
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}
ctd_status ctd_train_get_state(ctd_engine* e, float* const* tensors16) {
  if (!e || !e->trainer || !tensors16) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdTrainer* t = e->trainer.get();
  for (int i = 0; i < 16; ++i) {
    if (!tensors16[i]) return CTD_EARG;
    if (i == 0)
      CTD_CUDA(e, cudaMemcpy2DAsync(tensors16[0], 418 * sizeof(float), ctd_tr_slot(t, 0), CTD_TR_IN * sizeof(float), 418 * sizeof(float), 512, cudaMemcpyDeviceToHost, e->stream));
    else
      CTD_CUDA(e, cudaMemcpyAsync(tensors16[i], ctd_tr_slot(t, i), ctd_tr_count[i] * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  }
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// the gradients of the last optimiser step in the same 16-tensor layout (running statistics have none: zeros) -- test hook
ctd_status ctd_train_get_grads(ctd_engine* e, float* const* tensors16) {
  if (!e || !e->trainer || !tensors16) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdTrainer* t = e->trainer.get();
  for (int i = 0; i < 16; ++i) {
    if (!tensors16[i]) return CTD_EARG;
    const bool stat = i == 4 || i == 5 || i == 10 || i == 11;
    if (stat) { memset(tensors16[i], 0, ctd_tr_count[i] * sizeof(float)); continue; }
    const float* src = t->G + (ctd_tr_slot(t, i) - t->P);
    if (i == 0)
      CTD_CUDA(e, cudaMemcpy2DAsync(tensors16[0], 418 * sizeof(float), src, CTD_TR_IN * sizeof(float), 418 * sizeof(float), 512, cudaMemcpyDeviceToHost, e->stream));
    else
      CTD_CUDA(e, cudaMemcpyAsync(tensors16[i], src, ctd_tr_count[i] * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  }
  CTD_CUDA(e, cudaStreamSynchronize(e->stream));
  return CTD_OK;
}

// C [M][N] (ldc) = A [M][K] (lda) . B [N][K]^T (ldb) + bias, optional ReLU, on the tensor cores (N multiple of 128, K of 32)
static void ctd_tr_gemm(ctd_engine* e, const float* A, int lda, const float* B, int ldb, const float* bias, float* C, int ldc, int M, int N, int K, int relu) {
  ctd_k_linear_tc<<<dim3((M + CTD_TC_BM - 1) / CTD_TC_BM, N / CTD_TC_BN), 128, CTD_TC_SMEM, e->stream>>>(A, lda, B, ldb, bias, C, ldc, M, K, relu, e->d_tc_err);
  e->launches++;
}
static void ctd_tr_transpose(ctd_engine* e, const float* in, int R, int C, int ld_in, float* out, int ld_out) {
  ctd_k_tr_transpose<<<dim3((C + 31) / 32, (ld_out + 31) / 32), dim3(32, 8), 0, e->stream>>>(in, R, C, ld_in, out, ld_out);
  e->launches++;
}
// forward of one batch already gathered into t->X / t->T; train: batch statistics + dropout, else running statistics
static void ctd_tr_forward(ctd_engine* e, CtdTrainer* t, uint32_t B, int train, uint64_t seed) {
  typedef CtdTrainLayout L;
  const uint32_t bp = t->bp;
  ctd_tr_gemm(e, t->X, CTD_TR_IN, t->P + L::w1, CTD_TR_IN, t->P + L::b1, t->Z1, CTD_TR_H1, (int)B, CTD_TR_H1, CTD_TR_IN, 0);
  ctd_k_tr_bn_fwd<<<CTD_TR_H1 / 32, dim3(32, 8), 0, e->stream>>>(t->Z1, CTD_TR_H1, B, bp, t->P + L::g1, t->P + L::be1, t->rm1, t->rv1, t->inv1, t->H1, train, seed, t->step, 1);
  ctd_tr_gemm(e, t->H1, CTD_TR_H1, t->P + L::w2, CTD_TR_H1, t->P + L::b2, t->Z2, CTD_TR_H2, (int)B, CTD_TR_H2, CTD_TR_H1, 0);
  ctd_k_tr_bn_fwd<<<CTD_TR_H2 / 32, dim3(32, 8), 0, e->stream>>>(t->Z2, CTD_TR_H2, B, bp, t->P + L::g2, t->P + L::be2, t->rm2, t->rv2, t->inv2, t->H2, train, seed, t->step, 2);
  ctd_tr_gemm(e, t->H2, CTD_TR_H2, t->P + L::w3, CTD_TR_H2, t->P + L::b3, t->H3, CTD_TR_H3, (int)B, CTD_TR_H3, CTD_TR_H2, 1);
  e->launches += 2;
}

// one epoch of train_node_value_only: every batch of `perm` order (model.train()), then the evaluation pass over the validation
// set in its own order (model.eval()).  *train_loss / *eval_loss: mean over batches of the batch-mean KL loss (train.py:46-69).
ctd_status ctd_train_epoch(ctd_engine* e, uint64_t seed, float lr, const uint32_t* perm, double* train_loss, double* eval_loss) {
  if (!e || !e->trainer) return CTD_EARG;
  CTD_CUDA(e, cudaSetDevice(e->device));
  CtdTrainer* t = e->trainer.get();
  typedef CtdTrainLayout L;
  const uint32_t bp = t->bp;
  if (perm) CTD_CUDA(e, cudaMemcpyAsync(t->perm, perm, (size_t)t->n_train * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  double tl = 0.0, el = 0.0;
  uint32_t nb = 0;
  for (uint32_t first = 0; first < t->n_train; first += t->batch, ++nb) {
    const uint32_t B = t->n_train - first < t->batch ? t->n_train - first : t->batch;
    ctd_k_tr_gather<<<bp, 128, 0, e->stream>>>(t->feat_tr, t->val_tr, perm ? t->perm.get() : nullptr, first, B, bp, t->X, t->T);
    ctd_tr_forward(e, t, B, 1, seed);
    CTD_CUDA(e, cudaMemsetAsync(t->loss, 0, sizeof(double), e->stream));
    CTD_CUDA(e, cudaMemsetAsync(t->G, 0, L::total * sizeof(float), e->stream));
    ctd_k_tr_head<<<(B + 127) / 128, 128, 0, e->stream>>>(t->H3, t->P + L::w4, t->P + L::b4, t->T, B, t->dY, t->loss);
    // ---- backward
    ctd_k_tr_fc4_bwd<<<bp, CTD_TR_H3, 0, e->stream>>>(t->dY, t->P + L::w4, t->H3, B, bp, t->dZ3);
    ctd_k_tr_fc4_wgrad<<<6, CTD_TR_H3, 0, e->stream>>>(t->dY, t->H3, B, t->G + L::w4, t->G + L::b4);
    ctd_tr_transpose(e, t->dZ3, (int)bp, CTD_TR_H3, CTD_TR_H3, t->dZ3T, (int)bp);
    ctd_tr_transpose(e, t->H2, (int)bp, CTD_TR_H2, CTD_TR_H2, t->H2T, (int)bp);
    ctd_tr_gemm(e, t->dZ3T, (int)bp, t->H2T, (int)bp, t->zero, t->G + L::w3, CTD_TR_H2, CTD_TR_H3, CTD_TR_H2, (int)bp, 0);      // dW3 = dZ3^T . H2
    ctd_k_tr_colsum<<<CTD_TR_H3 / 32, dim3(32, 8), 0, e->stream>>>(t->dZ3, CTD_TR_H3, B, t->G + L::b3);
    ctd_tr_transpose(e, t->P + L::w3, CTD_TR_H3, CTD_TR_H2, CTD_TR_H2, t->W3T, CTD_TR_H3);
    ctd_tr_gemm(e, t->dZ3, CTD_TR_H3, t->W3T, CTD_TR_H3, t->zero, t->dH2, CTD_TR_H2, (int)B, CTD_TR_H2, CTD_TR_H3, 0);           // dH2 = dZ3 . W3
    ctd_k_tr_bn_bwd<<<CTD_TR_H2 / 32, dim3(32, 8), 0, e->stream>>>(t->dH2, t->Z2, t->H2, CTD_TR_H2, B, bp, t->P + L::g2, t->inv2, t->G + L::g2, t->G + L::be2);
    ctd_tr_transpose(e, t->dH2, (int)bp, CTD_TR_H2, CTD_TR_H2, t->dZ2T, (int)bp);
    ctd_tr_transpose(e, t->H1, (int)bp, CTD_TR_H1, CTD_TR_H1, t->H1T, (int)bp);
    ctd_tr_gemm(e, t->dZ2T, (int)bp, t->H1T, (int)bp, t->zero, t->G + L::w2, CTD_TR_H1, CTD_TR_H2, CTD_TR_H1, (int)bp, 0);      // dW2 = dZ2^T . H1
    ctd_k_tr_colsum<<<CTD_TR_H2 / 32, dim3(32, 8), 0, e->stream>>>(t->dH2, CTD_TR_H2, B, t->G + L::b2);
    ctd_tr_transpose(e, t->P + L::w2, CTD_TR_H2, CTD_TR_H1, CTD_TR_H1, t->W2T, CTD_TR_H2);
    ctd_tr_gemm(e, t->dH2, CTD_TR_H2, t->W2T, CTD_TR_H2, t->zero, t->dH1, CTD_TR_H1, (int)B, CTD_TR_H1, CTD_TR_H2, 0);           // dH1 = dZ2 . W2
    ctd_k_tr_bn_bwd<<<CTD_TR_H1 / 32, dim3(32, 8), 0, e->stream>>>(t->dH1, t->Z1, t->H1, CTD_TR_H1, B, bp, t->P + L::g1, t->inv1, t->G + L::g1, t->G + L::be1);
    ctd_tr_transpose(e, t->dH1, (int)bp, CTD_TR_H1, CTD_TR_H1, t->dZ1T, (int)bp);
    ctd_tr_transpose(e, t->X, (int)bp, CTD_TR_IN, CTD_TR_IN, t->XT, (int)bp);
    ctd_tr_gemm(e, t->dZ1T, (int)bp, t->XT, (int)bp, t->zero, t->G + L::w1, CTD_TR_IN, CTD_TR_H1, CTD_TR_IN, (int)bp, 0);        // dW1 = dZ1^T . X
    ctd_k_tr_colsum<<<CTD_TR_H1 / 32, dim3(32, 8), 0, e->stream>>>(t->dH1, CTD_TR_H1, B, t->G + L::b1);
    // ---- Adam
    t->step += 1;
    const float bc1 = 1.f - powf(0.9f, (float)t->step), bc2 = 1.f - powf(0.999f, (float)t->step);
    ctd_k_tr_adam<<<(unsigned)((L::total + 255) / 256), 256, 0, e->stream>>>(t->P, t->G, t->M, t->V, L::total, lr, bc1, bc2);
    e->launches += 10;
    CTD_CUDA(e, cudaGetLastError());
    double h = 0.0;
    CTD_CUDA(e, cudaMemcpyAsync(&h, t->loss, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    tl += h / (double)B;
  }
  if (train_loss) *train_loss = nb ? tl / nb : 0.0;
  uint32_t vb = 0;
  for (uint32_t first = 0; first < t->n_val; first += t->batch, ++vb) {
    const uint32_t B = t->n_val - first < t->batch ? t->n_val - first : t->batch;
    ctd_k_tr_gather<<<bp, 128, 0, e->stream>>>(t->feat_va, t->val_va, nullptr, first, B, bp, t->X, t->T);
    ctd_tr_forward(e, t, B, 0, seed);
    CTD_CUDA(e, cudaMemsetAsync(t->loss, 0, sizeof(double), e->stream));
    ctd_k_tr_head<<<(B + 127) / 128, 128, 0, e->stream>>>(t->H3, t->P + L::w4, t->P + L::b4, t->T, B, nullptr, t->loss);
    e->launches += 2;
    CTD_CUDA(e, cudaGetLastError());
    double h = 0.0;
    CTD_CUDA(e, cudaMemcpyAsync(&h, t->loss, sizeof(double), cudaMemcpyDeviceToHost, e->stream));
    CTD_CUDA(e, cudaStreamSynchronize(e->stream));
    el += h / (double)B;
  }
  if (eval_loss) *eval_loss = vb ? el / vb : 0.0;
  int terr = 0;
  CTD_CUDA(e, cudaMemcpy(&terr, e->d_tc_err, sizeof(int), cudaMemcpyDeviceToHost));
  if (terr) { CTD_CUDA(e, cudaMemset(e->d_tc_err, 0, sizeof(int))); snprintf(e->err, sizeof(e->err), "tcgen05 GEMM: mbarrier wait timed out"); return CTD_ECUDA; }
  return CTD_OK;
}

}  // extern "C"
