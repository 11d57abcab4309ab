// ctd_search.cuh -- the two MCCFR search kernels (cfr_train / one wave of cfr_pred), shared by two translation units like
// ctd_playout.cuh: ctd_kernels.cu instantiates them for any ruleset, ctd_preset_search.cu with CTD_FIXED_PRESET (everything
// outside the preset eight unreachable) -- both kernels are instruction-fetch bound, so the smaller image is the faster one.
#pragma once
#include "ctd_playout.cuh"
#include "ctd_mccfr.cuh"
#define CTD_FULL 0xFFFFFFFFu

#ifndef CTD_MCCFR_KERNEL_NAME
#define CTD_MCCFR_KERNEL_NAME ctd_k_mccfr
#define CTD_MCCFR_PRED_KERNEL_NAME ctd_k_mccfr_pred
#endif

struct CtdMccfrArgs {
  uint32_t n_roots;            // work items of this launch
  const uint32_t* tree_list;   // work item -> root index; null: root index = first_root + item
  const ctd_state* roots;
  const CtdKnow* knows;
  const uint8_t* used_cards;
  const uint64_t* gids;
  uint64_t seed;
  uint32_t iterations;
  uint32_t n0_log2;            // chunk 0 of every tree holds 2^n0_log2 nodes
  CtdTreeHdr* hdrs;            // [capacity]
  CtdArena arena;              // what trees initialised by this launch allocate from
  ctd_mccfr_result* results;
  unsigned long long* counter;
  uint64_t* opts_scratch;  // [gridDim.x * CTD_WARPS_PER_BLOCK][CTD_MCCFR_OPT_CAP]
  uint32_t first_root;
  int resume;                  // 1: continue the trees an earlier launch grew (root-parallel rounds)
  uint32_t* n_epool;           // [1] or null: bumped for every tree that ends with CTD_TREE_EPOOL (the host then looks for them)
};

static __device__ void ctd_write_result(CtdTree& T, ctd_mccfr_result* r) {
  const CtdTreeHdr& h = *T.hdr;
  r->status = h.status; r->n_nodes = h.n_nodes; r->iterations = h.iterations; r->rng_draws = h.rng_draws;
  r->live_option = ctd_live_choice(T);
  if (h.n_nodes == 0) { r->n_children = 0; r->role_pick = 0; r->viewer = 0; r->player = 0; return; }   // refused root: no tree
  const CtdNode& n = ctd_node(T, 0);
  r->n_children = n.n_children; r->role_pick = (n.flags & CTD_NF_ROLE_PICK) ? 1 : 0;
  r->viewer = h.viewer; r->player = n.player;
  for (int i = 0; i < 6; ++i) { r->node_value[i] = n.V[i]; r->winning_probabilities[i] = n.P[i]; }
  const uint32_t K = n.n_children < CTD_MCCFR_MAX_RESULT ? n.n_children : CTD_MCCFR_MAX_RESULT;
  const bool rp = n.flags & CTD_NF_ROLE_PICK;
  const uint32_t na = n.n_children == 0 ? 0 : (rp ? 60 : K);
  if (n.n_children == 0) return;
  const CtdChild* kids = ctd_kids(T, n);
  for (uint32_t i = 0; i < K; ++i) r->options[i] = kids[i].desc;
  const double *R = ctd_R(T, n), *S = ctd_S(T, n), *C = ctd_C(T, n);
  for (uint32_t i = 0; i < na; ++i) { r->cumulative_regrets[i] = R[i]; r->strategy[i] = S[i]; r->cumulative_strategy[i] = C[i]; }
}

#define CTD_MCCFR_MIN_BLOCKS 3 /* 80 registers: fewer spills on the single active lane; 24 trees per SM resident (measured best at the 4096-root configuration) */
#ifndef CTD_NO_TRAIN_KERNEL
__global__ void __launch_bounds__(CTD_BLOCK, CTD_MCCFR_MIN_BLOCKS) CTD_MCCFR_KERNEL_NAME(CtdMccfrArgs a) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK];
  __shared__ __align__(16) uint8_t scratch[CTD_WARPS_PER_BLOCK][CTD_TREE_SCRATCH];
  __shared__ __align__(16) ctd_state tstage[CTD_WARPS_PER_BLOCK];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  uint64_t* opts = a.opts_scratch + ((size_t)blockIdx.x * CTD_WARPS_PER_BLOCK + wib) * CTD_MCCFR_OPT_CAP;
  for (;;) {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(a.counter, 1ull);
    t = __shfl_sync(CTD_FULL, t, 0);
    if (t >= a.n_roots) break;
    t = a.tree_list ? a.tree_list[t] : t + a.first_root;
    // Every lane runs the same scalar search on the same data (identical values to identical addresses, control flow
    // uniform, the warp stays converged): no lane does anything the others do not, but leaf operations that are
    // lane-parallel by nature -- moving a 1.8 KB node between HBM and the working set -- can split their work over the
    // lanes without restructuring the walk.
    {
      CtdTree T;
      T.w = &works[wib]; T.kn = &knows[wib]; T.opts = opts; T.scratch = scratch[wib]; T.stage = &tstage[wib];
      T.vnet = nullptr; T.act = nullptr;
      CtdTreeHdr* hdr = &a.hdrs[t];
      CtdWork& w = *T.w;
      T.hdr = hdr;
      if (a.resume) {
        ctd_chance_init(w, a.seed, a.gids[t], 0);
        w.stream = 1;
        w.err = 0;
        T.kn->err = 0;   // the working set is rebuilt from the tree on the first node load
        ctd_tree_stage_used(T);
        ctd_tree_attach(T, hdr, a.arena);
        ctd_cfr_train(T, a.iterations, true);
        if (a.results) ctd_write_result(T, &a.results[t]);
      } else {
      for (int i = 0; i < 80; ++i) hdr->used_cards[i] = i < 76 ? a.used_cards[t * 76 + i] : 0;
      ctd_copy16(T.stage, &a.roots[t], (int)sizeof(ctd_state));
      ctd_unpack(T.stage, w);
      ctd_chance_init(w, a.seed, a.gids[t], 0);
      w.stream = 1;
      w.err = 0;
      ctd_copy16(T.kn, &a.knows[t], (int)sizeof(CtdKnow));
      ctd_tree_stage_used(T);
#ifdef CTD_FIXED_PRESET
      if (w.ruleset != CTD_RULESET_PRESET) {   // the caller named the wrong ruleset for this root: refuse, do not run
        hdr->n_nodes = 0; hdr->iterations = 0; hdr->rng_draws = 0; hdr->status = CTD_TREE_EENGINE; hdr->child_used = 0; hdr->arr_used = 0;
        if (a.results) { a.results[t].status = CTD_TREE_EENGINE; a.results[t].n_nodes = 0; a.results[t].n_children = 0; a.results[t].iterations = 0; }
      } else
#endif
      {
      ctd_tree_init(T, hdr, a.arena, a.n0_log2, T.kn->viewer, a.gids[t], false, false);
      ctd_cfr_train(T, a.iterations);
      if (a.results) ctd_write_result(T, &a.results[t]);
      }
      }
      if (lane == 0 && a.n_epool && (hdr->status & CTD_TREE_EPOOL)) atomicAdd(a.n_epool, 1u);
    }
    __syncwarp();
  }
}
#endif  // CTD_NO_TRAIN_KERNEL

struct CtdPredArgs {
  CtdMccfrArgs m;
  uint32_t max_depth;
  int first;          // 1: build the trees' roots in this launch
  float* feat;        // [n_roots][CTD_FEATURES_PAD]
  float* pred;        // [n_roots][8]
  uint8_t* pending;   // [n_roots]
  uint32_t* n_pending;   // [0] trees waiting for a leaf value, [1] trees that yielded mid-walk
  uint32_t budget;       // iterations a tree may walk in one wave
  int fused;             // 1: every warp evaluates its own leaves with `net` (one launch, no waves)
  CtdValueNet net;
};

#ifndef CTD_NO_PRED_KERNEL
// one wave of CFRNode.cfr_pred for every tree: walk until a leaf value is needed (or the budget is spent)
__global__ void __launch_bounds__(CTD_BLOCK, CTD_MCCFR_MIN_BLOCKS) CTD_MCCFR_PRED_KERNEL_NAME(CtdPredArgs p) {
  __shared__ CtdWork works[CTD_WARPS_PER_BLOCK];
  __shared__ CtdKnow knows[CTD_WARPS_PER_BLOCK];
  __shared__ __align__(16) uint8_t scratch[CTD_WARPS_PER_BLOCK][CTD_TREE_SCRATCH];
  __shared__ __align__(16) ctd_state tstage[CTD_WARPS_PER_BLOCK];
  extern __shared__ __align__(16) float acts[];   // fused mode: CTD_ACT_FLOATS floats per warp (dynamic: the block then holds more than 48 KB)
  const CtdMccfrArgs& a = p.m;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  uint64_t* opts = a.opts_scratch + ((size_t)blockIdx.x * CTD_WARPS_PER_BLOCK + wib) * CTD_MCCFR_OPT_CAP;
  for (;;) {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(a.counter, 1ull);
    t = __shfl_sync(CTD_FULL, t, 0);
    if (t >= a.n_roots) break;
    t = a.tree_list ? a.tree_list[t] : t + a.first_root;
    {   // all lanes on the same scalar walk, see ctd_k_mccfr
      CtdTree T;
      T.w = &works[wib]; T.kn = &knows[wib]; T.opts = opts; T.scratch = scratch[wib]; T.stage = &tstage[wib];
      CtdTreeHdr* hdr = &a.hdrs[t];
      T.hdr = hdr;
      T.vnet = p.fused ? &p.net : nullptr; T.act = p.fused ? acts + wib * CTD_ACT_FLOATS : nullptr;
      CtdWork& w = *T.w;
      if (p.first) {
        for (int i = 0; i < 80; ++i) hdr->used_cards[i] = i < 76 ? a.used_cards[t * 76 + i] : 0;
        ctd_copy16(T.stage, &a.roots[t], (int)sizeof(ctd_state));
        ctd_unpack(T.stage, w);
        ctd_chance_init(w, a.seed, a.gids[t], 0);
        w.stream = 1;
        w.err = 0;
        ctd_copy16(T.kn, &a.knows[t], (int)sizeof(CtdKnow));
        ctd_tree_stage_used(T);
#ifdef CTD_FIXED_PRESET
        if (w.ruleset != CTD_RULESET_PRESET) {   // the caller named the wrong ruleset for this root: refuse, do not run
          hdr->n_nodes = 0; hdr->iterations = 0; hdr->rng_draws = 0; hdr->status = CTD_TREE_EENGINE; hdr->phase = 3;
          hdr->child_used = 0; hdr->arr_used = 0; hdr->n0_log2 = a.n0_log2; hdr->arena = a.arena.base; hdr->chunk[0] = 0;
        } else
#endif
        ctd_tree_init(T, hdr, a.arena, a.n0_log2, T.kn->viewer, a.gids[t], false, true);
      } else {
        ctd_chance_init(w, a.seed, a.gids[t], 0);
        w.stream = 1;
        w.err = 0;
        T.kn->err = 0;  // the working set is rebuilt from the tree on the first node load of this wave
        ctd_tree_stage_used(T);
      }
      ctd_tree_attach(T, hdr, a.arena);
      int r = CTD_PRED_DONE;
      if (hdr->phase != 3)
        r = ctd_cfr_pred_advance(T, a.iterations, p.max_depth, p.feat + t * CTD_FEATURES_PAD, p.pred + t * 8, p.budget);
      p.pending[t] = r == CTD_PRED_WAIT ? 1 : 0;
      if (r == CTD_PRED_WAIT && lane == 0) atomicAdd(p.n_pending, 1u);
      if (r == CTD_PRED_YIELD && lane == 0) atomicAdd(p.n_pending + 1, 1u);
      if (r == CTD_PRED_DONE && a.results) ctd_write_result(T, &a.results[t]);
      if (r == CTD_PRED_DONE && lane == 0 && a.n_epool && (hdr->status & CTD_TREE_EPOOL)) atomicAdd(a.n_epool, 1u);   // (a finished tree is counted by every later wave too: the host only asks "any?")
    }
    __syncwarp();
  }
}
#define CTD_PRED_FUSED_SMEM (CTD_WARPS_PER_BLOCK * CTD_ACT_FLOATS * sizeof(float))
#endif  // CTD_NO_PRED_KERNEL
