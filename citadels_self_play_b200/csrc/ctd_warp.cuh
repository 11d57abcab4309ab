// ctd_warp.cuh -- warp-cooperative option choice for the fused playout kernel.
//
// One warp owns one game.  For a random playout only two things are needed from Agent.get_options
// (game/agent.py:50-83): how many legal options there are, and which one is the k-th in the reference's list order.
// Here the lanes evaluate the option predicates in parallel -- lane i looks at card i of a hand / building i of a
// city -- and ballots turn the predicates into bit masks: counts are popcounts, "de-duplicate by type, first
// occurrence wins" (game/agent_functions.py:28-32, :99-103, :117-118, :479-480) is __match_any_sync + lowest lane,
// and the k-th option is the k-th set bit (__fns).  Scalars of the record are read by every lane from shared
// memory (broadcast), so control flow stays uniform and branchy character abilities diverge per game, not per lane.
//
// States outside the fast path (Wizard's take-from-hand, Lighthouse, hands over 32 cards) fall back to the scalar
// enumerator on lane 0 (ctd_engine.cuh), which is also the definition both paths are tested against
// (ctd_k_choose_check in ctd_kernels.cu: every k of every step of the recorded reference games).
#pragma once
#include "ctd_engine.cuh"

#define CTD_CHOOSE_BUF 32
/* descriptors kept by the scalar fallback (256 B = one packed record); longer lists are selected by a second enumeration pass */

#ifdef __CUDACC__
#define CTD_ALL 0xFFFFFFFFu

// scalar fallback: lane 0 materialises the list, draws k, picks
// CHECK: the checker's form (ctd_k_choose_check: report the count, take a given k).  The playout kernels instantiate CHECK = false,
// where count_out / want are dead on entry and cost neither registers nor code.
template <bool CHECK>
static __device__ __noinline__ uint64_t ctd_choose_scalar(CtdWork& w, int lane, uint64_t* buf, uint32_t* count_out_, int want_) {
  uint32_t* const count_out = CHECK ? count_out_ : nullptr;
  const int want = CHECK ? want_ : -1;
  CTD_ASSUME_SHARED(&w);
  uint64_t d = 0;
  uint32_t n = 0;
  if (lane == 0) {
    // the Seer's and the Scholar's enumerations are not pure (chance draws, shrinking list): remember what they touch
    // so that a second selecting pass regenerates the same list
    const uint32_t draws0 = w.draws, tape0 = w.tape_pos;
    const uint8_t n7 = w.n_seven;
    uint8_t s7[7];
    for (int i = 0; i < 7; ++i) s7[i] = w.seven[i];
    CtdEmit e{buf, CTD_CHOOSE_BUF, 0, 0xFFFFFFFFu, 0};
    ctd_enumerate(w, e);
    n = e.n;
    if (n != 0) {
      uint32_t k = want >= 0 ? (uint32_t)want : ctd_randbelow(w, n);
      if (k < CTD_CHOOSE_BUF && k < n) {
        d = buf[k];
      } else if (k < n) {
        const uint32_t draws1 = w.draws, tape1 = w.tape_pos;
        w.draws = draws0; w.tape_pos = tape0; w.buf_blk = 0xFFFFFFFFu; w.n_seven = n7;
        for (int i = 0; i < 7; ++i) w.seven[i] = s7[i];
        CtdEmit e2{buf, 0, 0, k, 0};
        ctd_enumerate(w, e2);
        d = e2.got;
        w.draws = draws1; w.tape_pos = tape1; w.buf_blk = 0xFFFFFFFFu;
      }
    }
  }
  if (count_out) *count_out = __shfl_sync(CTD_ALL, n, 0);
  return __shfl_sync(CTD_ALL, d, 0);
}

// position of the k-th (0-based) set bit: the lane that owns it finds itself, one ballot tells everybody
__device__ __forceinline__ int ctd_kth_bit(uint32_t mask, uint32_t k, int lane) {
  const bool mine = ((mask >> lane) & 1) && (uint32_t)__popc(mask & ((1u << lane) - 1)) == k;
  return __ffs(__ballot_sync(CTD_ALL, mine)) - 1;
}

// "first card of its type in this list" for lane < n (lanes beyond n never match anything)
__device__ __forceinline__ bool ctd_first_of_type(int lane, int n, int t) {
  const int key = lane < n ? t : 64 + lane;
  const uint32_t m = __match_any_sync(CTD_ALL, key);
  return lane < n && (__ffs(m) - 1) == lane;
}

// printed cost by type, 3 bits each, ten types per 32-bit word (game/config.py:2-80)
__device__ __forceinline__ int ctd_cost_w(int t) {
  const uint32_t w0 = 1u | 2u << 3 | 4u << 6 | 2u << 9 | 5u << 12 | 3u << 15 | 2u << 18 | 3u << 21 | 5u << 24 | 1u << 27;
  const uint32_t w1 = 2u | 3u << 3 | 1u << 6 | 4u << 9 | 3u << 12 | 5u << 15 | 5u << 18 | 3u << 21 | 6u << 24 | 2u << 27;
  const uint32_t w2 = 6u | 5u << 3 | 5u << 6 | 6u << 9 | 5u << 12 | 6u << 15 | 6u << 18 | 3u << 21 | 6u << 24 | 3u << 27;
  const uint32_t w3 = 5u | 5u << 3 | 6u << 6 | 5u << 9 | 4u << 12 | 6u << 15 | 5u << 18 | 4u << 21 | 0u << 24 | 5u << 27;
  const int q = t / 10;
  const uint32_t w = q == 0 ? w0 : (q == 1 ? w1 : (q == 2 ? w2 : w3));
  return (int)((w >> (3 * (t - 10 * q))) & 7);
}

// Count the options of the game in `w`, draw k (or take `want` >= 0, used by the checker), return the k-th.
// *count_out (optional) receives the number of options.  Every lane returns the same descriptor; 0 = none.
// Structure: (A) classify the state and count -- all ballots happen here; (B) ONE draw; (C) select.
enum { CTD_PM_ROLE_PICK, CTD_PM_GOLD_OR_CARD, CTD_PM_SINGLE, CTD_PM_KEEP, CTD_PM_KEEP_LIBRARY, CTD_PM_WITCH, CTD_PM_MAIN };

#ifndef CTD_CHOOSE_LINKAGE
#define CTD_CHOOSE_LINKAGE static
#endif
// `ring_`, `ring` and the `ring != nullptr` draw below are unused; kept so that the callers' code stays unchanged
template <bool CHECK = false>
CTD_CHOOSE_LINKAGE __device__ __noinline__ uint64_t ctd_warp_choose(CtdWork& w, int lane, uint64_t* buf, uint32_t* count_out_ = nullptr,
                                                 int want_ = -1, const uint32_t* ring_ = nullptr) {
  uint32_t* const count_out = CHECK ? count_out_ : nullptr;
  const int want = CHECK ? want_ : -1;
  const uint32_t* const ring = nullptr;
  const int p = w.player, st = w.state;
  if ((w.gflags & 2) || p >= 6) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);
  const uint64_t me = (uint64_t)p << 6;
  int mode = -1;
  uint32_t total = 0, m0 = 0, m1 = 0, m2 = 0;   // mode-specific masks
  uint64_t single = 0;
  // main-round class counts
  // (the seven small ones share one register: bit 0 beg, 1 war gold, 2 smithy, 3 magic school (x5), bits 8-15 lab, 16-23 weapon storage,
  // 24-31 museum -- the function runs under a 32-register bound and spills what does not fit)
  uint32_t c_build = 0, c_char = 0, cx = 0;
  int nm = 0, nh = 0;
  uint64_t own = 0;
  if (st == 0) {  // pick_role_options: one per role still on offer, rank ascending
    mode = CTD_PM_ROLE_PICK; m0 = w.rtc_mask; total = __popc(m0);
  } else {
    const int role = w.role[p];
    if (role >= 8) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);  // None / Bewitched: error paths
    nm = role * 3 + w.variant[role];
    const int rp = w.rprops[role];
    if (rp & CTD_RP_DEAD) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);
    if (st == 1) {
      mode = CTD_PM_GOLD_OR_CARD; total = w.n_deck > 1 ? 2 : 1;
    } else if (st == 3 && !(rp & CTD_RP_BLACKMAIL)) {
      mode = CTD_PM_SINGLE; total = 1; single = CTD_K_EMPTY | me;
    } else if (st == 6) {
      mode = CTD_PM_SINGLE; total = 1; single = (uint64_t)(w.gold[p] > 0 ? CTD_K_GRAVEYARD : CTD_K_EMPTY) | me;
    } else if (st == 2 || st == 5) {
      const int nb = w.n_bld[p];
      {  // which building types do I own: lanes OR their building's bit
        uint64_t bit = 0;
        if (lane < nb) bit = 1ull << ctd_ctype(w.bld[p][lane]);
        own = (uint64_t)__reduce_or_sync(CTD_ALL, (uint32_t)bit) | ((uint64_t)__reduce_or_sync(CTD_ALL, (uint32_t)(bit >> 32)) << 32);
      }
      if (st == 2) {  // which_card_to_keep_options
        const int n = w.n_jd[p];
        if (n > 32) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);
        if ((own >> 20) & 1) {  // Library: every pair i < j, no de-duplication
          mode = CTD_PM_KEEP_LIBRARY; m0 = (uint32_t)n; total = (uint32_t)(n * (n - 1) / 2);
        } else {
          mode = CTD_PM_KEEP;
          m0 = __ballot_sync(CTD_ALL, ctd_first_of_type(lane, n, lane < n ? ctd_ctype(w.jd[p][lane]) : 0));
          total = __popc(m0);
        }
      } else if (nm == CTD_WITCH) {
        mode = CTD_PM_WITCH; total = 7;
      } else if (rp & CTD_RP_POSSESSED) {
        mode = CTD_PM_SINGLE; total = 1;
        single = CTD_K_FINISH | me | ctd_f_next_witch(1) | ctd_f_crown(nm == CTD_KING || nm == CTD_PATRICIAN);
      } else {
        // ------------------------------------------------------------ main_round_options, the reference's order
        nh = w.n_hand[p];
        const bool lighthouse = ((own >> 29) & 1) && (w.pflags[p] & CTD_PF_LIGHTHOUSE);
        const uint32_t tier_ab = (1u << CTD_SPY) | (1u << CTD_WIZARD) | (1u << CTD_KING) | (1u << CTD_ABBOT) | (1u << CTD_ALCHEMIST) |
                                 (1u << CTD_NAVIGATOR) | (1u << CTD_WARLORD) | (1u << CTD_ASSASSIN) | (1u << CTD_THIEF) |
                                 (1u << CTD_MAGICIAN) | (1u << CTD_BISHOP) | (1u << CTD_MERCHANT) | (1u << CTD_ARCHITECT);
        if (nh > 32 || lighthouse || !((tier_ab >> nm) & 1)) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);
        mode = CTD_PM_MAIN;
        const int gold = w.gold[p], done = w.done;
        const int hc = lane < nh ? w.hand[p][lane] : 0, ht = ctd_ctype(hc);
        const bool hfirst = ctd_first_of_type(lane, nh, ht);
        const bool unique = hc >= 16 && hc < 40;
        if (w.n_trade + w.n_nontrade < ctd_build_limit(nm)) {  // 1. builds (Factory makes uniques dearer)
          const int cost = ctd_cost_w(ht) + ((((own >> 35) & 1) && unique) ? 1 : 0);
          m0 = __ballot_sync(CTD_ALL, hfirst && cost <= gold);
        }
        c_build = __popc(m0);
        if (!(done & CTD_DM_CHARACTER)) {  // 2. character
          if (nm == CTD_SPY) { CTD_NOT_CLASSIC(); c_char = 25; }
          else if (nm == CTD_ASSASSIN) { CTD_NOT_PRESET(); c_char = 7; }
          else if (nm == CTD_THIEF) { CTD_NOT_PRESET(); c_char = 6; }
          else if (nm == CTD_NAVIGATOR) { CTD_NOT_CLASSIC(); c_char = 2; }
          else if (nm == CTD_KING) c_char = 1;
          else if (nm == CTD_BISHOP || nm == CTD_MERCHANT || nm == CTD_ARCHITECT) { CTD_NOT_PRESET(); c_char = 1; }
          else if (nm == CTD_WIZARD) {
            CTD_NOT_CLASSIC();
            m1 = __ballot_sync(CTD_ALL, lane < 6 && lane != p && w.n_hand[lane < 6 ? lane : 0] > 0);
            c_char = __popc(m1);
          } else if (nm == CTD_ABBOT) {
            CTD_NOT_CLASSIC();
            m1 = __ballot_sync(CTD_ALL, lane < nh && ctd_csuit(hc) == CTD_SUIT_RELIGION);
            c_char = m1 ? __popc(m1) + 1 : 0;
          } else if (nm == CTD_MAGICIAN) {
            CTD_NOT_PRESET();
            c_char = 5 + __reduce_add_sync(CTD_ALL, lane < nh ? ctd_magician_count(nh, lane + 1) : 0u);
          } else if (nm == CTD_WARLORD) {
            // lane = (seat, slot): seats 0..2 in m1, seats 3..5 in m2, ten building slots per seat (cities of >= 7 are immune)
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
              const int q = half * 3 + lane / 10, i = lane % 10;
              const int nq = lane < 30 ? w.n_bld[q] : 0;
              const bool live = lane < 30 && nq < 7 && i < nq && ctd_name(w, q) != CTD_BISHOP;
              const int c = live ? w.bld[q][i] : 0, t = ctd_ctype(c);
              const uint32_t grp = __match_any_sync(CTD_ALL, live ? (q << 6) | t : 1024 + lane);
              const bool ok = live && (__ffs(grp) - 1) == lane && ctd_cost_w(t) - 1 <= gold && t != 17;
              const uint32_t mm = __ballot_sync(CTD_ALL, ok);
              if (half == 0) m1 = mm; else m2 = mm;
            }
            c_char = __popc(m1) + __popc(m2);
          }
        }
        if (nm == CTD_ABBOT && !(done & CTD_DM_BEGGED)) cx |= 1u;
        if (nm == CTD_WARLORD && !(done & CTD_DM_TAKE_GOLD)) cx |= 2u;
        if (((own >> 21) & 1) && gold >= 2 && !(done & CTD_DM_SMITHY)) cx |= 4u;
        if (((own >> 25) & 1) && !(done & CTD_DM_MAGIC_SCHOOL)) cx |= 8u;
        if (((own >> 22) & 1) && !(done & CTD_DM_LAB)) cx |= (uint32_t)nh << 8;
        if ((own >> 27) & 1) {
          const uint32_t ws = (uint32_t)(w.n_bld[0] + w.n_bld[1] + w.n_bld[2] + w.n_bld[3] + w.n_bld[4] + w.n_bld[5] - nb);
          if (ws > 255u) return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);   // beyond the packed field (no real game gets near)
          cx |= ws << 16;
        }
        uint32_t m_mus = 0;
        if (((own >> 34) & 1) && !(done & CTD_DM_MUSEUM)) m_mus = __ballot_sync(CTD_ALL, hfirst);
        cx |= (uint32_t)__popc(m_mus) << 24;
        if (nm != CTD_WARLORD) m2 = m_mus;          // m2 is free unless the Warlord uses it ...
        else single = m_mus;                        // ... then the museum mask travels in `single`
        total = c_build + c_char + (cx & 1u) + ((cx >> 1) & 1u) + ((cx >> 2) & 1u) + ((cx >> 3) & 1u) * 5u + ((cx >> 8) & 255u) +
                ((cx >> 16) & 255u) + (cx >> 24) + 1;
      }
    } else {
      return ctd_choose_scalar<CHECK>(w, lane, buf, count_out, want);
    }
  }
  if (count_out) *count_out = total;
  if (total == 0) return 0;
  // ---------------------------------------------------------------- (B) one draw
  uint32_t k;
  if (want >= 0) {
    k = (uint32_t)want;
  } else if (ring != nullptr) {                     // never taken (see `ring` above)
    const uint32_t dr = w.draws;
    k = (uint32_t)(((uint64_t)ring[dr & 127u] * total) >> 32);
    __syncwarp();
    if (lane == 0) w.draws = dr + 1;
  } else {
    k = 0;
    if (lane == 0) k = ctd_randbelow(w, total);
    k = __shfl_sync(CTD_ALL, k, 0);
  }
  // ---------------------------------------------------------------- (C) select
  switch (mode) {
    case CTD_PM_ROLE_PICK: return CTD_K_ROLE_PICK | me | ctd_f_rank(ctd_kth_bit(m0, k, lane));
    case CTD_PM_GOLD_OR_CARD: return CTD_K_GOLD_OR_CARD | me | ctd_f_named(k == 0 ? CTD_N_GOLD : CTD_N_CARD);
    case CTD_PM_SINGLE: return single;
    case CTD_PM_KEEP: return CTD_K_KEEP | me | ctd_f_a(ctd_ctype(w.jd[p][ctd_kth_bit(m0, k, lane)]));
    case CTD_PM_KEEP_LIBRARY: {
      const int n = (int)m0;
      int i = 0;
      while (k >= (uint32_t)(n - 1 - i)) { k -= (uint32_t)(n - 1 - i); ++i; }
      return CTD_K_KEEP | me | ctd_f_a(ctd_ctype(w.jd[p][i])) | ctd_f_b(ctd_ctype(w.jd[p][i + 1 + (int)k]));
    }
    case CTD_PM_WITCH: return CTD_K_BEWITCHING | me | ctd_f_rank(1 + (int)k);
    default: break;
  }
  if (k < c_build) {
    const int t = ctd_ctype(w.hand[p][ctd_kth_bit(m0, k, lane)]);
    const int rep = (((own >> t) & 1) && !w.replicas[p]) ? w.replicas[p] + 1 : 0;
    return CTD_K_BUILD | me | ctd_f_a(t) | ctd_f_replica(rep);
  }
  k -= c_build;
  if (k < c_char) {
    int q = (int)k / 5;            // Spy: five suits per other seat; Magician swaps: one per other seat
    q += q >= p ? 1 : 0;
    int q1 = (int)k;
    q1 += q1 >= p ? 1 : 0;
    switch (nm) {
      case CTD_ASSASSIN: CTD_NOT_PRESET(); return CTD_K_ASSASSINATION | me | ctd_f_rank(1 + (int)k);
      case CTD_THIEF: CTD_NOT_PRESET(); return CTD_K_STEAL | me | ctd_f_rank(2 + (int)k);
      case CTD_SPY: CTD_NOT_CLASSIC(); return CTD_K_SPY | me | ctd_f_target(q) | ctd_f_named(CTD_N_TRADE + (int)k % 5);
      case CTD_MAGICIAN: CTD_NOT_PRESET(); {
        if (k < 5) return CTD_K_MAGIC_HAND_CHANGE | me | ctd_f_target(q1);
        k -= 5;  // every discard_and_draw option has the same effect; recover (r, j) for the descriptor
        int r = 1;
        for (; r <= nh; ++r) {
          const uint32_t c = ctd_magician_count(nh, r);
          if (k < c) break;
          k -= c;
        }
        return CTD_K_DISCARD_AND_DRAW | me | ctd_f_r(r) | ctd_f_j(k);
      }
      case CTD_WIZARD: CTD_NOT_CLASSIC(); return CTD_K_LOOK_AT_HAND | me | ctd_f_target(ctd_kth_bit(m1, k, lane));
      case CTD_KING: return CTD_K_TAKE_CROWN_KING | me;
      case CTD_BISHOP: CTD_NOT_PRESET(); return CTD_K_BISHOP | me;
      case CTD_MERCHANT: CTD_NOT_PRESET(); return CTD_K_MERCHANT | me;
      case CTD_ARCHITECT: CTD_NOT_PRESET(); return CTD_K_ARCHITECT | me;
      case CTD_ABBOT: CTD_NOT_CLASSIC(); return CTD_K_ABBOT | me | ctd_f_count((int)k) | ctd_f_r((int)__popc(m1));
      case CTD_NAVIGATOR: CTD_NOT_CLASSIC(); return CTD_K_NAVIGATOR | me | ctd_f_named(k == 0 ? CTD_N_4GOLD : CTD_N_4CARD);
      default: {  // CTD_WARLORD: (seat, slot) lanes, seats 0..2 then 3..5
        const uint32_t c1 = __popc(m1);
        const uint32_t mm = k < c1 ? m1 : m2;
        const int l = ctd_kth_bit(mm, k < c1 ? k : k - c1, lane);
        const int q2 = (k < c1 ? 0 : 3) + l / 10;
        return CTD_K_WARLORD | me | ctd_f_target(q2) | ctd_f_a(ctd_ctype(w.bld[q2][l % 10]));
      }
    }
  }
  k -= c_char;
  const uint32_t c_beg = cx & 1u, c_wgold = (cx >> 1) & 1u, c_smithy = (cx >> 2) & 1u, c_ms = ((cx >> 3) & 1u) * 5u,
                 c_lab = (cx >> 8) & 255u, c_ws = (cx >> 16) & 255u, c_mus = cx >> 24;
  if (k < c_beg) return CTD_K_ABBOT_BEG | me;
  k -= c_beg;
  if (k < c_wgold) return CTD_K_TAKE_GOLD_WAR | me;
  k -= c_wgold;
  if (k < c_smithy) return CTD_K_SMITHY | me;
  k -= c_smithy;
  if (k < c_lab) return CTD_K_LAB | me | ctd_f_a(ctd_ctype(w.hand[p][k]));
  k -= c_lab;
  if (k < c_ms) return CTD_K_MAGIC_SCHOOL | me | ctd_f_named(CTD_N_TRADE + (int)k);
  k -= c_ms;
  if (k < c_ws) {
    int q = 0;
    for (;; ++q) {
      if (q == p) continue;
      const uint32_t c = w.n_bld[q];
      if (k < c) break;
      k -= c;
    }
    return CTD_K_WEAPON_STORAGE | me | ctd_f_target(q) | ctd_f_a(ctd_ctype(w.bld[q][k]));
  }
  k -= c_ws;
  if (k < c_mus) {
    const uint32_t m_mus = nm != CTD_WARLORD ? m2 : (uint32_t)single;
    return CTD_K_MUSEUM | me | ctd_f_a(ctd_ctype(w.hand[p][ctd_kth_bit(m_mus, k, lane)]));
  }
  return CTD_K_FINISH | me;
}
#endif
