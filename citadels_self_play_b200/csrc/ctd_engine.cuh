// ctd_engine.cuh -- the Citadels rules engine: on-chip working state, legal-option enumeration and
// state transition.  Written from the behaviour of the reference (paths below are relative to the
// reference repository root), not from its code structure: the reference walks Python object graphs
// (Card/Deck/Agent/option); this engine works on a flat working record that lives in shared memory (in the fused playout: thread-local memory) for
// the whole life of a game and is only packed to the 256-byte HBM record (ctd_state) at the API boundary.
//
// Execution model on the device.  The fused random playout (ctd_playout.cuh) gives every thread a game of its own: the
// working record sits in that thread's local memory, and the thread chooses with the scalar enumerator (count, draw,
// select) and applies with `ctd_apply`.  The other kernels (MCCFR, arena, step-wise API) give one warp one game: the
// record sits in the warp's slice of shared memory and the transition (`ctd_apply`), a scalar, order-sensitive list
// manipulation, runs on lane 0.  Enumeration (`ctd_enumerate`) is one scalar visitor walk that defines the option order:
// it materialises option lists (CtdEmit) or counts and selects the k-th option (CtdPick, ctd_playout.cuh).
//
// The same source compiles for the host (tests/hostsim) so the rules can be replayed against the golden
// traces without a GPU; that build is a test vehicle, never a fallback of the product.
#pragma once
#include <stdint.h>
#include <stddef.h>
#include "../../include/citadels_b200.h"

#if defined(__CUDACC__) && defined(CTD_DEVICE_ONLY)
#define CTD_HD __device__ /* a second translation unit must not emit host copies of the inline rules code */
#define CTD_NI __noinline__
#define CTD_LOOP _Pragma("unroll 1")
#define CTD_UNROLL _Pragma("unroll")
#elif defined(__CUDACC__)
#define CTD_HD __host__ __device__
// out-of-line on the device: the playout kernel's warps sit at unrelated points of the rules code, so the
// instruction footprint (not the arithmetic) is what the SM front end sees; one copy of each helper.
#define CTD_NI __noinline__
#define CTD_LOOP _Pragma("unroll 1")
#define CTD_UNROLL _Pragma("unroll")
#else
#define CTD_HD
#define CTD_NI
#define CTD_LOOP
#define CTD_UNROLL
#endif
// On the device every CtdKnow, and every CtdWork of the warp-per-game kernels, lives in shared memory (they declare them
// __shared__).  Telling the compiler turns the generic LD.E / ST.E (+ descriptor moves and 64-bit address arithmetic) of the
// out-of-line rules code into LDS / STS with immediate offsets.  The fused playout units define CTD_WORK_LOCAL: there each
// thread plays its own game in a CtdWork of its own local memory (ctd_playout.cuh), and the same hint gives LDL / STL.
#if defined(__CUDA_ARCH__)
#define CTD_ASSUME_SHARED(p) __builtin_assume(__isShared(p))
#define CTD_ASSUME_GLOBAL(p) __builtin_assume(__isGlobal(p))
#ifdef CTD_WORK_LOCAL
#define CTD_ASSUME_WORK(p) __builtin_assume(__isLocal(p))
#else
#define CTD_ASSUME_WORK(p) CTD_ASSUME_SHARED(p)
#endif
#else
#define CTD_ASSUME_SHARED(p)
#define CTD_ASSUME_GLOBAL(p)
#define CTD_ASSUME_WORK(p)
#endif
#define CTD_ASSUME_SHARED_K(p) CTD_ASSUME_SHARED(p)
// (Only references to whole records carry the hint.  Hinting the raw list pointers of ctd_take_like & co. as well made
// the kernels fault on the device -- either hint alone was fine, both together were not -- so those stay generic.)

// ------------------------------------------------------------------------------------------ constants
// CTD_FIXED_PRESET (set by ctd_preset_playout.cu / ctd_preset_search.cu only): the translation unit plays the preset ruleset exclusively -- Witch,
// Spy, Wizard, King, Abbot, Alchemist, Navigator, Warlord (game/game.py:479-486) -- so every option kind and character
// outside it is unreachable and the compiler drops that code.
#ifdef CTD_FIXED_PRESET
#define CTD_NOT_PRESET() __builtin_unreachable()
#else
#define CTD_NOT_PRESET() ((void)0)
#endif
// CTD_FIXED_CLASSIC (ctd_classic_playout.cu): the classic eight only -- Assassin, Thief, Magician, King, Bishop, Merchant,
// Architect, Warlord (the characters BASELINE.json's north_star names; game/config.py:83-91, first variant of every rank).
#ifdef CTD_FIXED_CLASSIC
#define CTD_NOT_CLASSIC() __builtin_unreachable()
#else
#define CTD_NOT_CLASSIC() ((void)0)
#endif
// Container capacities.  The fused playout units (ctd_*_playout.cu) define CTD_SMALL_CAPS: real games of the fixed rulesets
// stay far below them (hand 25, city 9, museum 14, just_drawn 33 over 5e5 games) and the working record is what occupies
// their shared memory.  Everything that touches CFR trees uses the large set: hypothetical games inside a tree do not end
// when a city jumps past seven districts (Game.is_last_round tests == 7, game/game.py:173-181) and run on for hundreds of
// steps (cities of 42, hands of 31, museums of 21 seen in 4096 random-ruleset trees of 200 iterations).
#ifdef CTD_SMALL_CAPS
#define CTD_HAND_CAP 48
#define CTD_BLD_CAP 32
#define CTD_MUS_CAP 32
#define CTD_JD_CAP 48
#elif !defined(CTD_HAND_CAP)
#define CTD_HAND_CAP 64
#define CTD_BLD_CAP 64
#define CTD_MUS_CAP 48
#define CTD_JD_CAP 48
#endif /* Smithy / Park draw into just_drawn_cards and nothing empties it until the next card pick: 33 seen in 5e5 classic games */
#define CTD_DECK_CAP 128 /* ring buffer, power of two */
#define CTD_DISC_CAP 128

enum { CTD_SUIT_TRADE = 0, CTD_SUIT_WAR, CTD_SUIT_RELIGION, CTD_SUIT_LORD, CTD_SUIT_UNIQUE };
enum { CTD_ROLE_NONE = 8, CTD_ROLE_BEWITCHED = 9 };
// role name id = rank*3 + variant (game/config.py:83-91)
enum {
  CTD_ASSASSIN = 0, CTD_WITCH, CTD_MAGISTRATE, CTD_THIEF, CTD_SPY, CTD_BLACKMAILER, CTD_MAGICIAN, CTD_WIZARD,
  CTD_SEER, CTD_KING, CTD_EMPEROR, CTD_PATRICIAN, CTD_BISHOP, CTD_ABBOT, CTD_CARDINAL, CTD_MERCHANT,
  CTD_ALCHEMIST, CTD_TRADER, CTD_ARCHITECT, CTD_NAVIGATOR, CTD_SCHOLAR, CTD_WARLORD, CTD_DIPLOMAT, CTD_MARSHAL,
  CTD_NAME_NONE, CTD_NAME_BEWITCHED
};
// option kinds = index in game/option.py:34-45
enum {
  CTD_K_ROLE_PICK = 0, CTD_K_GOLD_OR_CARD, CTD_K_KEEP, CTD_K_BLACKMAIL_RESPONSE, CTD_K_REVEAL_BLACKMAIL,
  CTD_K_REVEAL_WARRANT, CTD_K_BUILD, CTD_K_EMPTY, CTD_K_FINISH, CTD_K_GHOST_TOWN, CTD_K_SMITHY, CTD_K_LAB,
  CTD_K_MAGIC_SCHOOL, CTD_K_WEAPON_STORAGE, CTD_K_LIGHTHOUSE, CTD_K_MUSEUM, CTD_K_GRAVEYARD, CTD_K_TAKE_GOLD_WAR,
  CTD_K_ASSASSINATION, CTD_K_MAGISTRATE_WARRANT, CTD_K_BEWITCHING, CTD_K_STEAL, CTD_K_BLACKMAIL, CTD_K_SPY,
  CTD_K_MAGIC_HAND_CHANGE, CTD_K_DISCARD_AND_DRAW, CTD_K_LOOK_AT_HAND, CTD_K_TAKE_FROM_HAND, CTD_K_SEER,
  CTD_K_GIVE_BACK_CARD, CTD_K_TAKE_CROWN_KING, CTD_K_GIVE_CROWN, CTD_K_TAKE_CROWN_PAT, CTD_K_BISHOP,
  CTD_K_CARDINAL, CTD_K_ABBOT, CTD_K_ABBOT_BEG, CTD_K_MERCHANT, CTD_K_ALCHEMIST, CTD_K_TRADER, CTD_K_ARCHITECT,
  CTD_K_NAVIGATOR, CTD_K_SCHOLAR, CTD_K_SCHOLAR_PICK, CTD_K_WARLORD, CTD_K_MARSHAL, CTD_K_DIPLOMAT
};
// named choices, game/option.py:69-83
enum { CTD_N_GOLD = 0, CTD_N_CARD, CTD_N_PAY, CTD_N_NOT_PAY, CTD_N_REVEAL, CTD_N_NOT_REVEAL, CTD_N_4GOLD, CTD_N_4CARD,
       CTD_N_TRADE };
// already_done_moves flags
enum { CTD_DM_SMITHY = 1, CTD_DM_LAB = 2, CTD_DM_MAGIC_SCHOOL = 4, CTD_DM_MUSEUM = 8, CTD_DM_CHARACTER = 16,
       CTD_DM_BEGGED = 32, CTD_DM_TAKE_GOLD = 64 };
enum { CTD_NEXT_NONE = 0, CTD_NEXT_ALIAS, CTD_NEXT_RESET_CA, CTD_NEXT_EMPTY };
enum { CTD_PF_LIGHTHOUSE = 1, CTD_PF_FIRST7 = 2, CTD_PF_WITCH = 4 };
enum { CTD_RP_DEAD = 1, CTD_RP_WARRANT = 6, CTD_RP_POSSESSED = 8, CTD_RP_ROBBED = 16, CTD_RP_BLACKMAIL = 96 };

// ------------------------------------------------------------------------------------------ card tables
// game/config.py:2-80.  Tables are folded into immediates so neither host nor device needs memory for them.
CTD_HD inline int ctd_ctype(int c) { return c >= 40 ? 25 : c; }
CTD_HD inline int ctd_suit_of_type(int t) { return (t >= 6) + (t >= 10) + (t >= 13) + (t >= 16); }
CTD_HD inline int ctd_csuit(int c) { return c >= 40 ? c - 40 : ctd_suit_of_type(c); }
CTD_HD inline int ctd_cost_of_type(int t) {
  // 3 bits per type: 1,2,4,2,5,3,2,3,5,1,2,3,1,4,3,5,5,3,6,2,6 | 5,5,6,5,6,6,3,6,3,5,5,6,5,4,6,5,4,0,5
  const uint64_t lo = 1ull | 2ull << 3 | 4ull << 6 | 2ull << 9 | 5ull << 12 | 3ull << 15 | 2ull << 18 | 3ull << 21 |
                      5ull << 24 | 1ull << 27 | 2ull << 30 | 3ull << 33 | 1ull << 36 | 4ull << 39 | 3ull << 42 |
                      5ull << 45 | 5ull << 48 | 3ull << 51 | 6ull << 54 | 2ull << 57 | 6ull << 60;
  const uint64_t hi = 5ull | 5ull << 3 | 6ull << 6 | 5ull << 9 | 6ull << 12 | 6ull << 15 | 3ull << 18 | 6ull << 21 |
                      3ull << 24 | 5ull << 27 | 5ull << 30 | 6ull << 33 | 5ull << 36 | 4ull << 39 | 6ull << 42 |
                      5ull << 45 | 4ull << 48 | 0ull << 51 | 5ull << 54;
  return (int)((t < 21 ? lo >> (3 * t) : hi >> (3 * (t - 21))) & 7);
}
CTD_HD inline int ctd_ccost(int c) { return ctd_cost_of_type(ctd_ctype(c)); }
// i-th card of building_cards + unique_building_cards in list order (game/config.py:2-80)
CTD_HD inline int ctd_base_deck(int i) {
  // copies of types 0..15: 5,3,3,4,2,3,3,3,2,3,3,3,3,4,5,3  -> cumulative ends
  const uint8_t ends[16] = {5, 8, 11, 15, 17, 20, 23, 26, 28, 31, 34, 37, 40, 44, 49, 52};
  if (i < 52) {
    int t = 0;
    CTD_LOOP while (i >= ends[t]) ++t;
    return t;
  }
  i -= 52;  // uniques: 16,17,17,18,...,37,39
  if (i == 0) return 16;
  if (i <= 2) return 17;
  if (i == 23) return 39;
  return 15 + i;
}

// ------------------------------------------------------------------------------------------ descriptors
CTD_HD inline uint64_t ctd_opt(int kind, int perp) { return (uint64_t)kind | ((uint64_t)perp << 6); }
CTD_HD inline uint64_t ctd_f_target(int q) { return (uint64_t)(q + 1) << 9; }
CTD_HD inline uint64_t ctd_f_a(int t) { return (uint64_t)(t + 1) << 12; }
CTD_HD inline uint64_t ctd_f_b(int t) { return (uint64_t)(t + 1) << 18; }
CTD_HD inline uint64_t ctd_f_rank(int r) { return (uint64_t)(r + 1) << 24; }
CTD_HD inline uint64_t ctd_f_named(int n) { return (uint64_t)(n + 1) << 28; }
CTD_HD inline uint64_t ctd_f_replica(int r) { return (uint64_t)(r & 0xF) << 32; }
CTD_HD inline uint64_t ctd_f_build(int b) { return (uint64_t)(b & 1) << 36; }
CTD_HD inline uint64_t ctd_f_next_witch(int b) { return (uint64_t)(b & 1) << 37; }
CTD_HD inline uint64_t ctd_f_crown(int b) { return (uint64_t)(b & 1) << 38; }
CTD_HD inline uint64_t ctd_f_count(int c) { return (uint64_t)(c & 0x3F) << 39; }
CTD_HD inline uint64_t ctd_f_r(int r) { return (uint64_t)(r & 0x3F) << 45; }
CTD_HD inline uint64_t ctd_f_j(uint32_t j) { return (uint64_t)(j & 0x3FF) << 51; }

// ------------------------------------------------------------------------------------------ working record
struct alignas(16) CtdWork {
  uint8_t hand[6][CTD_HAND_CAP];
  uint8_t bld[6][CTD_BLD_CAP];
  uint8_t mus[6][CTD_MUS_CAP];
  uint8_t jd[6][CTD_JD_CAP];
  uint8_t deck[CTD_DECK_CAP];  // ring: element i is deck[(deck_head + i) & 127]
  uint8_t disc[CTD_DISC_CAP];
  int32_t gold[6];     // Agent.gold: a Python int in the reference; in run-away hypothetical games inside CFR trees a robbed
                       // seat that is sampled as the Thief doubles its own purse every round (11114 seen in 200 iterations)
  int16_t points[6];   // Game.points at terminal (a 32-district city scores far beyond a signed byte)
  uint8_t n_hand[6], n_bld[6], n_mus[6], n_jd[6];
  uint8_t deck_head, n_deck, n_disc;
  uint8_t role[6];
  int8_t replicas[6];
  uint8_t pflags[6];
  uint8_t rprops[8];
  uint8_t variant[8];
  uint8_t order[6];
  uint8_t used_roles[6];
  uint8_t used_len, rtc_mask, state, player, done, n_trade, n_nontrade, next_player, next_mode, crown, gflags;
  int8_t winner;
  uint8_t wiz_target;
  uint8_t warrant_building, ruleset, err;
  uint8_t seer_mask;   // game.seer_taken_card_from (seat order) as a mask
  uint8_t n_seven;     // game.seven_drawn_cards
  uint8_t seven[7];
  uint8_t snap_pad[10];
  // ---- everything above is the game itself: CTD_SNAP_BYTES, copied verbatim into MCCFR tree nodes ----
  uint8_t scratch[128];
  // chance: Philox4x32-10 keyed (seed, gid) or a recorded tape
  uint32_t k0, k1, g0, g1;
  uint32_t stream;  // Philox counter word 1: 0 = game chance, 1 = CFR tree
  uint32_t draws;
  uint32_t buf[4];
  uint32_t buf_blk;
  uint32_t* ring;     // unused; kept so that the kernels' shared-memory layout and code stay unchanged
  uint32_t ring_hi;
  const uint8_t* tape;
  uint32_t tape_pos, tape_len;
  uint32_t steps;
};

#define CTD_SNAP_BYTES (6 * (CTD_HAND_CAP + CTD_BLD_CAP + CTD_MUS_CAP + CTD_JD_CAP) + CTD_DECK_CAP + CTD_DISC_CAP + 144)
static_assert(offsetof(CtdWork, scratch) == CTD_SNAP_BYTES && CTD_SNAP_BYTES % 16 == 0, "CtdWork snapshot region");

// ------------------------------------------------------------------------------------------ chance
CTD_HD CTD_NI inline void ctd_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                              uint32_t out[4]) {
  CTD_LOOP for (int i = 0; i < 10; ++i) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

CTD_HD inline void ctd_chance_init(CtdWork& w, uint64_t seed, uint64_t gid, uint32_t draws) {
  w.k0 = (uint32_t)seed; w.k1 = (uint32_t)(seed >> 32);
  w.g0 = (uint32_t)gid; w.g1 = (uint32_t)(gid >> 32);
  w.draws = draws;
  w.stream = 0;
  w.buf_blk = 0xFFFFFFFFu;
  w.tape = nullptr; w.tape_pos = 0; w.tape_len = 0;
  w.ring = nullptr; w.ring_hi = 0;   // kept so that the kernels' code stays unchanged
}

CTD_HD inline uint32_t ctd_u32(CtdWork& w) {
  uint32_t blk = w.draws >> 2;
  if (blk != w.buf_blk) {
    ctd_philox(blk, w.stream, w.g0, w.g1, w.k0, w.k1, w.buf);
    w.buf_blk = blk;
  }
  return w.buf[w.draws++ & 3];
}
CTD_HD inline uint32_t ctd_randbelow(CtdWork& w, uint32_t n) { return (uint32_t)(((uint64_t)ctd_u32(w) * n) >> 32); }
// a chance draw that is part of the game itself (role variants, crown seat of a random game): one tape byte in replay mode
CTD_HD inline uint32_t ctd_randbelow_any(CtdWork& w, uint32_t n) {
  if (w.tape != nullptr) {
    if (w.tape_pos + 1 > w.tape_len) { w.err |= CTD_ERR_TAPE; return 0; }
    uint32_t v = w.tape[w.tape_pos++];
    if (v >= n) { w.err |= CTD_ERR_TAPE; v = 0; }
    return v;
  }
  return ctd_randbelow(w, n);
}

// Shuffle n elements addressed through `at(i)`.  Philox: Fisher-Yates from the top (the loop shape of
// CPython's random.shuffle); tape: new[k] = old[tape[k]].  n <= 1 consumes nothing.
template <class At>
CTD_HD inline void ctd_shuffle(CtdWork& w, int n, At at) {
  if (n <= 1) return;
  if (w.tape != nullptr) {
    if (w.tape_pos + (uint32_t)n > w.tape_len) { w.err |= CTD_ERR_TAPE; return; }
    CTD_LOOP for (int i = 0; i < n; ++i) w.scratch[i] = at(i);
    CTD_LOOP for (int i = 0; i < n; ++i) {
      int src = w.tape[w.tape_pos + i];
      if (src >= n) { w.err |= CTD_ERR_TAPE; src = 0; }
      at(i) = w.scratch[src];
    }
    w.tape_pos += n;
    return;
  }
  CTD_LOOP for (int i = n - 1; i > 0; --i) {
    int j = (int)ctd_randbelow(w, (uint32_t)(i + 1));
    uint8_t a = at(i), b = at(j);
    at(i) = b; at(j) = a;
  }
}


// every shuffle of a contiguous byte array goes through one out-of-line copy (the kernels pay for their instruction footprint)
#ifndef CTD_SHUFFLE_ATTR
#define CTD_SHUFFLE_ATTR CTD_NI
#endif
CTD_HD CTD_SHUFFLE_ATTR inline void ctd_shuffle_bytes(CtdWork& w, uint8_t* a, int n) {
  ctd_shuffle(w, n, [a](int i) -> uint8_t& { return a[i]; });
}

// ------------------------------------------------------------------------------------------ knowledge (CFR path)
// What one observer ("viewer") believes: Agent.known_roles / Agent.known_hands (game/agent.py:25-26,
// game/helper_classes.py:37-71), plus the looked-at hand of whoever used the Wizard this round
// (the HandKnowledge the state-10 enumerator reads, game/agent_functions.py:311).  Playouts do not carry it.
#define CTD_KN_HK_MAX 64 /* the Seer adds up to five one-card entries a round, each lives five rounds; with a Wizard, a Spy and a
                            Lighthouse at work as well, hypothetical games inside CFR trees were seen to pass 32 */
#define CTD_KN_POOL 256
#define CTD_KN_WIZ_CAP 48
enum { CTD_HK_WIZARD = 1, CTD_HK_USED = 2 };
struct CtdHK {           // one HandKnowledge in four bytes (bit 0 upwards: pid 4, conf 3, flags 2, n 8, off 9)
  int32_t pid : 4;       // -1 = the deck (Lighthouse)
  uint32_t conf : 3;     // 5..1, dropped at 0 (game/agent.py:100-109)
  uint32_t flags : 2;
  uint32_t n : 8;
  uint32_t off : 9;      // into pool
  uint32_t pad : 6;
};
static_assert(sizeof(CtdHK) == 4, "CtdHK layout");
struct alignas(16) CtdKnow {
  uint8_t viewer;
  uint8_t conf_mask;  // bit q: known_roles[*][q].confirmed (the same for every observer)
  uint8_t n_hk;
  uint8_t wiz_n;
  uint16_t kr[6];     // viewer's possible_roles per seat: bit r = rank r, bit 8 = "Bewitched"
  CtdHK hk[CTD_KN_HK_MAX];
  uint8_t wiz_cards[CTD_KN_WIZ_CAP];
  uint8_t pool[CTD_KN_POOL];
  uint16_t pool_used;
  uint8_t err;
  uint8_t pad[13];
};
static_assert(sizeof(CtdKnow) == 592, "CtdKnow layout");
struct CtdKnowSet {  // the observers being tracked: 1 (CFR viewer) or 6 (root generation); n == 0 in playouts
  CtdKnow* k;
  int n;
};

CTD_HD inline void ctd_kn_init(CtdKnow& k, int viewer) {
  uint8_t* raw = (uint8_t*)&k;
  CTD_LOOP for (int i = 0; i < (int)sizeof(CtdKnow); ++i) raw[i] = 0;
  k.viewer = (uint8_t)viewer;
}
// Agent.substract_from_known_hand_confidences_and_clear_wizard + reset_known_roles (game/agent.py:100-114)
CTD_HD CTD_NI inline void ctd_kn_setup_round(CtdKnow& k) {
  CTD_ASSUME_SHARED_K(&k);
  int keep = 0;
  uint16_t pos = 0;
  CTD_LOOP for (int i = 0; i < k.n_hk; ++i) {
    CtdHK h = k.hk[i];
    h.conf -= 1;
    h.flags = 0;
    if (h.conf != 0) {
      CTD_LOOP for (int j = 0; j < h.n; ++j) k.pool[pos + j] = k.pool[h.off + j];  // entries only move down
      h.off = pos;
      pos += h.n;
      k.hk[keep++] = h;
    }
  }
  CTD_LOOP for (int i = keep; i < k.n_hk; ++i) { CtdHK z = {}; k.hk[i] = z; }
  CTD_LOOP for (int j = pos; j < k.pool_used; ++j) k.pool[j] = 0;  // unused bytes stay zero (records compare bytewise)
  k.n_hk = (uint8_t)keep;
  k.pool_used = pos;
  CTD_LOOP for (int q = 0; q < 6; ++q) k.kr[q] = 0;
  k.conf_mask = 0;
  CTD_LOOP for (int j = 0; j < k.wiz_n; ++j) k.wiz_cards[j] = 0;
  k.wiz_n = 0;
}
CTD_HD CTD_NI inline void ctd_kn_add_hk(CtdKnow& k, int pid, const uint8_t* cards, int n, int ring_head, int ring_mask,
                                        bool wizard) {
  CTD_ASSUME_SHARED_K(&k);
  if (k.n_hk >= CTD_KN_HK_MAX || k.pool_used + n > CTD_KN_POOL) {
#ifdef CTD_HOST_DEBUG
    fprintf(stderr, "knowledge overflow: %d entries, pool %d + %d\n", (int)k.n_hk, (int)k.pool_used, n);
#endif
    k.err |= CTD_ERR_OVERFLOW; return; }
  CtdHK& h = k.hk[k.n_hk++];
  h.pid = pid; h.conf = 5; h.flags = wizard ? CTD_HK_WIZARD : 0; h.n = (uint32_t)n; h.off = k.pool_used; h.pad = 0;
  CTD_LOOP for (int i = 0; i < n; ++i) k.pool[k.pool_used + i] = cards[(ring_head + i) & ring_mask];
  k.pool_used += (uint16_t)n;
}
// remove the first card of type t from entry i (Deck.get_a_card_like_it on the HandKnowledge copy)
CTD_HD CTD_NI inline void ctd_kn_hk_remove(CtdKnow& k, int i, int t) {
  CTD_ASSUME_SHARED_K(&k);
  CtdHK& h = k.hk[i];
  CTD_LOOP for (int j = 0; j < h.n; ++j)
    if (ctd_ctype(k.pool[h.off + j]) == t) {
      CTD_LOOP for (int x = h.off + j; x + 1 < k.pool_used; ++x) k.pool[x] = k.pool[x + 1];
      --h.n;
      --k.pool_used;
      k.pool[k.pool_used] = 0;
      CTD_LOOP for (int e = i + 1; e < k.n_hk; ++e) k.hk[e].off -= 1;
      return;
    }
}
// confirm_role_knowledges (game/option_functions.py:608-622): every observer learns `seat`'s role;
// the filter on the other entries is a no-op (SURVEY.md A.5b)
CTD_HD inline void ctd_kn_confirm(CtdKnowSet ks, int seat, int role) {
  CTD_LOOP for (int i = 0; i < ks.n; ++i) {
    ks.k[i].kr[seat] = (uint16_t)(1u << (role == CTD_ROLE_BEWITCHED ? 8 : role));
    ks.k[i].conf_mask |= (uint8_t)(1u << seat);
  }
}

// ------------------------------------------------------------------------------------------ list helpers
CTD_HD CTD_NI inline bool ctd_has(const uint8_t* a, int n, int t) {
  CTD_LOOP for (int i = 0; i < n; ++i) if (ctd_ctype(a[i]) == t) return true;
  return false;
}
CTD_HD CTD_NI inline int ctd_count_type(const uint8_t* a, int n, int t) {
  int k = 0;
  CTD_LOOP for (int i = 0; i < n; ++i) k += ctd_ctype(a[i]) == t;
  return k;
}
CTD_HD CTD_NI inline int ctd_count_suit(const uint8_t* a, int n, int s) {
  int k = 0;
  CTD_LOOP for (int i = 0; i < n; ++i) k += ctd_csuit(a[i]) == s;
  return k;
}
CTD_HD inline int ctd_remove_at(uint8_t* a, uint8_t& n, int i) {
  int c = a[i];
  CTD_LOOP for (int k = i; k + 1 < n; ++k) a[k] = a[k + 1];
  --n;
  return c;
}
// Deck.get_a_card_like_it (game/deck.py:49-55): first card of that type; the requested card is fabricated
// when none matches.
CTD_HD CTD_NI inline int ctd_take_like(uint8_t* a, uint8_t& n, int t) {
  CTD_LOOP for (int i = 0; i < n; ++i)
    if (ctd_ctype(a[i]) == t) return ctd_remove_at(a, n, i);
  return t;
}
CTD_HD CTD_NI inline void ctd_append(CtdWork& w, uint8_t* a, uint8_t& n, int cap, int c) {
  CTD_ASSUME_WORK(&w);
  if (n >= cap) {
#ifdef CTD_HOST_DEBUG
    fprintf(stderr, "overflow cap %d list-offset %ld state %d\n", cap, (long)(a - (uint8_t*)&w), w.state);
#endif
    w.err |= CTD_ERR_OVERFLOW; return; }
  a[n++] = (uint8_t)c;
}
CTD_HD inline uint8_t& ctd_dk(CtdWork& w, int i) { return w.deck[(w.deck_head + i) & (CTD_DECK_CAP - 1)]; }
CTD_HD inline void ctd_deck_push(CtdWork& w, int c) {
  if (w.n_deck >= CTD_DECK_CAP - 1) {
#ifdef CTD_HOST_DEBUG
    fprintf(stderr, "deck overflow\n");
#endif
    w.err |= CTD_ERR_OVERFLOW; return; }
  ctd_dk(w, w.n_deck) = (uint8_t)c;
  ++w.n_deck;
}
CTD_HD inline void ctd_disc_push(CtdWork& w, int c) { ctd_append(w, w.disc, w.n_disc, CTD_DISC_CAP, c); }

// reshuffle_deck_if_empty (game/option_functions.py:564-570)
CTD_HD CTD_NI inline void ctd_reshuffle_if_empty(CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  if (w.n_deck == 0 && w.n_disc != 0) {
    uint8_t* d = w.disc;
    ctd_shuffle_bytes(w, d, w.n_disc);
    w.deck_head = 0;
    CTD_LOOP for (int i = 0; i < w.n_disc; ++i) w.deck[i] = w.disc[i];
    w.n_deck = w.n_disc;
    w.n_disc = 0;
  }
}
// reshuffle + draw_card; returns -1 for "Deck Empty" (game/deck.py:57-60), which add_card drops (:62-70)
CTD_HD CTD_NI inline int ctd_draw(CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  ctd_reshuffle_if_empty(w);
  if (w.n_deck == 0) return -1;
  int c = w.deck[w.deck_head];
  w.deck_head = (w.deck_head + 1) & (CTD_DECK_CAP - 1);
  --w.n_deck;
  return c;
}
CTD_HD inline void ctd_draw_to_hand(CtdWork& w, int p) {
  int c = ctd_draw(w);
  if (c >= 0) ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, c);
}
CTD_HD inline void ctd_draw_to_jd(CtdWork& w, int p) {
  int c = ctd_draw(w);
  if (c >= 0) ctd_append(w, w.jd[p], w.n_jd[p], CTD_JD_CAP, c);
}

CTD_HD inline int ctd_name(const CtdWork& w, int p) {
  int r = w.role[p];
  if (r < 8) return r * 3 + w.variant[r];
  return r == CTD_ROLE_NONE ? CTD_NAME_NONE : CTD_NAME_BEWITCHED;
}
// Game.get_player_from_role_id (game/game.py:403-412); -1 when nobody holds it
CTD_HD CTD_NI inline int ctd_player_from_rank(const CtdWork& w, int rank) {
  CTD_ASSUME_WORK(&w);
  int want = rank < 0 ? CTD_ROLE_BEWITCHED : rank;
  CTD_LOOP for (int p = 0; p < 6; ++p) if (w.role[p] == want) return p;
  return -1;
}
CTD_HD inline bool ctd_owns(const CtdWork& w, int p, int t) { return ctd_has(w.bld[p], w.n_bld[p], t); }
CTD_HD inline void ctd_clear_done(CtdWork& w) { w.done = 0; w.n_trade = 0; w.n_nontrade = 0; }

// ------------------------------------------------------------------------------------------ round machine
// Game.setup_round (game/game.py:144-171)
template <bool KN = true>
CTD_HD CTD_NI inline void ctd_setup_round(CtdWork& w, CtdKnowSet ks = CtdKnowSet{nullptr, 0}) {
  CTD_ASSUME_WORK(&w);
  CTD_LOOP for (int r = 0; r < 8; ++r) w.rprops[r] = 0;
  w.used_len = 0;
  CTD_LOOP for (int i = 0; i < 6; ++i) w.used_roles[i] = 0;
  // random.shuffle(list(roles.items())); with 6 players exactly one role is popped face down
  uint8_t* s = w.scratch + 64;
  CTD_LOOP for (int i = 0; i < 8; ++i) s[i] = (uint8_t)i;
  ctd_shuffle_bytes(w, s, 8);
  w.rtc_mask = (uint8_t)(0xFF & ~(1u << s[7]));
  // turn order rotates by the crowned seat's id, applied to the already rotated list
  int c = w.crown;
  uint8_t o[6];
  CTD_LOOP for (int i = 0; i < 6; ++i) o[i] = w.order[(i + c) % 6];
  CTD_LOOP for (int i = 0; i < 6; ++i) w.order[i] = o[i];
  w.state = 0;
  w.player = w.order[0];
  ctd_clear_done(w);
  w.next_mode = CTD_NEXT_NONE;
  w.next_player = 0;
  w.wiz_target = 0xFF;  // Agent.substract_from_known_hand_confidences_and_clear_wizard (game/agent.py:100-109)
  if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i) ctd_kn_setup_round(ks.k[i]);
}

// Game.refresh_used_roles (game/game.py:349-357); value+1 encoding keeps Bewitched (-1) sortable as 0
CTD_HD CTD_NI inline bool ctd_refresh_used_roles(CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  uint8_t v[6];
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    int r = w.role[p];
    if (r == CTD_ROLE_NONE) { w.err |= CTD_ERR_REF_RAISE; return false; }
    v[p] = (uint8_t)(r == CTD_ROLE_BEWITCHED ? 0 : r + 1);
  }
  CTD_LOOP for (int i = 1; i < 6; ++i) {  // insertion sort
    uint8_t x = v[i];
    int j = i - 1;
    CTD_LOOP while (j >= 0 && v[j] > x) { v[j + 1] = v[j]; --j; }
    v[j + 1] = x;
  }
  CTD_LOOP for (int i = 0; i < 6; ++i) w.used_roles[i] = v[i];
  w.used_len = 6;
  return true;
}

// Game.setup_next_player (game/game.py:391-401); current < 0 == None
CTD_HD CTD_NI inline void ctd_setup_next_player(CtdWork& w, int current) {
  CTD_ASSUME_WORK(&w);
  int nxt;
  if (w.state == 0) {
    if (!ctd_refresh_used_roles(w)) return;
    w.state = 1;
    nxt = ctd_player_from_rank(w, (int)w.used_roles[0] - 1);
  } else if (current >= 0) {
    w.state = 1;
    int r = w.role[current];
    if (r == CTD_ROLE_NONE) { w.err |= CTD_ERR_REF_RAISE; return; }
    uint8_t key = (uint8_t)(r == CTD_ROLE_BEWITCHED ? 0 : r + 1);
    int i = 0;
    CTD_LOOP while (i < w.used_len && w.used_roles[i] != key) ++i;
    if (i + 1 >= w.used_len) { w.err |= CTD_ERR_REF_RAISE; return; }
    nxt = ctd_player_from_rank(w, (int)w.used_roles[i + 1] - 1);
    ctd_clear_done(w);
  } else {
    w.err |= CTD_ERR_REF_RAISE;
    return;
  }
  if (nxt < 0) { w.err |= CTD_ERR_REF_RAISE; return; }
  w.player = (uint8_t)nxt;
}

// Agent.count_points (game/agent.py:116-143)
CTD_HD CTD_NI inline int ctd_count_points(const CtdWork& w, int p) {
  CTD_ASSUME_WORK(&w);
  int pts = 0;
  const uint8_t* b = w.bld[p];
  int n = w.n_bld[p];
  bool well = ctd_has(b, n, 31);
  CTD_LOOP for (int i = 0; i < n; ++i) {
    int t = ctd_ctype(b[i]);
    pts += ctd_cost_of_type(t);
    if (t == 18 || t == 23) pts += 2;
    if (well && ctd_csuit(b[i]) == CTD_SUIT_UNIQUE) pts += 1;
  }
  if (n >= 7) pts += 2;
  if (w.pflags[p] & CTD_PF_FIRST7) pts += 4;
  pts += w.n_mus[p];
  if (ctd_has(b, n, 37)) pts += w.gold[p];
  if (ctd_has(b, n, 39)) pts += w.n_hand[p];
  return pts;
}

// Game.check_game_ending (game/game.py:359-368): first arg-max wins
CTD_HD CTD_NI inline bool ctd_check_game_ending(CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  if (!(w.gflags & 1)) return false;
  int best = -1000, bi = 0;
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    int pts = ctd_count_points(w, p);
    w.points[p] = (int16_t)pts;
    if (pts > best) { best = pts; bi = p; }
  }
  w.gflags |= 2;
  w.winner = (int8_t)bi;
  return true;
}

// move_crown + troneroom_owner_gold (game/option_functions.py:625-631, :588-595)
CTD_HD CTD_NI inline void ctd_move_crown(CtdWork& w, int target) {
  CTD_ASSUME_WORK(&w);
  w.crown = (uint8_t)target;
  CTD_LOOP for (int p = 0; p < 6; ++p)
    if (ctd_owns(w, p, 32)) { w.gold[p] += 1; break; }
}

// Game.is_last_round (game/game.py:173-181)
CTD_HD inline void ctd_is_last_round(CtdWork& w) {
  if (w.gflags & 1) return;
  // runs after every carry_out: one flat test first, the per-seat loop only in the step that completes a city
  const bool any = (w.n_bld[0] == 7) | (w.n_bld[1] == 7) | (w.n_bld[2] == 7) | (w.n_bld[3] == 7) | (w.n_bld[4] == 7) |
                   (w.n_bld[5] == 7);
  if (!any) return;
  CTD_LOOP for (int p = 0; p < 6; ++p)
    if (w.n_bld[p] == 7) { w.gflags |= 1; w.pflags[p] |= CTD_PF_FIRST7; }
}

// Game.set_preset (game/game.py:420-489): Deck() shuffles the 76 cards, fixed hands are pulled by type
CTD_HD CTD_NI inline void ctd_deal_preset(CtdWork& w, int ruleset, uint8_t* used_cards_out = nullptr) {
  CTD_ASSUME_WORK(&w);
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    w.n_hand[p] = w.n_bld[p] = w.n_mus[p] = w.n_jd[p] = 0;
    w.gold[p] = 2; w.role[p] = CTD_ROLE_NONE; w.replicas[p] = 0; w.pflags[p] = 0;
    w.order[p] = (uint8_t)p; w.points[p] = 0; w.used_roles[p] = 0;
  }
  CTD_LOOP for (int r = 0; r < 8; ++r) w.rprops[r] = 0;
  const uint8_t preset_variant[8] = {1, 1, 1, 0, 1, 1, 1, 0};
  CTD_LOOP for (int r = 0; r < 8; ++r) w.variant[r] = ruleset == CTD_RULESET_PRESET ? preset_variant[r] : 0;
  w.used_len = 0; w.rtc_mask = 0; w.state = 0; w.player = 0xFF;
  ctd_clear_done(w);
  w.next_player = 0; w.next_mode = CTD_NEXT_NONE; w.crown = 3; w.gflags = 0; w.winner = -1;
  w.wiz_target = 0xFF; w.warrant_building = 0xFF; w.ruleset = (uint8_t)ruleset; w.err = 0; w.steps = 0;
  w.seer_mask = 0; w.n_seven = 0;
  CTD_LOOP for (int i = 0; i < 7; ++i) w.seven[i] = 0;
  w.n_disc = 0; w.deck_head = 0;
  if (ruleset == CTD_RULESET_RANDOM) {
    // Game.set_random_game (game/game.py:491-520): random.sample(uniques, 14) = first 14 of a 24-permutation, Deck()
    // shuffle of the 66 cards, four cards each dealt round-robin from the top, a random variant per rank, a shuffled
    // pick order, a random crown.
    uint8_t* u = w.scratch + 96;  // the tape form of ctd_shuffle stages through scratch[0, n): keep clear of it
    CTD_LOOP for (int i = 0; i < 24; ++i) u[i] = (uint8_t)i;
    ctd_shuffle_bytes(w, u, 24);
    CTD_LOOP for (int i = 0; i < 52; ++i) w.deck[i] = (uint8_t)ctd_base_deck(i);
    CTD_LOOP for (int i = 0; i < 14; ++i) w.deck[52 + i] = (uint8_t)ctd_base_deck(52 + u[i]);
    w.n_deck = 66;
    uint8_t* dk = w.deck;
    ctd_shuffle_bytes(w, dk, 66);
    if (used_cards_out != nullptr) {
      CTD_LOOP for (int i = 0; i < 76; ++i) used_cards_out[i] = i < 66 ? w.deck[i] : 0xFF;
    }
    CTD_LOOP for (int r = 0; r < 4; ++r)
      CTD_LOOP for (int p = 0; p < 6; ++p) w.hand[p][r] = w.deck[r * 6 + p];
    CTD_LOOP for (int p = 0; p < 6; ++p) w.n_hand[p] = 4;
    w.deck_head = 24;
    w.n_deck = 42;
    CTD_LOOP for (int r = 0; r < 8; ++r) w.variant[r] = (uint8_t)ctd_randbelow_any(w, 3);
    uint8_t* o = w.order;
    ctd_shuffle_bytes(w, o, 6);
    w.crown = (uint8_t)ctd_randbelow_any(w, 6);
    return;
  }
  CTD_LOOP for (int i = 0; i < 76; ++i) w.deck[i] = (uint8_t)ctd_base_deck(i);
  w.n_deck = 76;
  uint8_t* d = w.deck;
  ctd_shuffle_bytes(w, d, 76);
  if (used_cards_out != nullptr)  // self.used_cards = deepcopy(self.deck) (game/game.py:424)
    CTD_LOOP for (int i = 0; i < 76; ++i) used_cards_out[i] = w.deck[i];
  // The fixed hands ({0,0,16,17,18,19} {1,1,20,21,22,23} {2,3,24,25,26,27} {3,4,28,29,30,31} {4,0,32,33,34,35}
  // {0,1,36,37,39,0}) are pulled one card at a time with get_a_card_like_it (first match in the shuffled deck), seat
  // by seat.  The i-th request for type t therefore receives the i-th copy of t in deck order, so one pass over the
  // deck serves all 36 requests: slot = (seat << 3 | position in hand) of the next unserved request for that type.
  CTD_LOOP for (int p = 0; p < 6; ++p) w.n_hand[p] = 6;
  uint8_t served[5] = {0, 0, 0, 0, 0};
  const uint8_t slot_common[5][5] = {{0 << 3 | 0, 0 << 3 | 1, 4 << 3 | 1, 5 << 3 | 0, 5 << 3 | 5},
                                     {1 << 3 | 0, 1 << 3 | 1, 5 << 3 | 1, 0xFF, 0xFF},
                                     {2 << 3 | 0, 0xFF, 0xFF, 0xFF, 0xFF},
                                     {2 << 3 | 1, 3 << 3 | 0, 0xFF, 0xFF, 0xFF},
                                     {3 << 3 | 1, 4 << 3 | 0, 0xFF, 0xFF, 0xFF}};
  uint32_t unique_done = 0;  // bit (t - 16): the single request for unique type t has been served
  int out = 0;
  CTD_LOOP for (int j = 0; j < 76; ++j) {
    const int t = w.deck[j];
    int slot = 0xFF;
    if (t < 5) {
      if (served[t] < 5) { slot = slot_common[t][served[t]]; if (slot != 0xFF) ++served[t]; }
    } else if (t >= 16 && !((unique_done >> (t - 16)) & 1)) {
      unique_done |= 1u << (t - 16);
      const int u = t == 39 ? 22 : t - 16;  // 16,17,18..37,39 -> 0..22 (the second Keep is never requested)
      slot = ((u >> 2) << 3) | (2 + (u & 3));
    }
    if (slot != 0xFF) w.hand[slot >> 3][slot & 7] = (uint8_t)t;
    else w.deck[out++] = (uint8_t)t;
  }
  w.n_deck = (uint8_t)out;
}

// ------------------------------------------------------------------------------------------ enumeration
// Visitor that materialises options into a buffer and/or selects the `want`-th one.
struct CtdEmit {
  uint64_t* buf;
  uint32_t cap;
  uint32_t n;
  uint32_t want;
  uint64_t got;
  CTD_HD void one(uint64_t d) {
    if (n < cap) buf[n] = d;
    if (n == want) got = d;
    ++n;
  }
  // cnt options that differ only in the ordinal field j
  CTD_HD void range(uint64_t base, uint32_t cnt) {
    if (want >= n && want - n < cnt) got = base | ctd_f_j(want - n);
    CTD_LOOP for (uint32_t j = 0; j < cnt && n + j < cap; ++j) buf[n + j] = base | ctd_f_j(j);
    n += cnt;
  }
};

CTD_HD inline int ctd_build_limit(int name) {  // Agent.get_build_limit (game/agent.py:87-98)
  if (name == CTD_ARCHITECT) return 3;
  if (name == CTD_SCHOLAR) return 2;
  if (name == CTD_BISHOP || name == CTD_NAVIGATOR) return 0;
  return 1;
}
// cost as the enumerators see it: Factory (35) makes uniques dearer (game/agent_functions.py:113-114)
CTD_HD inline int ctd_build_cost(int c, bool factory) {
  return ctd_ccost(c) + ((factory && ctd_csuit(c) == CTD_SUIT_UNIQUE) ? 1 : 0);
}
CTD_HD inline uint64_t ctd_binom(int n, int r) {
  if (r > n - r) r = n - r;
  uint64_t v = 1;
  CTD_LOOP for (int i = 1; i <= r; ++i) v = v * (uint64_t)(n - r + i) / (uint64_t)i;
  return v;
}
// number of discard_and_draw options of subset size r for a hand of n (game/agent_functions.py:290-294):
// range(0, C, max(round(C/1e2), 1)) with CPython's round-half-even
CTD_HD CTD_NI inline uint32_t ctd_magician_count(int n, int r) {
  uint64_t c = ctd_binom(n, r);
  uint64_t q = c / 100, rem = c % 100;
  uint64_t step = rem > 50 ? q + 1 : (rem < 50 ? q : q + (q & 1));
  if (step < 1) step = 1;
  return (uint32_t)((c + step - 1) / step);
}

// ---- deluxe characters (tier C) ----
#define CTD_N_NOTHING 13 /* give_crown's "nothing": descriptor only, not in the reference's names table */

// emperor_options (game/agent_functions.py:368-382)
template <class E>
CTD_HD CTD_NI inline void ctd_emperor_options(const CtdWork& w, int p, bool dead, E& e) {
  CTD_ASSUME_WORK(&w);
  CTD_LOOP for (int q = 0; q < 6; ++q) {
    if (q == p) continue;
    const uint64_t base = ctd_opt(CTD_K_GIVE_CROWN, p) | ctd_f_target(q);
    if (w.n_hand[q] != 0 && !dead) e.one(base | ctd_f_named(CTD_N_CARD));
    if (w.gold[q] != 0 && !dead) e.one(base | ctd_f_named(CTD_N_GOLD));
    if ((w.gold[q] == 0 && w.n_hand[q] == 0) || dead) e.one(base | ctd_f_named(CTD_N_NOTHING));
  }
}

// cardinal_options (game/agent_functions.py:393-419): for every seat (own included) and every hand card the seat can
// "afford", the combinations of (gold - cost) other cards to hand over, thinned to about a hundred per card
template <class E>
CTD_HD CTD_NI inline void ctd_cardinal_options(const CtdWork& w, int p, E& e) {
  CTD_ASSUME_WORK(&w);
  const uint8_t* hand = w.hand[p];
  const int nh = w.n_hand[p];
  uint64_t own = 0;
  CTD_LOOP for (int i = 0; i < w.n_bld[p]; ++i) own |= 1ull << ctd_ctype(w.bld[p][i]);
  const bool factory_owned = (own >> 35) & 1;
  CTD_LOOP for (int q = 0; q < 6; ++q)
    CTD_LOOP for (int i = 0; i < nh; ++i) {
      const int c = hand[i], t = ctd_ctype(c);
      const bool factory = factory_owned && ctd_csuit(c) == CTD_SUIT_UNIQUE;
      const int cost = ctd_ccost(c) + (factory ? 1 : 0);
      const int replica = (((own >> t) & 1) && !w.replicas[p]) ? w.replicas[p] + 1 : 0;
      if (cost > w.gold[q]) continue;
      const int ex = w.gold[q] - cost;
      if (nh - 1 < ex) continue;
      int n_other = 0;
      CTD_LOOP for (int x = 0; x < nh; ++x) n_other += ctd_ctype(hand[x]) != t;
      if (ex > n_other) continue;
      const uint64_t total = ctd_binom(n_other, ex);
      const uint64_t qd = total / 100, rem = total % 100;
      uint64_t step = rem > 50 ? qd + 1 : (rem < 50 ? qd : qd + (qd & 1));
      if (step < 1) step = 1;
      const uint32_t cnt = (uint32_t)((total + step - 1) / step);
      e.range(ctd_opt(CTD_K_CARDINAL, p) | ctd_f_target(q) | ctd_f_a(t) | ctd_f_replica(replica) | ctd_f_build(factory) | ctd_f_count(ex), cnt);
    }
}

// seer_give_back_card (game/agent_functions.py:332-361).  The enumeration itself draws chance: for every position,
// every hand card and three times over it shuffles the other cards (cumulatively) and takes the first k-1.
template <class E>
CTD_HD CTD_NI inline void ctd_seer_give_back_options(CtdWork& w, int p, E& e) {
  CTD_ASSUME_WORK(&w);
  int k = 0;
  CTD_LOOP for (int q = 0; q < 6; ++q) k += (w.seer_mask >> q) & 1;
  const int n = w.n_hand[p];
  uint8_t* rem = w.scratch + 64;  // <= 48 cards; the tape form of ctd_shuffle stages through scratch[0, n <= 48)
  CTD_LOOP for (int pos = 0; pos < k; ++pos)
    CTD_LOOP for (int ci = 0; ci < n; ++ci) {
      const int card = w.hand[p][ci], tc = ctd_ctype(card);
      int nr = 0;
      CTD_LOOP for (int x = 0; x < n; ++x)
        if (ctd_ctype(w.hand[p][x]) != tc) rem[nr++] = w.hand[p][x];
      CTD_LOOP for (int rep = 0; rep < 3; ++rep) {
        ctd_shuffle_bytes(w, rem, nr);
        // row = rem[:k-1] with the card inserted at `pos` (list.insert past the end appends); zip() stops at k
        int take = nr < k - 1 ? nr : k - 1;
        int ins = pos < take ? pos : take;
        uint64_t d = ctd_opt(CTD_K_GIVE_BACK_CARD, p);
        const int shift[5] = {12, 18, 39, 45, 51};
        int out = 0;
        CTD_LOOP for (int x = 0; x <= take && out < k && out < 5; ++x) {
          if (x == ins) { d |= (uint64_t)(tc + 1) << shift[out++]; if (out >= k || out >= 5) break; }
          if (x < take) d |= (uint64_t)(ctd_ctype(rem[x]) + 1) << shift[out++];
        }
        e.one(d);
      }
    }
}

// scholar_give_back_options (game/agent_functions.py:462-470).  copy() is shallow, so the reference removes from the
// very list it iterates: every call shrinks seven_drawn_cards, and every option shares what is left.
template <class E>
CTD_HD CTD_NI inline void ctd_scholar_give_back_options(CtdWork& w, int p, E& e) {
  CTD_ASSUME_WORK(&w);
  int i = 0;
  while (i < w.n_seven) {
    const int t = ctd_ctype(w.seven[i]);
    ctd_take_like(w.seven, w.n_seven, t);
    e.one(ctd_opt(CTD_K_SCHOLAR_PICK, p) | ctd_f_a(t));
    ++i;
  }
}

// character_options (game/agent_functions.py:156-209) and the per-role enumerators it dispatches to
template <class E>
CTD_HD CTD_NI inline void ctd_character_options(const CtdWork& w, int p, int nm, E& e) {
  CTD_ASSUME_WORK(&w);
  if (!(w.done & CTD_DM_CHARACTER)) {
    switch (nm) {
      case CTD_ASSASSIN: CTD_NOT_PRESET();  // :213-218
        CTD_LOOP for (int r = 1; r < 8; ++r) e.one(ctd_opt(CTD_K_ASSASSINATION, p) | ctd_f_rank(r));
        break;
      case CTD_THIEF: CTD_NOT_PRESET();  // :246-253
        CTD_LOOP for (int r = 2; r < 8; ++r) e.one(ctd_opt(CTD_K_STEAL, p) | ctd_f_rank(r));
        break;
      case CTD_SPY: CTD_NOT_CLASSIC();  // :274-281
        CTD_LOOP for (int q = 0; q < 6; ++q)
          if (q != p)
            CTD_LOOP for (int s = 0; s < 5; ++s) e.one(ctd_opt(CTD_K_SPY, p) | ctd_f_target(q) | ctd_f_named(CTD_N_TRADE + s));
        break;
      case CTD_MAGICIAN: CTD_NOT_PRESET(); {  // :284-296
        CTD_LOOP for (int q = 0; q < 6; ++q)
          if (q != p) e.one(ctd_opt(CTD_K_MAGIC_HAND_CHANGE, p) | ctd_f_target(q));
        int n = w.n_hand[p];
        CTD_LOOP for (int r = 1; r <= n; ++r) e.range(ctd_opt(CTD_K_DISCARD_AND_DRAW, p) | ctd_f_r(r), ctd_magician_count(n, r));
        break;
      }
      case CTD_WIZARD: CTD_NOT_CLASSIC();  // :298-308
        CTD_LOOP for (int q = 0; q < 6; ++q)
          if (q != p && w.n_hand[q] > 0) e.one(ctd_opt(CTD_K_LOOK_AT_HAND, p) | ctd_f_target(q));
        break;
      case CTD_KING: e.one(ctd_opt(CTD_K_TAKE_CROWN_KING, p)); break;  // :364-366
      case CTD_BISHOP: CTD_NOT_PRESET(); e.one(ctd_opt(CTD_K_BISHOP, p)); break;         // :389-391
      case CTD_ABBOT: CTD_NOT_CLASSIC(); {                                                // :422-430
        int n = ctd_count_suit(w.hand[p], w.n_hand[p], CTD_SUIT_RELIGION);
        if (n > 0)
          CTD_LOOP for (int k = 0; k <= n; ++k) e.one(ctd_opt(CTD_K_ABBOT, p) | ctd_f_count(k) | ctd_f_r(n));
        break;
      }
      case CTD_MERCHANT: CTD_NOT_PRESET(); e.one(ctd_opt(CTD_K_MERCHANT, p)); break;    // :438-440
      case CTD_ALCHEMIST: CTD_NOT_CLASSIC(); break;                                       // :442-444
      case CTD_ARCHITECT: CTD_NOT_PRESET(); e.one(ctd_opt(CTD_K_ARCHITECT, p)); break;  // :451-452
      case CTD_NAVIGATOR: CTD_NOT_CLASSIC();                                              // :454-455
        e.one(ctd_opt(CTD_K_NAVIGATOR, p) | ctd_f_named(CTD_N_4GOLD));
        e.one(ctd_opt(CTD_K_NAVIGATOR, p) | ctd_f_named(CTD_N_4CARD));
        break;
      case CTD_WARLORD:  // :473-482
        CTD_LOOP for (int q = 0; q < 6; ++q) {
          if (w.n_bld[q] >= 7 || ctd_name(w, q) == CTD_BISHOP) continue;
          uint64_t seen = 0;
          CTD_LOOP for (int i = 0; i < w.n_bld[q]; ++i) {
            int c = w.bld[q][i], t = ctd_ctype(c);
            if (ctd_ccost(c) - 1 <= w.gold[p] && t != 17 && !((seen >> t) & 1)) {
              seen |= 1ull << t;
              e.one(ctd_opt(CTD_K_WARLORD, p) | ctd_f_target(q) | ctd_f_a(t));
            }
          }
        }
        break;
      case CTD_MAGISTRATE: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // :221-234  real target x pairs of fake targets among ranks 1..7
        CTD_LOOP for (int real = 1; real < 8; ++real)
          CTD_LOOP for (int a = 1; a < 8; ++a)
            CTD_LOOP for (int b = a + 1; b < 8; ++b)
              if (real != a && real != b)
                e.one(ctd_opt(CTD_K_MAGISTRATE_WARRANT, p) | ctd_f_rank(real) | ctd_f_named(a) | ctd_f_count(b));
        break;
      case CTD_BLACKMAILER: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // :255-272  ordered pairs of un-possessed ranks 2..7
        CTD_LOOP for (int a = 2; a < 8; ++a) {
          if (w.rprops[a] & CTD_RP_POSSESSED) continue;
          CTD_LOOP for (int b = a + 1; b < 8; ++b) {
            if (w.rprops[b] & CTD_RP_POSSESSED) continue;
            e.one(ctd_opt(CTD_K_BLACKMAIL, p) | ctd_f_rank(a) | ctd_f_named(b));
            e.one(ctd_opt(CTD_K_BLACKMAIL, p) | ctd_f_rank(b) | ctd_f_named(a));
          }
        }
        break;
      case CTD_SEER: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); e.one(ctd_opt(CTD_K_SEER, p)); break;            // :328-329
      case CTD_EMPEROR: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); ctd_emperor_options(w, p, false, e); break;   // :368-382
      case CTD_PATRICIAN: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); e.one(ctd_opt(CTD_K_TAKE_CROWN_PAT, p)); break;  // :384-386
      case CTD_CARDINAL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); ctd_cardinal_options(w, p, e); break;        // :393-419
      case CTD_TRADER: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); e.one(ctd_opt(CTD_K_TRADER, p)); break;        // :446-448
      case CTD_SCHOLAR: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); if (w.n_deck != 0) e.one(ctd_opt(CTD_K_SCHOLAR, p)); break;  // :457-460
      case CTD_MARSHAL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // :484-492
        CTD_LOOP for (int q = 0; q < 6; ++q) {
          if (q == p || w.n_bld[q] >= 7 || ctd_name(w, q) == CTD_BISHOP) continue;
          uint64_t seen = 0;
          CTD_LOOP for (int i = 0; i < w.n_bld[q]; ++i) {
            const int c = w.bld[q][i], t = ctd_ctype(c), cost = ctd_ccost(c);
            if (cost <= w.gold[p] && cost <= 3 && !ctd_owns(w, p, t) && t != 17 && !((seen >> t) & 1)) {
              seen |= 1ull << t;
              e.one(ctd_opt(CTD_K_MARSHAL, p) | ctd_f_target(q) | ctd_f_a(t));
            }
          }
        }
        break;
      case CTD_DIPLOMAT: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // :494-504
        CTD_LOOP for (int q = 0; q < 6; ++q) {
          if (q == p || w.n_bld[q] >= 7 || ctd_name(w, q) == CTD_BISHOP) continue;
          CTD_LOOP for (int i = 0; i < w.n_bld[q]; ++i) {
            const int te = ctd_ctype(w.bld[q][i]);
            if (te == 17 || ctd_owns(w, p, te)) continue;
            CTD_LOOP for (int j = 0; j < w.n_bld[p]; ++j) {
              const int to = ctd_ctype(w.bld[p][j]);
              if (ctd_cost_of_type(te) - ctd_cost_of_type(to) > w.gold[p]) continue;
              // de-duplicate on (target, taken type, given type): any earlier pair of the same types in this city
              bool dup = false;
              CTD_LOOP for (int i2 = 0; i2 <= i && !dup; ++i2) {
                if (ctd_ctype(w.bld[q][i2]) != te) continue;
                const int jmax = i2 == i ? j : w.n_bld[p];
                CTD_LOOP for (int j2 = 0; j2 < jmax && !dup; ++j2) dup = ctd_ctype(w.bld[p][j2]) == to;
              }
              if (!dup) e.one(ctd_opt(CTD_K_DIPLOMAT, p) | ctd_f_target(q) | ctd_f_a(te) | ctd_f_b(to));
            }
          }
        }
        break;
      default: break;
    }
  }
  if (nm == CTD_ABBOT && !(w.done & CTD_DM_BEGGED)) e.one(ctd_opt(CTD_K_ABBOT_BEG, p));  // :199-202
  if ((nm == CTD_WARLORD || nm == CTD_MARSHAL || nm == CTD_DIPLOMAT) && !(w.done & CTD_DM_TAKE_GOLD))
    e.one(ctd_opt(CTD_K_TAKE_GOLD_WAR, p));  // :204-207
}

// main_round_options (game/agent_functions.py:133-147); concatenation order is observable
template <class E>
CTD_HD CTD_NI inline void ctd_main_round_options(const CtdWork& w, int p, int nm, E& e) {
  CTD_ASSUME_WORK(&w);
  const uint8_t* bld = w.bld[p];
  const int nb = w.n_bld[p];
  const uint8_t* hand = w.hand[p];
  const int nh = w.n_hand[p];
  // which effect buildings do I own
  uint64_t own = 0;
  CTD_LOOP for (int i = 0; i < nb; ++i) own |= 1ull << ctd_ctype(bld[i]);
  // build_options / get_builds (:108-130)
  {
    int built = nm == CTD_TRADER ? w.n_nontrade : w.n_trade + w.n_nontrade;
    if (built < ctd_build_limit(nm)) {
      bool factory = (own >> 35) & 1;
      uint64_t seen = 0;
      CTD_LOOP for (int i = 0; i < nh; ++i) {
        int c = hand[i], t = ctd_ctype(c);
        int replica = (((own >> t) & 1) && !w.replicas[p]) ? w.replicas[p] + 1 : 0;
        if (ctd_build_cost(c, factory) <= w.gold[p] && !((seen >> t) & 1)) {
          seen |= 1ull << t;
          e.one(ctd_opt(CTD_K_BUILD, p) | ctd_f_a(t) | ctd_f_replica(replica));
        }
      }
    }
  }
  ctd_character_options(w, p, nm, e);
  if (((own >> 21) & 1) && w.gold[p] >= 2 && !(w.done & CTD_DM_SMITHY)) e.one(ctd_opt(CTD_K_SMITHY, p));  // :54-57
  if (((own >> 22) & 1) && !(w.done & CTD_DM_LAB))                                                      // :59-65
    CTD_LOOP for (int i = 0; i < nh; ++i) e.one(ctd_opt(CTD_K_LAB, p) | ctd_f_a(ctd_ctype(hand[i])));
  if (!(w.done & CTD_DM_MAGIC_SCHOOL) && ((own >> 25) & 1))                                             // :67-74
    CTD_LOOP for (int s = 0; s < 5; ++s) e.one(ctd_opt(CTD_K_MAGIC_SCHOOL, p) | ctd_f_named(CTD_N_TRADE + s));
  if ((own >> 27) & 1)                                                                                  // :76-83
    CTD_LOOP for (int q = 0; q < 6; ++q)
      if (q != p)
        CTD_LOOP for (int i = 0; i < w.n_bld[q]; ++i)
          e.one(ctd_opt(CTD_K_WEAPON_STORAGE, p) | ctd_f_target(q) | ctd_f_a(ctd_ctype(w.bld[q][i])));
  if (((own >> 29) & 1) && (w.pflags[p] & CTD_PF_LIGHTHOUSE)) {                                          // :85-94
    uint64_t seen = 0;
    CTD_LOOP for (int i = 0; i < w.n_deck; ++i) {
      int t = ctd_ctype(w.deck[(w.deck_head + i) & (CTD_DECK_CAP - 1)]);
      if (!((seen >> t) & 1)) { seen |= 1ull << t; e.one(ctd_opt(CTD_K_LIGHTHOUSE, p) | ctd_f_a(t)); }
    }
  }
  if (((own >> 34) & 1) && !(w.done & CTD_DM_MUSEUM)) {                                                  // :96-105
    uint64_t seen = 0;
    CTD_LOOP for (int i = 0; i < nh; ++i) {
      int t = ctd_ctype(hand[i]);
      if (!((seen >> t) & 1)) { seen |= 1ull << t; e.one(ctd_opt(CTD_K_MUSEUM, p) | ctd_f_a(t)); }
    }
  }
  e.one(ctd_opt(CTD_K_FINISH, p));
}

// wizard_take_from_hand_options (game/agent_functions.py:310-326).  `cards` is the looked-at hand copy
// (HandKnowledge.hand); in a playout it equals the target's current hand.  `replica` leaks across iterations.
template <class E>
CTD_HD CTD_NI inline void ctd_wizard_take_options(const CtdWork& w, int p, const uint8_t* cards, int n, E& e) {
  CTD_ASSUME_WORK(&w);
  int q = w.wiz_target;
  uint64_t own = 0;
  CTD_LOOP for (int i = 0; i < w.n_bld[p]; ++i) own |= 1ull << ctd_ctype(w.bld[p][i]);
  bool factory = (own >> 35) & 1;
  uint64_t seen_take = 0, seen_b0 = 0, seen_b1 = 0;
  int replica = 0;
  uint32_t before = e.n;
  CTD_LOOP for (int i = 0; i < n; ++i) {
    int c = cards[i], t = ctd_ctype(c);
    if (!((seen_take >> t) & 1)) {
      seen_take |= 1ull << t;
      e.one(ctd_opt(CTD_K_TAKE_FROM_HAND, p) | ctd_f_target(q) | ctd_f_a(t));
    }
    if ((own >> t) & 1) replica = w.replicas[p] + 1;
    uint64_t& seen = replica == 0 ? seen_b0 : seen_b1;
    if (ctd_build_cost(c, factory) <= w.gold[p] && !((seen >> t) & 1)) {
      seen |= 1ull << t;
      e.one(ctd_opt(CTD_K_TAKE_FROM_HAND, p) | ctd_f_target(q) | ctd_f_a(t) | ctd_f_build(1) | ctd_f_replica(replica));
    }
  }
  if (e.n == before) e.one(ctd_opt(CTD_K_EMPTY, p));
}

// Agent.get_options (game/agent.py:50-83).  An empty result with err set means the reference would raise.
template <class E>
CTD_HD CTD_NI inline void ctd_enumerate(CtdWork& w, E& e, const CtdKnow* kn = nullptr) {
  CTD_ASSUME_WORK(&w);
  if (w.gflags & 2) return;  // terminal: the reference's loops stop here
  const int p = w.player;
  const int st = w.state;
  if (p >= 6) { w.err |= CTD_ERR_REF_RAISE; return; }
  if (st == 0) {  // pick_role_options (game/agent_functions.py:13-14)
    CTD_LOOP for (int r = 0; r < 8; ++r)
      if ((w.rtc_mask >> r) & 1) e.one(ctd_opt(CTD_K_ROLE_PICK, p) | ctd_f_rank(r));
    return;
  }
  const int role = w.role[p];
  if (role == CTD_ROLE_NONE) { w.err |= CTD_ERR_REF_RAISE; return; }
  const int nm = ctd_name(w, p);
  const bool king = nm == CTD_KING || nm == CTD_PATRICIAN;
  if (role == CTD_ROLE_BEWITCHED || !(w.rprops[role] & CTD_RP_DEAD)) {
    switch (st) {
      case 1:  // gold_or_card_options (:16-17)
        e.one(ctd_opt(CTD_K_GOLD_OR_CARD, p) | ctd_f_named(CTD_N_GOLD));
        if (w.n_deck > 1) e.one(ctd_opt(CTD_K_GOLD_OR_CARD, p) | ctd_f_named(CTD_N_CARD));
        return;
      case 2: {  // which_card_to_keep_options (:19-33)
        const uint8_t* jd = w.jd[p];
        int n = w.n_jd[p];
        if (ctd_owns(w, p, 20)) {
          CTD_LOOP for (int i = 0; i < n; ++i)
            CTD_LOOP for (int j = i + 1; j < n; ++j)
              e.one(ctd_opt(CTD_K_KEEP, p) | ctd_f_a(ctd_ctype(jd[i])) | ctd_f_b(ctd_ctype(jd[j])));
        } else {
          uint64_t seen = 0;
          CTD_LOOP for (int i = 0; i < n; ++i) {
            int t = ctd_ctype(jd[i]);
            if (!((seen >> t) & 1)) { seen |= 1ull << t; e.one(ctd_opt(CTD_K_KEEP, p) | ctd_f_a(t)); }
          }
        }
        return;
      }
      case 3:  // blackmail_response_options (:35-38)
        if (role == CTD_ROLE_BEWITCHED) { w.err |= CTD_ERR_REF_RAISE; return; }
        if (w.rprops[role] & CTD_RP_BLACKMAIL) {
          CTD_NOT_PRESET(); CTD_NOT_CLASSIC();
          e.one(ctd_opt(CTD_K_BLACKMAIL_RESPONSE, p) | ctd_f_named(CTD_N_PAY));
          e.one(ctd_opt(CTD_K_BLACKMAIL_RESPONSE, p) | ctd_f_named(CTD_N_NOT_PAY));
        } else {
          e.one(ctd_opt(CTD_K_EMPTY, p));
        }
        return;
      case 6:  // graveyard_options (:150-153)
        e.one(ctd_opt(w.gold[p] > 0 ? CTD_K_GRAVEYARD : CTD_K_EMPTY, p));
        return;
      case 4:  // reveal_blackmail_as_blackmailer_options (:40-41)
        CTD_NOT_PRESET(); CTD_NOT_CLASSIC();
        e.one(ctd_opt(CTD_K_REVEAL_BLACKMAIL, p) | ctd_f_target(w.next_player) | ctd_f_named(CTD_N_REVEAL));
        e.one(ctd_opt(CTD_K_REVEAL_BLACKMAIL, p) | ctd_f_target(w.next_player) | ctd_f_named(CTD_N_NOT_REVEAL));
        return;
      case 7:  // reveal_warrant_as_magistrate_options (:43-44)
        CTD_NOT_PRESET(); CTD_NOT_CLASSIC();
        e.one(ctd_opt(CTD_K_REVEAL_WARRANT, p) | ctd_f_target(w.next_player) | ctd_f_named(CTD_N_REVEAL));
        e.one(ctd_opt(CTD_K_REVEAL_WARRANT, p) | ctd_f_target(w.next_player) | ctd_f_named(CTD_N_NOT_REVEAL));
        return;
      default: break;
    }
    if (nm == CTD_WITCH) {  // witch_options (:236-242)
      CTD_LOOP for (int r = 1; r < 8; ++r) e.one(ctd_opt(CTD_K_BEWITCHING, p) | ctd_f_rank(r));
      return;
    }
    if (role == CTD_ROLE_BEWITCHED) { w.err |= CTD_ERR_REF_RAISE; return; }
    if (!(w.rprops[role] & CTD_RP_POSSESSED)) {
      if (st == 5) {
        ctd_main_round_options(w, p, nm, e);
        return;
      }
      if (st == 8) { CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); ctd_seer_give_back_options(w, p, e); return; }
      if (st == 9) { CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); ctd_scholar_give_back_options(w, p, e); return; }
      if (st == 10) {
        int q = w.wiz_target;
        if (q >= 6) { w.err |= CTD_ERR_REF_RAISE; return; }
        if (kn != nullptr) ctd_wizard_take_options(w, p, kn->wiz_cards, kn->wiz_n, e);
        else ctd_wizard_take_options(w, p, w.hand[q], w.n_hand[q], e);
        return;
      }
      w.err |= CTD_ERR_REF_RAISE;  // the reference falls off its if-chain and returns None
      return;
    }
    e.one(ctd_opt(CTD_K_FINISH, p) | ctd_f_next_witch(1) | ctd_f_crown(king));
    return;
  }
  if (nm == CTD_EMPEROR && !(w.done & CTD_DM_CHARACTER)) { CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); ctd_emperor_options(w, p, true, e); return; }
  e.one(ctd_opt(CTD_K_FINISH, p) | ctd_f_crown(king));
}

// ------------------------------------------------------------------------------------------ transition
CTD_HD inline void ctd_to5(CtdWork& w, int p) { w.state = 5; w.player = (uint8_t)p; }

// game.gamestate = game.gamestate.next_gamestate (SURVEY.md A.3)
CTD_HD inline void ctd_restore_next(CtdWork& w) {
  if (w.next_mode == CTD_NEXT_NONE) { w.err |= CTD_ERR_REF_RAISE; return; }
  w.state = 5;
  w.player = w.next_player;
  if (w.next_mode == CTD_NEXT_RESET_CA) { ctd_clear_done(w); w.done = CTD_DM_CHARACTER; }
  else if (w.next_mode == CTD_NEXT_EMPTY) ctd_clear_done(w);
  w.next_mode = CTD_NEXT_NONE;
  w.next_player = 0;
}

// carry_out_building (game/option_functions.py:102-127)
CTD_HD CTD_NI inline void ctd_apply_build(CtdWork& w, int p, int t, int replica) {
  CTD_ASSUME_WORK(&w);
  int c = ctd_take_like(w.hand[p], w.n_hand[p], t);
  ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, c);
  if (ctd_name(w, p) != CTD_ALCHEMIST) w.gold[p] -= (int32_t)ctd_ccost(c);
  if (replica) w.replicas[p] = (int8_t)replica;
  if (ctd_csuit(c) == CTD_SUIT_TRADE) { if (w.n_trade < 15) ++w.n_trade; }
  else { if (w.n_nontrade < 15) ++w.n_nontrade; }
  if (t == 29) w.pflags[p] |= CTD_PF_LIGHTHOUSE;
  int r = w.role[p];
  if (r >= 8) { w.err |= CTD_ERR_REF_RAISE; return; }
  if (!(w.rprops[r] & CTD_RP_WARRANT)) {
    ctd_to5(w, p);
  } else {  // :121-127 any warrant, real or fake, interrupts for the Magistrate
    int m = ctd_player_from_rank(w, 0);
    if (m < 0) { w.err |= CTD_ERR_REF_RAISE; return; }
    w.warrant_building = (uint8_t)t;
    w.state = 7;
    w.player = (uint8_t)m;
    w.next_player = (uint8_t)p;
    w.next_mode = CTD_NEXT_ALIAS;
  }
}

// finish_main_sequnce_actions (game/option_functions.py:189-243).  Returns true when the game ended.
template <bool KN>
CTD_HD CTD_NI inline bool ctd_apply_finish(CtdWork& w, uint64_t d, CtdKnowSet ks) {
  CTD_ASSUME_WORK(&w);
  const int p = CTD_OPT_PERP(d);
  const int pr = w.role[p];
  if (pr >= 8) { w.err |= CTD_ERR_REF_RAISE; return false; }
  const bool dead = w.rprops[pr] & CTD_RP_DEAD;
  if (!dead && w.n_hand[p] == 0) {
    uint64_t own = 0;
    CTD_LOOP for (int i = 0; i < w.n_bld[p]; ++i) own |= 1ull << ctd_ctype(w.bld[p][i]);
    if ((own >> 28) & 1) { ctd_draw_to_jd(w, p); ctd_draw_to_jd(w, p); }  // Park: into just_drawn_cards
    if ((own >> 30) & 1) w.gold[p] += 1;                                  // Poorhouse
  }
  if (CTD_OPT_CROWN(d)) { if (KN) ctd_kn_confirm(ks, p, pr); ctd_move_crown(w, p); }
  else if (KN && dead) ctd_kn_confirm(ks, p, pr);
  if (CTD_OPT_NEXT_WITCH(d)) {  // :211-230 the witch takes over the possessed role
    int wi = ctd_player_from_rank(w, 0);
    if (wi < 0) { w.err |= CTD_ERR_REF_RAISE; return false; }
    w.state = 5;
    w.player = (uint8_t)wi;
    w.role[wi] = (uint8_t)pr;
    w.rprops[pr] &= (uint8_t)~CTD_RP_POSSESSED;
    w.role[p] = CTD_ROLE_BEWITCHED;
    if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i) {  // :222-226
      CtdKnow& k = ks.k[i];
      if (k.viewer != wi) k.kr[wi] = (uint16_t)(1u << pr);
      if (k.viewer != p) k.kr[p] = (uint16_t)(1u << 8);
    }
    ctd_clear_done(w);
    return false;
  }
  if (w.used_len == 0) { w.err |= CTD_ERR_REF_RAISE; return false; }
  if ((int)w.used_roles[w.used_len - 1] - 1 == pr) {  // last player of the round
    if (ctd_check_game_ending(w)) return true;
    ctd_setup_round<KN>(w, ks);
  } else {
    ctd_setup_next_player(w, p);
  }
  return false;
}

// option.carry_out (game/option.py:118-122).  Returns true when this step ended the game.
// KN = false instantiates the transition without the knowledge bookkeeping (the playout kernel: smaller image).
template <bool KN = true>
CTD_HD CTD_NI inline bool ctd_apply(CtdWork& w, uint64_t d, CtdKnowSet ks = CtdKnowSet{nullptr, 0}) {
  CTD_ASSUME_WORK(&w);
  const int k = CTD_OPT_KIND(d);
  const int p = CTD_OPT_PERP(d);
  bool won = false;
  switch (k) {
    case CTD_K_ROLE_PICK: {  // carry_out_role_pick (:6-30)
      int r = CTD_OPT_RANK(d);
      w.role[p] = (uint8_t)r;
      w.rtc_mask &= (uint8_t)~(1u << r);
      if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i) {  // only the picker's beliefs are written (:11-25)
        CtdKnow& k = ks.k[i];
        if (k.viewer != p) continue;
        int me = 0;
        while (me < 5 && w.order[me] != p) ++me;
        CTD_LOOP for (int oi = 0; oi < 6; ++oi) {
          int q = w.order[oi];
          if (q == p) continue;
          k.kr[q] = oi < me ? (uint16_t)(0xFF & ~w.rtc_mask & ~(1u << r)) : (uint16_t)w.rtc_mask;
        }
      }
      if (p != w.order[5]) {
        int i = 0;
        CTD_LOOP while (i < 5 && w.order[i] != p) ++i;
        w.state = 0;
        w.player = w.order[i + 1];
      } else {
        ctd_setup_next_player(w, -1);
      }
      break;
    }
    case CTD_K_GOLD_OR_CARD: {  // carry_out_gold_or_card (:33-55)
      int r = w.role[p];
      if (r == CTD_ROLE_NONE) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (KN) ctd_kn_confirm(ks, p, r);  // confirm_role_knowledges (:35)
      if (r >= 8) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (w.rprops[r] & CTD_RP_ROBBED) {
        int th = ctd_player_from_rank(w, 1);
        if (th < 0) { w.err |= CTD_ERR_REF_RAISE; break; }
        int g = w.gold[p];
        w.gold[th] += (int32_t)g;  // thief may be p itself only if p holds rank 1, which is never robbed by itself
        w.gold[p] = (int32_t)(th == p ? g : 0);
        if (th == p) w.gold[p] = 0;
      }
      if (CTD_OPT_NAMED(d) == CTD_N_GOLD) {
        w.gold[p] += 2;
        w.state = 3;
      } else {
        int n = ctd_owns(w, p, 16) ? 3 : 2;  // Observatory
        CTD_LOOP for (int i = 0; i < n; ++i) ctd_draw_to_jd(w, p);
        w.state = 2;
      }
      w.player = (uint8_t)p;
      break;
    }
    case CTD_K_KEEP: {  // carry_out_put_back_card (:58-66)
      int c = ctd_take_like(w.jd[p], w.n_jd[p], CTD_OPT_CARD_A(d));
      ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, c);
      if (CTD_OPT_CARD_B(d) >= 0) {
        c = ctd_take_like(w.jd[p], w.n_jd[p], CTD_OPT_CARD_B(d));
        ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, c);
      }
      CTD_LOOP for (int i = 0; i < w.n_jd[p]; ++i) ctd_deck_push(w, w.jd[p][i]);
      w.n_jd[p] = 0;
      w.state = 3;
      w.player = (uint8_t)p;
      break;
    }
    case CTD_K_EMPTY:  // carry_out_empty (:68-69); producers: agent_functions.py:38, :153, :325
      if (w.state == 3) {
        ctd_to5(w, p);
        ctd_clear_done(w);
        w.next_mode = CTD_NEXT_NONE;
        w.next_player = 0;
      } else {
        ctd_restore_next(w);
      }
      break;
    case CTD_K_BUILD: ctd_apply_build(w, p, CTD_OPT_CARD_A(d), CTD_OPT_REPLICA(d)); break;
    case CTD_K_FINISH: won = ctd_apply_finish<KN>(w, d, ks); break;
    case CTD_K_SMITHY:  // carry_out_smithy (:131-138): the cards go to just_drawn_cards
      w.gold[p] -= 2;
      CTD_LOOP for (int i = 0; i < 3; ++i) ctd_draw_to_jd(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_SMITHY;
      break;
    case CTD_K_LAB:  // carry_out_laboratory (:140-145)
      ctd_disc_push(w, ctd_take_like(w.hand[p], w.n_hand[p], CTD_OPT_CARD_A(d)));
      w.gold[p] += 1;
      ctd_to5(w, p);
      w.done |= CTD_DM_LAB;
      break;
    case CTD_K_MAGIC_SCHOOL: {  // carry_out_magic_school (:147-153): removed and re-appended with the new suit
      ctd_take_like(w.bld[p], w.n_bld[p], 25);
      int s = CTD_OPT_NAMED(d) - CTD_N_TRADE;
      ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, s == CTD_SUIT_UNIQUE ? 25 : 40 + s);
      ctd_to5(w, p);
      w.done |= CTD_DM_MAGIC_SCHOOL;
      break;
    }
    case CTD_K_MUSEUM:  // carry_out_museum (:161-165)
      ctd_append(w, w.mus[p], w.n_mus[p], CTD_MUS_CAP, ctd_take_like(w.hand[p], w.n_hand[p], CTD_OPT_CARD_A(d)));
      ctd_to5(w, p);
      w.done |= CTD_DM_MUSEUM;
      break;
    case CTD_K_WEAPON_STORAGE: {  // carry_out_weapon_storage (:167-171)
      int q = CTD_OPT_TARGET(d);
      ctd_disc_push(w, ctd_take_like(w.bld[p], w.n_bld[p], 27));
      ctd_disc_push(w, ctd_take_like(w.bld[q], w.n_bld[q], CTD_OPT_CARD_A(d)));
      ctd_to5(w, p);
      break;
    }
    case CTD_K_LIGHTHOUSE: {  // carry_out_lighthouse (:173-180)
      int t = CTD_OPT_CARD_A(d), c = t, n = w.n_deck;
      if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i)  // HandKnowledge(player_id=-1, hand=deepcopy(deck)) (:174)
        if (ks.k[i].viewer == p) ctd_kn_add_hk(ks.k[i], -1, w.deck, n, w.deck_head, CTD_DECK_CAP - 1, false);
      CTD_LOOP for (int i = 0; i < n; ++i)
        if (ctd_ctype(ctd_dk(w, i)) == t) {
          c = ctd_dk(w, i);
          CTD_LOOP for (int k = i; k + 1 < n; ++k) ctd_dk(w, k) = ctd_dk(w, k + 1);
          --w.n_deck;
          break;
        }
      ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, c);
      w.pflags[p] &= (uint8_t)~CTD_PF_LIGHTHOUSE;
      CtdWork* wp = &w;
      ctd_shuffle(w, w.n_deck, [wp](int i) -> uint8_t& { return ctd_dk(*wp, i); });
      ctd_to5(w, p);
      break;
    }
    case CTD_K_GRAVEYARD:  // carry_out_graveyard (:183-187): pops the LAST discard
      if (w.n_disc == 0) { w.err |= CTD_ERR_REF_RAISE; break; }
      ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, w.disc[--w.n_disc]);
      w.gold[p] -= 1;
      ctd_restore_next(w);
      break;
    case CTD_K_TAKE_GOLD_WAR:  // carry_out_take_gold_for_war (:553-559)
      w.gold[p] += (int32_t)ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_WAR);
      ctd_to5(w, p);
      w.done |= CTD_DM_TAKE_GOLD;
      break;
    case CTD_K_ASSASSINATION: CTD_NOT_PRESET();  // carry_out_assasination (:245-249)
      w.rprops[CTD_OPT_RANK(d)] |= CTD_RP_DEAD;
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_STEAL: CTD_NOT_PRESET();  // carry_out_stealing (:265-269)
      w.rprops[CTD_OPT_RANK(d)] |= CTD_RP_ROBBED;
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_BEWITCHING: CTD_NOT_CLASSIC();  // carry_out_bewitching (:259-262)
      w.rprops[CTD_OPT_RANK(d)] |= CTD_RP_POSSESSED;
      w.pflags[p] |= CTD_PF_WITCH;
      ctd_setup_next_player(w, p);
      break;
    case CTD_K_SPY: CTD_NOT_CLASSIC(); {  // carry_out_spying (:278-288)
      int q = CTD_OPT_TARGET(d), s = CTD_OPT_NAMED(d) - CTD_N_TRADE;
      int n = ctd_count_suit(w.hand[q], w.n_hand[q], s);
      int steal = n < w.gold[q] ? n : w.gold[q];
      w.gold[p] += (int32_t)steal;
      w.gold[q] -= (int32_t)steal;
      ctd_draw_to_hand(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_MAGIC_HAND_CHANGE: CTD_NOT_PRESET(); {  // carry_out_magicking (:291-293)
      int q = CTD_OPT_TARGET(d);
      int n = w.n_hand[p] > w.n_hand[q] ? w.n_hand[p] : w.n_hand[q];
      CTD_LOOP for (int i = 0; i < n; ++i) { uint8_t a = w.hand[p][i]; w.hand[p][i] = w.hand[q][i]; w.hand[q][i] = a; }
      uint8_t a = w.n_hand[p]; w.n_hand[p] = w.n_hand[q]; w.n_hand[q] = a;
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_DISCARD_AND_DRAW: CTD_NOT_PRESET(); {  // carry_out_magicking (:295-300): ignores the option's cards and removes
                                    // while iterating; draws as many cards as are left in hand
      int i = 0;
      CTD_LOOP while (i < w.n_hand[p]) {
        int t = ctd_ctype(w.hand[p][i]);
        ctd_deck_push(w, ctd_take_like(w.hand[p], w.n_hand[p], t));
        ++i;
      }
      int n = w.n_hand[p];
      CTD_LOOP for (int k = 0; k < n; ++k) ctd_draw_to_hand(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_LOOK_AT_HAND: CTD_NOT_CLASSIC();  // carry_out_wizard_hand_looking (:305-310)
      if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i) {
        CtdKnow& k = ks.k[i];
        int q = CTD_OPT_TARGET(d), n = w.n_hand[q];
        if (n > CTD_KN_WIZ_CAP) { k.err |= CTD_ERR_OVERFLOW; n = CTD_KN_WIZ_CAP; }
        CTD_LOOP for (int j = 0; j < CTD_KN_WIZ_CAP; ++j) k.wiz_cards[j] = j < n ? w.hand[q][j] : 0;
        k.wiz_n = (uint8_t)n;
        if (k.viewer == p) ctd_kn_add_hk(k, q, w.hand[q], w.n_hand[q], 0, 0xFFFF, true);
      }
      w.wiz_target = (uint8_t)CTD_OPT_TARGET(d);
      w.state = 10;
      w.player = (uint8_t)p;
      w.done |= CTD_DM_CHARACTER;
      w.next_player = (uint8_t)p;
      w.next_mode = CTD_NEXT_ALIAS;
      break;
    case CTD_K_TAKE_FROM_HAND: CTD_NOT_CLASSIC(); {  // carry_out_wizard_take_from_hand (:312-328)
      int q = CTD_OPT_TARGET(d), t = CTD_OPT_CARD_A(d);
      ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, ctd_take_like(w.hand[q], w.n_hand[q], t));
      if (CTD_OPT_BUILD(d)) ctd_apply_build(w, p, t, ctd_count_type(w.bld[p], w.n_bld[p], t));
      if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i) {  // the looked-at copy loses the card too (:320, :326)
        CtdKnow& k = ks.k[i];
        CTD_LOOP for (int j = 0; j < k.wiz_n; ++j)
          if (ctd_ctype(k.wiz_cards[j]) == t) {
            CTD_LOOP for (int x = j; x + 1 < k.wiz_n; ++x) k.wiz_cards[x] = k.wiz_cards[x + 1];
            --k.wiz_n;
            k.wiz_cards[k.wiz_n] = 0;
            break;
          }
        if (k.viewer == p)
          CTD_LOOP for (int h = 0; h < k.n_hk; ++h)
            if (k.hk[h].flags & CTD_HK_WIZARD) { ctd_kn_hk_remove(k, h, t); break; }
      }
      ctd_restore_next(w);
      break;
    }
    case CTD_K_TAKE_CROWN_KING:  // carry_out_take_crown_king (:354-363)
      w.gold[p] += (int32_t)ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_LORD);
      if (!(w.pflags[p] & CTD_PF_WITCH)) ctd_move_crown(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_BISHOP: CTD_NOT_PRESET();  // carry_out_bishop (:397-403)
      w.gold[p] += (int32_t)ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_RELIGION);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_MERCHANT: CTD_NOT_PRESET();  // carry_out_merchant (:442-449)
      w.gold[p] += (int32_t)(ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_TRADE) + 1);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_ABBOT: CTD_NOT_CLASSIC(); {  // carry_out_abbot (:405-412)
      int n = CTD_OPT_R(d), kc = CTD_OPT_COUNT(d);  // the option carries its own gold/card list
      w.gold[p] += (int32_t)(n - kc);
      CTD_LOOP for (int i = 0; i < kc; ++i) ctd_draw_to_hand(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_ABBOT_BEG: CTD_NOT_CLASSIC(); {  // carry_out_abbot_beg (:414-420): first richest seat pays, may be the abbot
      int rich = 0;
      CTD_LOOP for (int q = 1; q < 6; ++q) if (w.gold[q] > w.gold[rich]) rich = q;
      w.gold[rich] -= 1;
      int a = ctd_player_from_rank(w, 4);
      if (a < 0) { w.err |= CTD_ERR_REF_RAISE; break; }
      w.gold[a] += 1;
      ctd_to5(w, p);
      w.done |= CTD_DM_BEGGED;
      break;
    }
    case CTD_K_ARCHITECT: CTD_NOT_PRESET();  // carry_out_architect (:464-471)
      ctd_draw_to_hand(w, p);
      ctd_draw_to_hand(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_NAVIGATOR: CTD_NOT_CLASSIC();  // carry_out_navigator (:473-483)
      if (CTD_OPT_NAMED(d) == CTD_N_4CARD) CTD_LOOP for (int i = 0; i < 4; ++i) ctd_draw_to_hand(w, p);
      else w.gold[p] += 4;
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_WARLORD: {  // carry_out_warlord (:517-535) with settle_museum / settle_lighthouse (:573-586)
      int q = CTD_OPT_TARGET(d), t = CTD_OPT_CARD_A(d);
      int c = ctd_take_like(w.bld[q], w.n_bld[q], t);
      w.gold[p] -= (int32_t)(ctd_ccost(c) - 1);
      ctd_disc_push(w, c);
      if (ctd_count_type(w.bld[q], w.n_bld[q], t) > 1) w.replicas[q] -= 1;
      if (t == 34) {
        CTD_LOOP for (int i = 0; i < w.n_mus[q]; ++i) ctd_disc_push(w, w.mus[q][i]);
        w.n_mus[q] = 0;
      }
      if (t == 29 && (w.pflags[q] & CTD_PF_LIGHTHOUSE)) {
        w.pflags[q] &= (uint8_t)~CTD_PF_LIGHTHOUSE;
        w.pflags[p] |= CTD_PF_LIGHTHOUSE;
      }
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      int owner = -1;  // get_graveyard_owner (:597-601)
      CTD_LOOP for (int x = 0; x < 6; ++x) if (ctd_owns(w, x, 24)) { owner = x; break; }
      if (owner >= 0 && owner != p) {
        w.state = 6;
        w.player = (uint8_t)owner;
        w.next_player = (uint8_t)p;
        w.next_mode = CTD_NEXT_RESET_CA;  // GameState(..., already_done_moves=["character_ability"]) (:535)
      }
      break;
    }
    // ---- deluxe characters (tier C) ----
    case CTD_K_MAGISTRATE_WARRANT: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // carry_out_warranting (:251-257)
      w.rprops[CTD_OPT_RANK(d)] = (uint8_t)((w.rprops[CTD_OPT_RANK(d)] & ~CTD_RP_WARRANT) | (1 << 1));
      w.rprops[CTD_OPT_NAMED(d)] = (uint8_t)((w.rprops[CTD_OPT_NAMED(d)] & ~CTD_RP_WARRANT) | (2 << 1));
      w.rprops[CTD_OPT_COUNT(d)] = (uint8_t)((w.rprops[CTD_OPT_COUNT(d)] & ~CTD_RP_WARRANT) | (2 << 1));
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_REVEAL_WARRANT: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_magistrate_reaveal (:94-100)
      const int q = CTD_OPT_TARGET(d), rq = w.role[q];
      if (rq >= 8) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (CTD_OPT_NAMED(d) == CTD_N_REVEAL && ((w.rprops[rq] & CTD_RP_WARRANT) >> 1) == 1) {
        const int t = w.warrant_building;
        ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, ctd_take_like(w.bld[q], w.n_bld[q], t));
        w.gold[q] += (int32_t)ctd_cost_of_type(t);
        CTD_LOOP for (int r = 0; r < 8; ++r) w.rprops[r] &= (uint8_t)~CTD_RP_WARRANT;
      }
      ctd_restore_next(w);
      break;
    }
    case CTD_K_BLACKMAIL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // carry_out_blackmail (:271-276)
      w.rprops[CTD_OPT_RANK(d)] = (uint8_t)((w.rprops[CTD_OPT_RANK(d)] & ~CTD_RP_BLACKMAIL) | (1 << 5));
      w.rprops[CTD_OPT_NAMED(d)] = (uint8_t)((w.rprops[CTD_OPT_NAMED(d)] & ~CTD_RP_BLACKMAIL) | (2 << 5));
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_BLACKMAIL_RESPONSE: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_respond_to_blackmail (:71-82); int(gold/2) truncates toward zero
      const int bm = ctd_player_from_rank(w, 1);
      if (bm < 0) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (CTD_OPT_NAMED(d) == CTD_N_PAY) {
        const int half = w.gold[p] / 2;
        w.gold[bm] += (int32_t)half;
        w.gold[p] -= (int32_t)half;
        ctd_to5(w, p);
      } else {
        w.state = 4;
        w.player = (uint8_t)bm;
        w.next_player = (uint8_t)p;
        w.next_mode = CTD_NEXT_EMPTY;
      }
      break;
    }
    case CTD_K_REVEAL_BLACKMAIL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_responding_to_blackmail_response (:85-92)
      const int q = CTD_OPT_TARGET(d), rq = w.role[q];
      if (rq >= 8) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (CTD_OPT_NAMED(d) == CTD_N_REVEAL && ((w.rprops[rq] & CTD_RP_BLACKMAIL) >> 5) == 1) {
        w.gold[p] += w.gold[q];
        w.gold[q] = 0;
        CTD_LOOP for (int r = 0; r < 8; ++r) w.rprops[r] &= (uint8_t)~CTD_RP_BLACKMAIL;
      }
      ctd_restore_next(w);
      break;
    }
    case CTD_K_SEER: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_seer_take_a_card (:330-341): shuffle each hand, take its first card
      w.seer_mask = 0;
      CTD_LOOP for (int q = 0; q < 6; ++q) {
        if (q == p || w.n_hand[q] == 0) continue;
        uint8_t* h = w.hand[q];
        ctd_shuffle_bytes(w, h, w.n_hand[q]);
        ctd_reshuffle_if_empty(w);
        ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, ctd_remove_at(w.hand[q], w.n_hand[q], 0));
        w.seer_mask |= (uint8_t)(1u << q);
      }
      w.state = 8;
      w.player = (uint8_t)p;
      w.done |= CTD_DM_CHARACTER;
      w.next_player = (uint8_t)p;
      w.next_mode = CTD_NEXT_ALIAS;
      break;
    }
    case CTD_K_GIVE_BACK_CARD: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_seer_give_back_cards (:343-350)
      const int shift[5] = {12, 18, 39, 45, 51};
      int idx = 0;
      CTD_LOOP for (int q = 0; q < 6 && idx < 5; ++q) {
        if (!((w.seer_mask >> q) & 1)) continue;
        const int tv = (int)((d >> shift[idx++]) & 0x3F);
        if (tv == 0) break;  // zip() ran out of cards
        const int c = ctd_take_like(w.hand[p], w.n_hand[p], tv - 1);
        ctd_append(w, w.hand[q], w.n_hand[q], CTD_HAND_CAP, c);
        if (KN) CTD_LOOP for (int i = 0; i < ks.n; ++i)
          if (ks.k[i].viewer == p) { uint8_t cc = (uint8_t)c; ctd_kn_add_hk(ks.k[i], q, &cc, 1, 0, 0xFFFF, false); }
      }
      w.seer_mask = 0;
      ctd_restore_next(w);
      break;
    }
    case CTD_K_GIVE_CROWN: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_emperor (:377-393)
      const int q = CTD_OPT_TARGET(d);
      w.gold[p] += (int32_t)ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_LORD);
      if (CTD_OPT_NAMED(d) == CTD_N_CARD) {
        uint8_t* h = w.hand[q];
        ctd_shuffle_bytes(w, h, w.n_hand[q]);
        if (w.n_hand[q] != 0) ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, ctd_remove_at(w.hand[q], w.n_hand[q], 0));
      } else if (CTD_OPT_NAMED(d) == CTD_N_GOLD) {
        w.gold[p] += 1;
        w.gold[q] -= 1;
      }
      if (w.role[p] == CTD_ROLE_NONE) { w.err |= CTD_ERR_REF_RAISE; break; }
      if (KN) ctd_kn_confirm(ks, p, w.role[p]);
      ctd_move_crown(w, q);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_TAKE_CROWN_PAT: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_take_crown_patrician (:365-375)
      const int n = ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_LORD);
      CTD_LOOP for (int i = 0; i < n; ++i) ctd_draw_to_hand(w, p);
      if (!(w.pflags[p] & CTD_PF_WITCH)) ctd_move_crown(w, p);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_CARDINAL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_cardinal (:422-439): no build bookkeeping, no warrant check, gold clamped at 0
      const int q = CTD_OPT_TARGET(d), t = CTD_OPT_CARD_A(d), kc = CTD_OPT_COUNT(d);
      const int c = ctd_take_like(w.hand[p], w.n_hand[p], t);
      ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, c);
      int g = w.gold[p] - (ctd_ccost(c) - CTD_OPT_BUILD(d));
      w.gold[p] = (int32_t)(g < 0 ? 0 : g);
      if (CTD_OPT_REPLICA(d)) w.replicas[p] = (int8_t)CTD_OPT_REPLICA(d);
      if (kc != 0) {
        w.gold[q] -= (int32_t)kc;
        // other_cards = hand without the built type, in hand order; hand over the (j * step)-th kc-combination
        uint8_t* other = w.scratch;
        int no = 0;
        CTD_LOOP for (int x = 0; x < w.n_hand[p]; ++x)
          if (ctd_ctype(w.hand[p][x]) != t) other[no++] = w.hand[p][x];
        const uint64_t total = ctd_binom(no, kc);
        const uint64_t qd = total / 100, rem = total % 100;
        uint64_t step = rem > 50 ? qd + 1 : (rem < 50 ? qd : qd + (qd & 1));
        if (step < 1) step = 1;
        uint64_t idx = (uint64_t)CTD_OPT_J(d) * step;
        int x = 0;
        CTD_LOOP for (int r = kc; r > 0; --r) {  // unrank in itertools.combinations order
          for (;;) {
            const uint64_t cnt = ctd_binom(no - x - 1, r - 1);
            if (idx < cnt) break;
            idx -= cnt;
            ++x;
            if (x >= no) break;
          }
          if (x >= no) { w.err |= CTD_ERR_REF_RAISE; break; }
          ctd_append(w, w.hand[q], w.n_hand[q], CTD_HAND_CAP, ctd_take_like(w.hand[p], w.n_hand[p], ctd_ctype(other[x])));
          ++x;
        }
      }
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    case CTD_K_TRADER: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // carry_out_trader (:455-461)
      w.gold[p] += (int32_t)ctd_count_suit(w.bld[p], w.n_bld[p], CTD_SUIT_TRADE);
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    case CTD_K_SCHOLAR: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_scholar_draw (:485-496)
      w.n_seven = 0;
      const int n = w.n_deck < 7 ? w.n_deck : 7;
      CTD_LOOP for (int i = 0; i < n; ++i) {
        const int c = ctd_draw(w);
        if (c < 0) break;
        ctd_append(w, w.hand[p], w.n_hand[p], CTD_HAND_CAP, c);
        w.seven[w.n_seven++] = (uint8_t)c;
      }
      w.state = 9;
      w.player = (uint8_t)p;
      w.done |= CTD_DM_CHARACTER;
      w.next_player = (uint8_t)p;
      w.next_mode = CTD_NEXT_ALIAS;
      break;
    }
    case CTD_K_SCHOLAR_PICK: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();  // carry_out_scholar_put_back (:498-502): returns what the shrunk shared list still holds
      CTD_LOOP for (int i = 0; i < w.n_seven; ++i) ctd_deck_push(w, ctd_take_like(w.hand[p], w.n_hand[p], ctd_ctype(w.seven[i])));
      ctd_restore_next(w);
      w.n_seven = 0;
      CTD_LOOP for (int i = 0; i < 7; ++i) w.seven[i] = 0;
      break;
    case CTD_K_MARSHAL: CTD_NOT_PRESET(); CTD_NOT_CLASSIC();
    case CTD_K_DIPLOMAT: CTD_NOT_PRESET(); CTD_NOT_CLASSIC(); {  // carry_out_marshal (:505-515) / carry_out_diplomat (:538-551)
      const int q = CTD_OPT_TARGET(d), t = CTD_OPT_CARD_A(d);
      const int money = k == CTD_K_MARSHAL ? ctd_cost_of_type(t)
                                           : (ctd_cost_of_type(t) > ctd_cost_of_type(CTD_OPT_CARD_B(d))
                                                  ? ctd_cost_of_type(t) - ctd_cost_of_type(CTD_OPT_CARD_B(d))
                                                  : ctd_cost_of_type(CTD_OPT_CARD_B(d)) - ctd_cost_of_type(t));
      w.gold[p] -= (int32_t)money;
      w.gold[q] += (int32_t)money;
      ctd_append(w, w.bld[p], w.n_bld[p], CTD_BLD_CAP, ctd_take_like(w.bld[q], w.n_bld[q], t));
      if (k == CTD_K_DIPLOMAT)
        ctd_append(w, w.bld[q], w.n_bld[q], CTD_BLD_CAP, ctd_take_like(w.bld[p], w.n_bld[p], CTD_OPT_CARD_B(d)));
      if (ctd_count_type(w.bld[q], w.n_bld[q], t) > 1) w.replicas[q] -= 1;
      if (t == 34) {  // settle_museum, non-warlord branch: the tucked cards follow the Museum
        CTD_LOOP for (int i = 0; i < w.n_mus[q]; ++i) ctd_append(w, w.mus[p], w.n_mus[p], CTD_MUS_CAP, w.mus[q][i]);
        w.n_mus[q] = 0;
      }
      if (t == 29 && (w.pflags[q] & CTD_PF_LIGHTHOUSE)) {
        w.pflags[q] &= (uint8_t)~CTD_PF_LIGHTHOUSE;
        w.pflags[p] |= CTD_PF_LIGHTHOUSE;
      }
      ctd_to5(w, p);
      w.done |= CTD_DM_CHARACTER;
      break;
    }
    default: w.err |= CTD_ERR_UNIMPL; break;
  }
#ifdef CTD_HOST_DEBUG
  {  // container / purse maxima over everything this process played (cap study: tools/scan_status_cpu.py with HS_LIB=debug build)
    static int mx[5] = {0, 0, 0, 0, 0};
    bool up = false;
    for (int q = 0; q < 6; ++q) {
      const int v[5] = {w.n_hand[q], w.n_bld[q], w.n_mus[q], w.n_jd[q], w.gold[q] < 0 ? -w.gold[q] : w.gold[q]};
      for (int i = 0; i < 5; ++i) if (v[i] > mx[i]) { mx[i] = v[i]; up = true; }
    }
    if (up) fprintf(stderr, "MAX hand %d city %d museum %d just_drawn %d |gold| %d (steps %u)\n", mx[0], mx[1], mx[2], mx[3], mx[4], w.steps);
  }
#endif
  ctd_is_last_round(w);
  ++w.steps;
  return won;
}

// run_utils.create_game (run_utils.py:20-27)
CTD_HD CTD_NI inline void ctd_new_game(CtdWork& w, uint64_t seed, uint64_t gid, int ruleset) {
  CTD_ASSUME_WORK(&w);
  ctd_chance_init(w, seed, gid, 0);
  ctd_deal_preset(w, ruleset);
  ctd_setup_round(w);
}

// ------------------------------------------------------------------------------------------ pack / unpack
// Scalar forms (definition of the layout).
CTD_HD CTD_NI inline void ctd_pack(const CtdWork& w, ctd_state* s) {
  CTD_ASSUME_WORK(&w);
  {  // zero the record with eight-byte stores (ctd_state is 8-byte aligned)
    uint64_t* z = (uint64_t*)s;
    CTD_LOOP for (int i = 0; i < CTD_STATE_BYTES / 8; ++i) z[i] = 0;
  }
  int pos = 0, c = 0;
  bool ovf = false;
  uint8_t* arena = s->arena;
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    const uint8_t* src[4] = {w.hand[p], w.bld[p], w.mus[p], w.jd[p]};
    const int len[4] = {w.n_hand[p], w.n_bld[p], w.n_mus[p], w.n_jd[p]};
    CTD_UNROLL for (int k = 0; k < 4; ++k) {
      s->off[c++] = (uint8_t)pos;
      int n = len[k];
      if (pos + n > 128) { ovf = true; n = 128 - pos; }
      const uint8_t* a = src[k];
      CTD_LOOP for (int i = 0; i < n; ++i) arena[pos + i] = a[i];
      pos += n;
    }
  }
  s->off[c++] = (uint8_t)pos;
  {
    int n = w.n_deck;
    if (pos + n > 128) { ovf = true; n = 128 - pos; }
    CTD_LOOP for (int i = 0; i < n; ++i) arena[pos + i] = w.deck[(w.deck_head + i) & (CTD_DECK_CAP - 1)];
    pos += n;
  }
  s->off[c++] = (uint8_t)pos;
  {
    int n = w.n_disc;
    if (pos + n > 128) { ovf = true; n = 128 - pos; }
    CTD_LOOP for (int i = 0; i < n; ++i) arena[pos + i] = w.disc[i];
    pos += n;
  }
  s->off[c] = (uint8_t)pos;
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    // gold = sign-extended low byte + 256 * (2-bit signed page in gold_hi): -640 .. 383; records written before the page
    // existed (page 0) read back unchanged
    const int g = w.gold[p], lo = (int)(int8_t)(uint8_t)g, page = (g - lo) >> 8;
    if (page < -2 || page > 1) ovf = true;
    s->gold[p] = (int8_t)lo;
    if (p < 4) s->gold_hi03 |= (uint8_t)((page & 3) << (2 * p));
    else s->gold_hi45 |= (uint8_t)((page & 3) << (2 * (p - 4)));
    const int pts = w.points[p];
    if (pts < -128 || pts > 127) ovf = true;
    s->points[p] = (int8_t)(pts < -128 ? -128 : (pts > 127 ? 127 : pts));
    s->role[p] = w.role[p]; s->replicas[p] = w.replicas[p]; s->pflags[p] = w.pflags[p];
    s->order[p] = w.order[p]; s->used_roles[p] = w.used_roles[p];
  }
  CTD_LOOP for (int r = 0; r < 8; ++r) { s->rprops[r] = w.rprops[r]; s->variant[r] = w.variant[r]; }
  s->used_len = w.used_len; s->rtc_mask = w.rtc_mask; s->state = w.state; s->player = w.player; s->done = w.done;
  s->done_builds = (uint8_t)(w.n_trade | (w.n_nontrade << 4));
  const bool interrupt = w.state == 4 || (w.state >= 6 && w.state <= 10);
  s->next_player = interrupt ? w.next_player : 0;
  s->next_mode = interrupt ? w.next_mode : 0;
  s->crown = w.crown; s->gflags = w.gflags; s->winner = w.winner; s->wiz_target = w.wiz_target;
  s->warrant_building = w.warrant_building; s->ruleset = w.ruleset;
  s->err = (uint8_t)(w.err | (ovf ? CTD_ERR_OVERFLOW : 0));
  s->seer_mask = w.seer_mask; s->seven_n = w.n_seven;
  CTD_LOOP for (int i = 0; i < 7; ++i) s->seven[i] = i < w.n_seven ? w.seven[i] : 0;
  s->rng_draws = w.draws; s->tape_pos = (uint16_t)w.tape_pos; s->steps = (uint16_t)(w.steps > 65535u ? 65535u : w.steps);
  s->gid = (uint64_t)w.g0 | ((uint64_t)w.g1 << 32);
}

CTD_HD CTD_NI inline void ctd_unpack(const ctd_state* s, CtdWork& w) {
  CTD_ASSUME_WORK(&w);
  w.err = s->err;
  const uint8_t* arena = s->arena;
  int c = 0;
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    uint8_t* dst[4] = {w.hand[p], w.bld[p], w.mus[p], w.jd[p]};
    uint8_t* cnt[4] = {&w.n_hand[p], &w.n_bld[p], &w.n_mus[p], &w.n_jd[p]};
    const int cap[4] = {CTD_HAND_CAP, CTD_BLD_CAP, CTD_MUS_CAP, CTD_JD_CAP};
    CTD_UNROLL for (int k = 0; k < 4; ++k) {
      const int b = s->off[c] & 127;
      int len = (int)s->off[c + 1] - (int)s->off[c];
      ++c;
      if (len < 0) len = 0;
      if (len > cap[k]) { len = cap[k]; w.err |= CTD_ERR_OVERFLOW; }
      if (b + len > 128) len = 128 - b;
      uint8_t* a = dst[k];
      CTD_LOOP for (int i = 0; i < len; ++i) a[i] = arena[b + i];
      *cnt[k] = (uint8_t)len;
    }
  }
  w.deck_head = 0;
  {
    const int b = s->off[24] & 127;
    int len = (int)s->off[25] - (int)s->off[24];
    if (len < 0) len = 0;
    if (len > CTD_DECK_CAP - 1) { len = CTD_DECK_CAP - 1; w.err |= CTD_ERR_OVERFLOW; }
    if (b + len > 128) len = 128 - b;
    CTD_LOOP for (int i = 0; i < len; ++i) w.deck[i] = arena[b + i];
    w.n_deck = (uint8_t)len;
  }
  {
    const int b = s->off[25] & 127;
    int len = (int)s->off[26] - (int)s->off[25];
    if (len < 0) len = 0;
    if (b + len > 128) len = 128 - b;
    CTD_LOOP for (int i = 0; i < len; ++i) w.disc[i] = arena[b + i];
    w.n_disc = (uint8_t)len;
  }
  CTD_LOOP for (int p = 0; p < 6; ++p) {
    const int page2 = p < 4 ? (s->gold_hi03 >> (2 * p)) & 3 : (s->gold_hi45 >> (2 * (p - 4))) & 3;
    w.gold[p] = (int32_t)((int)s->gold[p] + 256 * ((page2 ^ 2) - 2));
    w.role[p] = s->role[p]; w.replicas[p] = s->replicas[p]; w.pflags[p] = s->pflags[p];
    w.order[p] = s->order[p]; w.used_roles[p] = s->used_roles[p]; w.points[p] = s->points[p];
  }
  CTD_LOOP for (int r = 0; r < 8; ++r) { w.rprops[r] = s->rprops[r]; w.variant[r] = s->variant[r]; }
  w.used_len = s->used_len; w.rtc_mask = s->rtc_mask; w.state = s->state; w.player = s->player; w.done = s->done;
  w.n_trade = s->done_builds & 15; w.n_nontrade = s->done_builds >> 4;
  w.next_player = s->next_player; w.next_mode = s->next_mode; w.crown = s->crown; w.gflags = s->gflags;
  w.winner = s->winner; w.wiz_target = s->wiz_target; w.warrant_building = s->warrant_building;
  w.ruleset = s->ruleset;
  w.seer_mask = s->seer_mask; w.n_seven = s->seven_n > 7 ? 7 : s->seven_n;
  CTD_LOOP for (int i = 0; i < 7; ++i) w.seven[i] = s->seven[i];
  w.draws = s->rng_draws; w.buf_blk = 0xFFFFFFFFu; w.tape_pos = s->tape_pos; w.steps = s->steps;
  w.ring = nullptr; w.ring_hi = 0;   // kept so that the kernels' code stays unchanged
  w.g0 = (uint32_t)s->gid; w.g1 = (uint32_t)(s->gid >> 32);
}
