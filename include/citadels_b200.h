/*
 * citadels_b200.h -- C ABI of the B200-native Citadels rollout engine.
 *
 * This is the drop-in boundary for the reference's hot path (SURVEY.md section 8(b)): legal-option
 * enumeration + state transition + random playout.  Every entry point names the reference
 * interface it replaces (paths relative to the reference repository root).  All functions return
 * a ctd_status (0 = OK).  Pointer arguments are HOST pointers unless the name ends in `_dev`
 * (device pointers on the handle's device).  No callbacks, no torch types.
 *
 * A handle owns `capacity` game slots in HBM.  A slot holds one 256-byte packed game record
 * (`ctd_state`, layout below) -- the equivalent of one reference `Game` object
 * (game/game.py:16-24, :522-540) without the CFR knowledge block.
 */
#ifndef CITADELS_B200_H
#define CITADELS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ctd_engine ctd_engine;

typedef enum {
  CTD_OK = 0,
  CTD_EARG = 1,   /* bad argument (null pointer, n > capacity, ...) */
  CTD_ECUDA = 2,  /* CUDA runtime error; see ctd_last_error() */
  CTD_ECAP = 3,   /* a fixed-size buffer was too small (options stride, tape) */
  CTD_ENOMEM = 4
} ctd_status;

/* rulesets: which variant of each of the 8 ranks is in play (game/config.py:83-91) */
#define CTD_RULESET_PRESET 0  /* Witch Spy Wizard King Abbot Alchemist Navigator Warlord, game/game.py:479-486 */
#define CTD_RULESET_CLASSIC 1 /* Assassin Thief Magician King Bishop Merchant Architect Warlord */
#define CTD_RULESET_RANDOM 2  /* Game(preset=False), game/game.py:491-520: 14 random uniques, 4 cards each, a random
                                 variant per rank (all 24 characters), random pick order and crown */

/* Packed game record.  Bytes [0,228) plus seer_mask / seven_n / seven[] are reference-visible state (tests compare
 * them bit for bit with a dump of the reference Game); the rest of [228,256) is engine-private. */
#define CTD_STATE_BYTES 256
#define CTD_STATE_VISIBLE_BYTES 228
typedef struct ctd_state {
  uint8_t arena[128];    /* card codes, 26 ordered containers back to back: per seat hand, buildings,
                            museum_cards, just_drawn_cards (game/agent.py:12-20); then deck, discard_deck.
                            code 0..39 = type_ID; 40..43 = Magic School with suit trade/war/religion/lord */
  uint8_t off[28];       /* off[c] = start of container c in arena; off[26] = total cards */
  int8_t gold[6];        /* Agent.gold (may go negative): low byte; see gold_hi03 / gold_hi45 for purses beyond a byte */
  uint8_t role[6];       /* 0..7 rank; 8 = None; 9 = "Bewitched" */
  int8_t replicas[6];    /* Agent.replicas (False == 0) */
  uint8_t pflags[6];     /* bit0 can_use_lighthouse, bit1 first_to_7, bit2 witch */
  uint8_t rprops[8];     /* RolePropery per rank: bit0 dead, bits1-2 warrant, bit3 possessed, bit4 robbed,
                            bits5-6 blackmail (0 None, 1 Real, 2 Fake) */
  uint8_t variant[8];    /* which of the 3 names of rank r is in game.roles */
  uint8_t order[6];      /* turn_orders_for_roles */
  uint8_t used_roles[6]; /* used_roles, value+1 (0 = -1 "Bewitched") */
  uint8_t used_len;
  uint8_t rtc_mask;      /* roles_to_choose_from */
  uint8_t state;         /* GameState.state 0..10 */
  uint8_t player;        /* GameState.player_id */
  uint8_t done;          /* already_done_moves flags: smithy, lab, magic_school, museum, character_ability,
                            begged, take_gold */
  uint8_t done_builds;   /* low nibble #trade_building, high nibble #non_trade_building */
  uint8_t next_player;   /* next_gamestate.player_id (only inside an interrupt state) */
  uint8_t next_mode;     /* 0 none, 1 same done-moves list, 2 reset to [character_ability], 3 empty */
  uint8_t crown;         /* seat holding the crown */
  uint8_t gflags;        /* bit0 ending, bit1 terminal */
  int8_t winner;         /* -1 until terminal */
  uint8_t wiz_target;    /* seat whose hand the acting Wizard looked at this round, 0xFF none */
  int8_t points[6];      /* Game.points at terminal */
  uint8_t warrant_building;
  uint8_t ruleset;
  /* ---- engine-private ---- */
  uint8_t err;           /* CTD_ERR_* flags */
  uint8_t seer_mask;     /* game.seer_taken_card_from as a seat mask (it is always in seat order) */
  uint8_t seven_n;       /* len(game.seven_drawn_cards) */
  uint8_t gold_hi03;     /* seats 0..3, two bits each: signed page p, gold = (int8) gold[seat] + 256 * p, p in -2..1 (0 in every
                            finished game of the reference; run-away games of Game(preset=False) and CFR's hypothetical games need it) */
  uint32_t rng_draws;    /* Philox draws consumed by this game so far */
  uint16_t tape_pos;     /* chance-tape cursor (replay mode) */
  uint16_t steps;        /* env steps applied to this slot (saturating) */
  uint8_t seven[7];      /* game.seven_drawn_cards (Scholar) */
  uint8_t gold_hi45;     /* seats 4, 5 (bits 0-3) */
  uint64_t gid;          /* Philox game id of this slot (counter words 2,3) */
} ctd_state;

#define CTD_ERR_OVERFLOW 1   /* a container exceeded its on-chip capacity */
#define CTD_ERR_REF_RAISE 2  /* the reference would raise here (KeyError/IndexError/...) */
#define CTD_ERR_UNIMPL 4     /* option kind outside the built tiers */
#define CTD_ERR_TAPE 8       /* chance tape exhausted or malformed */
#define CTD_ERR_MAXSTEPS 16  /* playout hit max_steps before terminal */

/* 64-bit option descriptor == one reference `option(name, **attrs)` (game/option.py:8-18).
 * kind is the index into the reference's action list, game/option.py:34-45. */
typedef uint64_t ctd_option;
#define CTD_OPT_KIND(d) ((int)((d) & 0x3F))
#define CTD_OPT_PERP(d) ((int)(((d) >> 6) & 7))
#define CTD_OPT_TARGET(d) ((int)(((d) >> 9) & 7) - 1)
#define CTD_OPT_CARD_A(d) ((int)(((d) >> 12) & 0x3F) - 1)
#define CTD_OPT_CARD_B(d) ((int)(((d) >> 18) & 0x3F) - 1)
#define CTD_OPT_RANK(d) ((int)(((d) >> 24) & 0xF) - 1)
#define CTD_OPT_NAMED(d) ((int)(((d) >> 28) & 0xF) - 1) /* index into game/option.py:69-83 */
#define CTD_OPT_REPLICA(d) ((int)((((d) >> 32) & 0xF) ^ 8) - 8)
#define CTD_OPT_BUILD(d) ((int)(((d) >> 36) & 1))
#define CTD_OPT_NEXT_WITCH(d) ((int)(((d) >> 37) & 1))
#define CTD_OPT_CROWN(d) ((int)(((d) >> 38) & 1))
#define CTD_OPT_COUNT(d) ((int)(((d) >> 39) & 0x3F))
#define CTD_OPT_R(d) ((int)(((d) >> 45) & 0x3F)) /* Magician: subset size; Abbot: length of the gold/card list */
#define CTD_OPT_J(d) ((int)(((d) >> 51) & 0x3FF))
/* field reuse by the deluxe characters: magistrate_warrant rank = real target, named = first fake, count = second fake;
 * blackmail rank = real, named = fake; give_crown named = 0 gold / 1 card / 13 nothing; cardinal_exchange a = built card,
 * build = factory flag, count = number of cards given, j = which thinned combination; diplomat_exchange a = taken,
 * b = given; give_back_card: card type + 1 per seat of seer_mask in fields a, b, count, r, j (0 = none). */

/* aggregate outcome statistics of a batch of playouts (what the reference's drivers tabulate from
 * compare_to_random.py:24-37 style loops) */
typedef struct ctd_playout_stats {
  uint64_t games;
  uint64_t steps;         /* sum of env steps */
  uint64_t steps_sq;
  uint64_t wins[6];
  int64_t points_sum[6];
  uint64_t points_sq[6];
  uint64_t errors;        /* games that ended with err != 0 */
  uint64_t max_steps;     /* longest game */
} ctd_playout_stats;

/* ---- lifetime ---- */
ctd_status ctd_create(int device, uint32_t capacity, ctd_engine** out);
void ctd_destroy(ctd_engine* e);
const char* ctd_last_error(const ctd_engine* e);
/* sizeof of the records that cross this boundary, for a binding to check its own layouts against: 0 ctd_state, 1 ctd_mccfr_result,
 * 2 ctd_target_meta, 3 knowledge block, 4 exported tree header, 5 exported node, 6 exported child entry, 7 ctd_playout_stats,
 * 8 ctd_arena_seat, 9 ctd_record_origin */
uint32_t ctd_sizeof(int what);
ctd_status ctd_sync(ctd_engine* e);
/* use an existing CUDA stream (cudaStream_t as void*); default is a stream the engine owns */
ctd_status ctd_set_stream(ctd_engine* e, void* cuda_stream);

/* Philox key used by ctd_step / ctd_playout_slots for slots that were loaded rather than reset */
ctd_status ctd_set_seed(ctd_engine* e, uint64_t seed);

/* ---- state in / out ---- */
/* run_utils.create_game (run_utils.py:20-27): Game(preset=True) + setup_round() for slots [0,n);
 * game i is keyed by (seed, first_gid + i). */
ctd_status ctd_reset(ctd_engine* e, uint32_t n, uint64_t seed, uint64_t first_gid, int ruleset);
/* copy.deepcopy(game) in / out of the engine (run_utils.py:36,40): n records of CTD_STATE_BYTES */
ctd_status ctd_load_states(ctd_engine* e, uint32_t first_slot, uint32_t n, const ctd_state* states);
ctd_status ctd_store_states(ctd_engine* e, uint32_t first_slot, uint32_t n, ctd_state* states);
/* device pointer to slot 0 (for zero-copy interop, e.g. torch.from_blob) */
ctd_status ctd_states_dev(ctd_engine* e, void** dev_ptr);

/* replay mode: per-slot chance tapes (recorded shuffles, new[k] = old[tape[k]]); tape_off has n+1 entries.
 * Slots with a tape draw chance from it instead of Philox.  n == 0 clears all tapes. */
ctd_status ctd_set_tapes(ctd_engine* e, uint32_t n, const uint8_t* tape, const uint32_t* tape_off);

/* ---- one game at a time (what the Python facade's Game / Agent.get_options / option.carry_out call) ----
 * The caller owns the record, the knowledge of all six observers (6 x CTD_KNOW_BYTES, may be NULL when CFR will
 * not be run from this game) and Game.used_cards (76 bytes). */
/* Game(preset=True); game.setup_round()  (run_utils.py:20-27) */
ctd_status ctd_game_new(ctd_engine* e, uint64_t seed, uint64_t gid, int ruleset, ctd_state* state, void* know6,
                        uint8_t* used_cards);
/* game.get_options_from_state()  (game/game.py:415-418).  Not const: the Seer's give-back list is built with fresh
 * shuffles and the Scholar's enumeration shrinks seven_drawn_cards in the reference too (game/agent_functions.py:332-361, :462-470) */
ctd_status ctd_game_options(ctd_engine* e, uint64_t seed, ctd_state* state, const void* know6, ctd_option* opts, uint32_t cap,
                            uint32_t* count);
/* option.carry_out(game)  (game/option.py:118-122); *winner = winning seat or -1 */
ctd_status ctd_game_step(ctd_engine* e, uint64_t seed, ctd_state* state, void* know6, ctd_option chosen, int8_t* winner);

/* game.sample_private_information(game.players[viewer], role_sample) (game/game.py:215-242): determinise what seat `viewer`
 * cannot see -- deck, the other hands, unconfirmed roles, which warrant / blackmail is real -- from its knowledge block, in place.
 * (Inside ctd_mccfr / ctd_mccfr_pred the kernels do this themselves; this is the single-game form of the facade.) */
ctd_status ctd_game_sample(ctd_engine* e, uint64_t seed, ctd_state* state, void* know6, const uint8_t* used_cards, int viewer,
                           int role_sample);

/* ---- the hot path ---- */
/* Game.get_options_from_state / Agent.get_options (game/game.py:415-418, game/agent.py:50-83) for slots
 * [0,n): opts[i*stride .. i*stride+counts[i]) in the reference's list order.  Terminal slots report 0.
 * counts[i] > stride => only the first `stride` were written (status CTD_ECAP) and no slot was changed: call again
 * with a larger stride.  On CTD_OK the slots of a Seer / Scholar give-back state carry what their enumeration did in
 * the reference too (chance draws, the shrunk seven_drawn_cards; game/agent_functions.py:332-361, :462-470). */
ctd_status ctd_enumerate(ctd_engine* e, uint32_t n, ctd_option* opts, uint32_t* counts, uint32_t stride);
/* (test hook) the fused playout kernel picks its option with a warp-cooperative count/select; this runs that path on
 * slots [0,n) for every k and reports how many picks differ from the ctd_enumerate list (0 everywhere = identical). */
ctd_status ctd_choose_check(ctd_engine* e, uint32_t n, uint32_t* mismatches);
/* option.carry_out(game) (game/option.py:118-122) for slots [0,n): chosen[i] == 0 skips slot i.
 * winner[i] = winning seat when that step ended the game, else -1 (the reference returns the winner
 * Agent or a falsy value). */
ctd_status ctd_step(ctd_engine* e, uint32_t n, const ctd_option* chosen, int8_t* winner);
/* the reference's random-playout loop (run_utils.py:37-41; compare_to_random.py:24-32 for seats on
 * random.choice): new preset games keyed (seed, first_gid+i), uniform-random option each step, to
 * terminal or max_steps.  Outputs may be NULL.  Runs fused on the device; slots are not touched. */
ctd_status ctd_playout(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                       uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps,
                       ctd_playout_stats* stats);
/* same loop continued from the states in slots [0,n) (create_a_close_to_finished_game's tail,
 * run_utils.py:37-41); the slots receive the terminal states. */
ctd_status ctd_playout_slots(ctd_engine* e, uint32_t n, uint32_t max_steps, int8_t* winner, uint16_t* steps);
/* device-resident variant used by bench.py: results stay in HBM, only stats come back.
 * elapsed_ms (may be NULL) receives the CUDA-event time of the playout kernel alone. */
ctd_status ctd_playout_dev(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                           uint32_t max_steps, ctd_playout_stats* stats, float* elapsed_ms);
/* ---- MCCFR (algorithms/deep_mccfr.py CFRNode) ----
 * A CFR root is a game slot plus what its player to move has learnt (Agent.known_hands / known_roles,
 * game/agent.py:25-26) -- 592 bytes, layout `CtdKnow` in csrc/ctd_engine.cuh -- plus Game.used_cards in deal
 * order (76 bytes, game/game.py:424) and the id that keys the tree's Philox stream. */
#define CTD_KNOW_BYTES 592
#define CTD_MCCFR_MAX_RESULT 128
typedef struct ctd_mccfr_result {
  uint32_t status;       /* 0 ok; bit 0 (1) terminal root -- the reference's run_mccfr raises ValueError; bit 4 (16) the reference
                            raises inside its rules code for this root (an exception out of cfr_train).  Engine limits: bit 1 (2)
                            device memory exhausted even after the retries; bit 2 (4) a container outgrew its capacity
                            (csrc/ctd_engine.cuh: hands of 64, cities of 64, museums / just_drawn of 48, 64 hand-knowledge entries in the
                            searching player's knowledge block; none seen in 287 000 scanned roots of the three rulesets) */
  uint32_t n_nodes;
  uint32_t iterations;
  uint32_t rng_draws;
  uint32_t n_children;   /* len(root.children); the first CTD_MCCFR_MAX_RESULT are in this record, ctd_mccfr_root_children reads any range */
  uint8_t role_pick;     /* root.role_pick_node: the arrays below are [6][10] (player-major) */
  uint8_t viewer;        /* original_player_id */
  uint8_t player;        /* root.current_player_id */
  uint8_t pad;
  ctd_option live_option;           /* run_mccfr's decision: root.action_choice(live=True)[1] (run_utils.py:82,86;
                                       algorithms/deep_mccfr.py:67-75, game/game.py:312-317), drawn from the tree's own chance
                                       stream right after the search; 0 for a terminal root (ValueError in the reference) */
  double node_value[6];             /* root.node_value */
  double winning_probabilities[6];  /* root.winning_probabilities */
  ctd_option options[CTD_MCCFR_MAX_RESULT];  /* option of child i */
  double cumulative_regrets[180];
  double strategy[180];
  double cumulative_strategy[180];
} ctd_mccfr_result;

/* run_utils.create_a_close_to_finished_game / create_a_random_game (run_utils.py:29-72) for slots [0,n): play game
 * (seed, first_gid+i) to terminal (T steps) and step back.
 *   CTD_ROOTS_CLOSE_TO_FINISHED  u uniform in [back_lo, back_hi]; root = step max(0, T - u), then forward along the same game
 *                                until the player to move has >= 2 options (run_utils.py:44-50; the reference's
 *                                randint(1, 30) is u + 1); the searching player is the player to move at the root.
 *   CTD_ROOTS_RANDOM_GAME        m uniform in [back_lo, back_hi]; root = games[-m] = step max(0, T + 1 - m), not moved forward
 *                                (run_utils.py:52-72).  The searching player is the player to move there, BEFORE the forced
 *                                moves CFRNode.skip_false_choice plays (run_utils.py:80-83, deep_mccfr.py:19-20).
 * Fills the slot, the searching player's knowledge block, used_cards and tree id on the device.
 * root_step (may be NULL) receives the index of the root in the game's step sequence. */
#define CTD_ROOTS_CLOSE_TO_FINISHED 0
#define CTD_ROOTS_RANDOM_GAME 1
ctd_status ctd_make_roots(ctd_engine* e, uint32_t n, uint64_t seed, uint64_t first_gid, int ruleset, uint32_t back_lo,
                          uint32_t back_hi, int flavour, uint32_t* root_step);
/* roots supplied by the caller (the facade's CFRNode(game, ...)) and read back */
ctd_status ctd_load_roots(ctd_engine* e, uint32_t n, const ctd_state* roots, const void* knows, const uint8_t* used_cards,
                          const uint64_t* gids);
ctd_status ctd_store_roots(ctd_engine* e, uint32_t n, ctd_state* roots, void* knows, uint8_t* used_cards, uint64_t* gids);
/* Tree memory.  The reference never refuses a root (its trees are Python objects), so trees are not fixed-size blocks: all trees
 * of a call allocate nodes and arrays from one arena in HBM; a tree that finds it exhausted is searched again from a larger one.
 * This reports the plan for n_roots trees: nodes in a tree's first chunk, bytes per node, bytes of the first arena. */
void ctd_mccfr_tree_shape(uint32_t iterations, int ruleset, uint32_t n_roots, uint32_t* first_chunk_nodes, uint32_t* node_bytes,
                          uint64_t* arena_bytes);
/* CFRNode(game, original_player_id=game.gamestate.player_id).cfr_train(iterations) (run_utils.py:83-85,
 * algorithms/deep_mccfr.py:187-205) on roots [0,n_roots), one tree per warp.  results[n_roots] (may be NULL) gets
 * the root's arrays; the trees stay on the device for ctd_mccfr_targets / ctd_mccfr_export / ctd_mccfr_root_children. */
ctd_status ctd_mccfr(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, int ruleset,
                     ctd_mccfr_result* results, float* elapsed_ms);
/* The trees of the last ctd_mccfr / ctd_mccfr_pred call, roots [first, first+n), as compact blocks back to back:
 *   header (128 B) | nodes (1008 B: 160 B header, the 256-byte game record, the knowledge block) | children (16 B) | doubles
 * (struct CtdTreeHdrOut / CtdNodeOut in csrc/ctd_mccfr.cuh; numpy mirror in layout.py).  sizes[n] always receives the byte size of
 * every block; with buf == NULL nothing else happens, otherwise buf (buf_bytes >= the sum of sizes) is filled.
 * This is what the facade's CFRNode.children walks (algorithms/deep_mccfr.py:24). */
ctd_status ctd_mccfr_export(ctd_engine* e, uint32_t first, uint32_t n, uint64_t* sizes, void* buf, uint64_t buf_bytes);
/* children [first, first+count) of the root of tree `tree`: option descriptors and, for vector roots, cumulative_regrets /
 * strategy / cumulative_strategy (zeros for a role-pick root, whose 6 x 10 arrays are complete in the result record) */
ctd_status ctd_mccfr_root_children(ctd_engine* e, uint32_t tree, uint32_t first, uint32_t count, ctd_option* options,
                                   double* cumulative_regrets, double* strategy, double* cumulative_strategy);

/* ---- root-parallel mode: NOT the reference's algorithm (its trees are private, algorithms/deep_mccfr.py:27-29; results differ from
 * the reference's by construction and are excluded from the parity gates).  BASELINE.json's configs[4] / north_star name it:
 * several GPUs search the SAME roots with different chance streams and pool the root's regrets / strategy / values with an
 * all-reduce every T iterations (host side: citadels_self_play_b200/parallel.py).  These two calls are what it needs. ---- */
/* `more_iterations` further iterations on the trees the last ctd_mccfr call left on the device (same n_roots, seed, ruleset) */
ctd_status ctd_mccfr_continue(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t more_iterations, int ruleset,
                              ctd_mccfr_result* results, float* elapsed_ms);
/* overwrite root.node_value [n_roots][6], root.cumulative_regrets and root.cumulative_strategy [n_roots][stride] (vector roots:
 * the first n_children entries; role-pick roots: 60) of those trees; winning_probabilities follow node_value */
ctd_status ctd_mccfr_root_set(ctd_engine* e, uint32_t n_roots, uint32_t stride, const double* cumulative_regrets,
                              const double* cumulative_strategy, const double* node_value);

/* ---- value model at depth-limited leaves (algorithms/models.py ValueOnlyNN(418, 512), eval mode) ----
 * Weights are passed BatchNorm-folded and transposed to [in][out]: w1t [448][512] (rows 418..447 zero), b1 [512],
 * w2t [512][256], b2 [256], w3t [256][128], b3 [128], w4t [128][6], b4 [6]  (value_model.fold() builds them from
 * the reference's state_dict, run_utils.py:11-18).
 * The engine holds CTD_MAX_VALUE_MODELS models, one slot per possible deep seat of an arena (CTD_SEAT_DEEP_MODEL); a slot
 * allocates its device memory on first load, and loading one slot leaves the others untouched.  ctd_set_value_model loads
 * slot 0, the model ctd_mccfr_pred and ctd_value_eval use. */
#define CTD_MAX_VALUE_MODELS 6
ctd_status ctd_set_value_model(ctd_engine* e, const float* w1t, const float* b1, const float* w2t, const float* b2,
                               const float* w3t, const float* b3, const float* w4t, const float* b4);
/* the same for slot `slot` in [0, CTD_MAX_VALUE_MODELS) (anything else: CTD_EARG) */
ctd_status ctd_set_value_model_slot(ctd_engine* e, int slot, const float* w1t, const float* b1, const float* w2t, const float* b2,
                                    const float* w3t, const float* b3, const float* w4t, const float* b4);
/* how leaf values are computed.
 *   0  batched, fp32 CUDA cores: ctd_mccfr_pred advances the trees in waves and evaluates all waiting leaves at once
 *   1  batched, tcgen05 tensor cores with 3xTF32 split precision (same waves)
 *   2  (default) fused: ctd_mccfr_pred is ONE launch; every warp evaluates the leaves its own tree meets, in fp32, and walks
 *      on -- no waves, nothing waits (the values equal backend 0 term for term).  Batched evaluations (ctd_value_eval, the
 *      data-generation paths) stay on the tensor cores. */
ctd_status ctd_set_value_backend(ctd_engine* e, int backend);
/* CFRNode.model_inference (algorithms/deep_mccfr.py:364-374) for n feature rows of 448 floats (418 used):
 * out6[i] = weight * square_and_normalize(model(features[i]))  (train_utils.py:143-145) */
ctd_status ctd_value_eval(ctd_engine* e, uint32_t n, const float* features, float weight, float* out6);
/* Game.encode_game (game/game.py:91-128) of roots [0,n) as their player to move sees them: n rows of 448 floats.
 * cfr_role_pick != 0 encodes role-pick states with player_id forced to 5, as CFRNode.expand_role_pick does
 * (algorithms/deep_mccfr.py:120-123); 0 is the plain game.encode_game() a caller gets (generate_test_data.py:14). */
ctd_status ctd_encode(ctd_engine* e, uint32_t n, int cfr_role_pick, float* features);
/* CFRNode(game, ..., model=model, training=False).cfr_pred(iterations, max_depth) (run_utils.py:78-81,
 * algorithms/deep_mccfr.py:207-229) on roots [0,n_roots).  Trees advance in waves: every tree walks until it needs a
 * leaf value, the value model runs once on the batch of all waiting leaves, the trees resume.
 * reward_weight is model_reward_weights (5 in the reference). */
ctd_status ctd_mccfr_pred(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, uint32_t max_depth, int ruleset,
                          float reward_weight, ctd_mccfr_result* results, float* elapsed_ms, uint32_t* waves_out);

/* ---- training targets (algorithms/deep_mccfr.py:258-274, :321-345; tuple format generate_test_data.py:25) ---- */
typedef struct ctd_target_meta {
  uint32_t tree;           /* root index */
  uint32_t node;           /* node index inside the tree block */
  uint32_t n_options;      /* K = len(node.children) */
  uint32_t option_offset;  /* first of the K entries in options[] / regrets[] */
  uint32_t seat;           /* gamestate.player_id the state was encoded with (random seat for role-pick nodes) */
  uint32_t role_pick;
  double node_value[6];    /* target_node_value */
} ctd_target_meta;
/* CFRNode.get_all_targets() over the trees left on the device by the last ctd_mccfr / ctd_mccfr_pred call with the
 * same n_roots (iterations / ruleset are ignored: the trees know their shape): one record per node of every tree that completed
 * (status 0) with children and node_value.sum() >= threshold (the
 * reference always uses 15, algorithms/deep_mccfr.py:268,:321), depth-first pre-order per tree.  Call once with the
 * four output pointers NULL to learn the sizes, then with buffers of *n_records rows of 448 floats / metas and
 * *n_option_slots descriptors / doubles (regrets: row `seat` of a role-pick node's matrix; all-zero rows become ones). */
ctd_status ctd_mccfr_targets(ctd_engine* e, uint32_t n_roots, uint64_t seed, uint32_t iterations, int ruleset, double threshold,
                             uint32_t* n_records, uint32_t* n_option_slots, float* features, ctd_target_meta* meta,
                             ctd_option* options, double* regrets);

/* ---- value-network training (algorithms/train.py:13-86 train_node_value_only): ValueOnlyNN(418, 512) in train mode (BatchNorm with
 * batch statistics, Dropout(0.2)), KLDivLoss(batchmean) on log(square_and_normalize(outputs) + 1e-10) vs square_and_normalize(labels),
 * Adam.  The dense products run on the tcgen05 kernel of the inference path.  Host loop (epochs, StepLR, best-eval checkpoint):
 * citadels_self_play_b200/train.py. ---- */
/* training set: features [n_train][418] (item[0] of the reference's target tuples) and node values [n_train][6] (item[2], float64);
 * validation set likewise; batch_size as in DataLoader(batch_size=...) */
ctd_status ctd_train_begin(ctd_engine* e, uint32_t n_train, const float* features, const double* node_values, uint32_t n_val,
                           const float* val_features, const double* val_node_values, uint32_t batch_size);
/* the 16 float32 tensors of ValueOnlyNN(418, 512).state_dict(), in its order (num_batches_tracked left out): fc1.weight [512][418],
 * fc1.bias, bn1.weight, bn1.bias, bn1.running_mean, bn1.running_var, fc2.weight [256][512], fc2.bias, bn2.*, fc3.weight [128][256],
 * fc3.bias, fc4.weight [6][128], fc4.bias.  set_state also resets the optimiser (Adam moments, step count). */
ctd_status ctd_train_set_state(ctd_engine* e, const float* const* tensors16);
ctd_status ctd_train_get_state(ctd_engine* e, float* const* tensors16);
/* (test hook) the gradients of the last optimiser step, same layout; the running statistics have none (zeros) */
ctd_status ctd_train_get_grads(ctd_engine* e, float* const* tensors16);
/* one epoch (train.py:36-69): every batch of the training set in `perm` order (n_train indices; NULL = as stored) with
 * learning rate lr, then the evaluation pass.  Dropout masks are Philox(seed, optimiser step, layer, element). */
ctd_status ctd_train_epoch(ctd_engine* e, uint64_t seed, float lr, const uint32_t* perm, double* train_loss, double* eval_loss);
void ctd_train_end(ctd_engine* e);

/* ---- arena (compare_to_random.py:8-37 with a player per seat) ----
 * Every game lives on the device from deal to end.  One kernel plays the random and forced moves of all games until each is
 * over or waits for a search seat with >= 2 legal options; those roots are searched in batches (one tree per game, tree id
 * (gid & (2^40 - 1)) | t << 40 for the game's t-th search) and the searches' live decisions are applied on the device.
 * Launches grow with decision rounds, not with env steps. */
#define CTD_SEAT_RANDOM 0  /* uniform over the legal options: Philox stream 4, draw (s >> 2, s & 3) for the record's steps s */
#define CTD_SEAT_PURE 1    /* run_mccfr -> cfr_train(iterations) */
#define CTD_SEAT_DEEP 2    /* run_mccfr -> cfr_pred(iterations, max_depth) with the value model in slot 0 (ctd_set_value_model) */
/* a deep seat on the value model in slot `slot` (ctd_set_value_model_slot): bits 8..15 of kind carry the slot, so CTD_SEAT_DEEP is
 * CTD_SEAT_DEEP_MODEL(0).  ctd_arena returns CTD_EARG for a kind with bits above 15, with slot bits on a random or pure seat, or whose
 * slot is >= CTD_MAX_VALUE_MODELS or holds no model.  Seats that differ only in their slot search in separate groups, each with
 * its own weights. */
#define CTD_SEAT_DEEP_MODEL(slot) (CTD_SEAT_DEEP | ((slot) << 8))
typedef struct ctd_arena_seat {
  int32_t kind;          /* CTD_SEAT_RANDOM, CTD_SEAT_PURE or CTD_SEAT_DEEP_MODEL(slot) */
  uint32_t iterations;
  uint32_t max_depth;    /* CTD_SEAT_DEEP only */
  float reward_weight;   /* CTD_SEAT_DEEP only: model_reward_weights */
} ctd_arena_seat;
/* compare_to_random.py:8-37 with a player per seat: n_games games to the end, on the device.  Outputs may be NULL.
 * searches[n] = searches made in game i.  Like ctd_mccfr, the call replaces the engine's slots and trees: on return slots
 * [0, min(n_games, capacity)) hold the final records of games [0, min(n_games, capacity)) (ctd_store_states reads them).
 * Game i is ctd_game_new(seed, first_gid + i, ruleset); a game ends at terminal, on an engine error, on a search status other
 * than 0 (the game's err gets CTD_ERR_REF_RAISE for status 16, else CTD_ERR_OVERFLOW) or after max_steps steps
 * (CTD_ERR_MAXSTEPS; max_steps <= 65535, the range of the record's steps field).  Errored games report winner -1 and count in stats->errors.  elapsed_ms (may be NULL) receives three
 * CUDA-event times: the advance phase (deal, advance and final kernels), the search phase (root gathers and searches) and the
 * apply phase. */
ctd_status ctd_arena(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                     const ctd_arena_seat seats[6], uint32_t max_steps, int8_t* winner, int8_t* points6,
                     uint16_t* steps, uint32_t* searches, ctd_playout_stats* stats, float* elapsed_ms);

/* ---- self-play training data: the arena records its searches' targets into a dataset the engine keeps in HBM ----
 * ctd_arena_record is ctd_arena plus recording: after each search of a group holding a recorded seat, the targets of its trees are
 * appended to the dataset (features, ctd_target_meta, options / regrets as ctd_mccfr_targets writes them, and a ctd_record_origin
 * per record).  The games, their outcomes, the final records and the statistics are those of ctd_arena with the same arguments:
 * recording only reads the trees, and the role-pick seat of a record is drawn from the targets' own stream (3) of its tree.
 * In the dataset, ctd_target_meta.tree is the game's index in its ctd_arena_record call and option_offset indexes the dataset's
 * option slots.  Records of one tree are consecutive in pre-order; trees are appended in no fixed order (the arena queues its games
 * with atomics), so the canonical order is (origin.gid, origin.search, row).
 * Capacity is enforced on the device: the trees of a search are kept in queue order while all their records and option slots fit;
 * a tree that does not fit is dropped whole and counted.
 * Records added by ctd_dataset_append (another engine's, or a saved dataset's) follow the ones already held.  Their tree stays
 * what it was in the call that recorded them, their origin is kept as given, and their option_offset is rebased to index this
 * dataset's option slots. */
typedef struct ctd_record_origin {
  uint64_t gid;          /* the game: ctd_game_new(seed, gid, ruleset) */
  uint32_t search;       /* the game's search number t: the tree id is (gid & (2^40 - 1)) | t << 40 */
  uint16_t step;         /* the record's steps at that search */
  uint8_t mover;         /* the seat whose search made the tree */
  int8_t winner;         /* the game's winner, filled in when the call ends; -1 for an errored game or one stopped at max_steps */
  int8_t points[6];      /* the game's points, filled in with the winner */
  uint8_t pad[2];
} ctd_record_origin;
#define CTD_RECORD_TREE 0  /* every target of the tree: CFRNode.get_all_targets(threshold) */
#define CTD_RECORD_ROOT 1  /* node 0 only, the position the game played, whenever it has children (threshold not applied) */
typedef struct ctd_record_opts {
  uint32_t seat_mask;    /* bit s: record the trees of seat s's searches (bits above 5: CTD_EARG) */
  int32_t mode;          /* CTD_RECORD_TREE or CTD_RECORD_ROOT */
  double threshold;      /* CTD_RECORD_TREE: node_value.sum() >= threshold (the reference uses 15); >= 0 */
} ctd_record_opts;
/* Note: a deep seat's tree in eval mode writes node_value only on a node's first backprop, so it sums to reward_weight (or 1 at a
 * terminal) and never reaches the reference's threshold of 15: record deep seats with CTD_RECORD_ROOT and train on
 * CTD_LABEL_WINNER, not on the model's own values. */
/* allocate the dataset (max_records rows of 448 floats, metas and origins; max_option_slots options and regrets) and clear it;
 * both sizes >= 1 */
ctd_status ctd_dataset_reserve(ctd_engine* e, uint32_t max_records, uint32_t max_option_slots);
/* empty the dataset (keeps its allocation) */
ctd_status ctd_dataset_clear(ctd_engine* e);
/* records and option slots held, trees and records dropped for want of room since the last reserve / clear (outputs may be NULL) */
ctd_status ctd_dataset_info(ctd_engine* e, uint32_t* n_records, uint32_t* n_option_slots, uint64_t* dropped_trees,
                            uint64_t* dropped_records);
/* records [first, first + n): features [n][448] f32, meta, origin (outputs may be NULL); first + n > n_records: CTD_EARG.
 * The outputs may be host memory or device memory on any GPU (the copies use cudaMemcpyDefault); the call returns once they are
 * written. */
ctd_status ctd_dataset_read(ctd_engine* e, uint32_t first, uint32_t n, float* features, ctd_target_meta* meta,
                            ctd_record_origin* origin);
/* option slots [first_slot, first_slot + n): descriptors and regrets (outputs may be NULL, host or device memory as for
 * ctd_dataset_read); beyond n_option_slots: CTD_EARG */
ctd_status ctd_dataset_read_options(ctd_engine* e, uint32_t first_slot, uint32_t n, ctd_option* options, double* regrets);
/* Append n_records records and n_option_slots option slots after the dataset's own: features [n_records][448] f32, meta, origin,
 * options and regrets [n_option_slots], laid out as ctd_dataset_read / ctd_dataset_read_options return them.  Every input may be
 * host memory or device memory on any GPU (cudaMemcpyDefault); device inputs must be complete when the call is made.  Each
 * meta.option_offset indexes the incoming options and is rebased by the dataset's n_option_slots; meta.tree and origin are kept
 * as given; the drop counts are not changed.  All or nothing: on any error the dataset is left as it was.
 * CTD_ECAP: the records or the slots do not fit the reservation.  CTD_EARG: no dataset reserved, a NULL input with n_records > 0
 * (options / regrets: with n_option_slots > 0), a meta with n_options == 0 or option_offset + n_options > n_option_slots, an origin
 * with mover > 5 or winner outside [-1, 5].  n_records == n_option_slots == 0 on a reserved dataset does nothing. */
ctd_status ctd_dataset_append(ctd_engine* e, uint32_t n_records, uint32_t n_option_slots, const float* features,
                              const ctd_target_meta* meta, const ctd_record_origin* origin, const ctd_option* options,
                              const double* regrets);
/* ctd_arena with recording.  rec: which seats, which mode, which threshold; CTD_EARG for a NULL rec, seat-mask bits above 5, an
 * unknown mode, a negative or NaN threshold, or no dataset reserved.  elapsed_ms (may be NULL) receives four CUDA-event times: the
 * three of ctd_arena and the recording (count, reserve and fill kernels per search, the outcome kernel at the end). */
ctd_status ctd_arena_record(ctd_engine* e, uint64_t n_games, uint64_t seed, uint64_t first_gid, int ruleset,
                            const ctd_arena_seat seats[6], uint32_t max_steps, int8_t* winner, int8_t* points6, uint16_t* steps,
                            uint32_t* searches, ctd_playout_stats* stats, const ctd_record_opts* rec, float* elapsed_ms);
/* ctd_train_begin with its rows gathered on the device from the dataset: records train_idx[n_train] and val_idx[n_val] (physical
 * rows).  label: CTD_LABEL_NODE_VALUE = meta.node_value (the reference's target), CTD_LABEL_WINNER = one-hot of origin.winner (a
 * single sample of what a pure tree's node_value estimates).  CTD_EARG for an index >= n_records, a winner label on a record whose
 * winner is -1, an unknown label, or whatever ctd_train_begin rejects. */
#define CTD_LABEL_NODE_VALUE 0
#define CTD_LABEL_WINNER 1
ctd_status ctd_train_begin_dataset(ctd_engine* e, uint32_t n_train, const uint32_t* train_idx, uint32_t n_val, const uint32_t* val_idx,
                                   int label, uint32_t batch_size);

/* number of kernels this engine has launched so far */
uint64_t ctd_launch_count(const ctd_engine* e);

#ifdef __cplusplus
}
#endif
#endif /* CITADELS_B200_H */
