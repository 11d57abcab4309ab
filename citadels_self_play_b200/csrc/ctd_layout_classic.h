// ctd_layout_classic.h -- placement of the per-step device functions of ctd_k_playout_classic.
// ptxas lays the device functions of a kernel out in the order of their mangled names.  The playout kernels are bound by the SM's
// instruction cache (profiles/README.md), and which of their hot lines share cache sets is worth +-5 %: tools/layout_search.py
// timed 230 orders (random, then hill-climbing on the best) of the 19 functions the loop runs every step (renamed here to equally long names with an order prefix, so that
// they sit in one block in exactly this order, apart from the once-per-game code); this is the best one found for this unit
// (classic 1.006e9 with the functions where their own names put them -> 1.141e9 env steps/s).  Regenerate with the tool after changing the rules code.
// The order was found for the warp-per-game kernel, which also ran the warp chooser (slot 18, since removed).  On the
// per-thread kernel (ctd_playout.cuh) this order still beats the functions' own names by 9.7 % (1.718e9 against 1.567e9
// env steps/s, profiles/README.md, round 3).
#pragma once
#define ctd_count_suit ctd_h00_count_suit________________
#define ctd_philox ctd_h01_philox____________________
#define ctd_has ctd_h02_has_______________________
#define ctd_append ctd_h03_append____________________
#define ctd_draw ctd_h04_draw______________________
#define ctd_reshuffle_if_empty ctd_h05_reshuffle_if_empty________
#define ctd_player_from_rank ctd_h06_player_from_rank__________
#define ctd_take_like ctd_h07_take_like_________________
#define ctd_setup_next_player ctd_h08_setup_next_player_________
#define ctd_refresh_used_roles ctd_h09_refresh_used_roles________
#define ctd_apply_finish ctd_h10_apply_finish______________
#define ctd_count_type ctd_h11_count_type________________
#define ctd_apply_build ctd_h12_apply_build_______________
#define ctd_check_game_ending ctd_h13_check_game_ending_________
#define ctd_move_crown ctd_h14_move_crown________________
#define ctd_shuffle_bytes ctd_h15_shuffle_bytes_____________
#define ctd_setup_round ctd_h16_setup_round_______________
#define ctd_apply ctd_h17_apply_____________________
