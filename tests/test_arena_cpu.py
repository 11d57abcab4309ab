"""The device arena's host-side pieces that need no GPU: the ctd_arena_seat mirror, the seat layout, the split of games over
ranks."""
import ctypes

import pytest


def test_arena_seat_record_matches_the_library():
    import __graft_entry__
    __graft_entry__.build()
    from citadels_self_play_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.ctd_sizeof.restype = ctypes.c_uint32
    assert lib.ctd_sizeof(8) == ctypes.sizeof(_lib.ArenaSeat) == 16
    assert [f[0] for f in _lib.ArenaSeat._fields_] == ["kind", "iterations", "max_depth", "reward_weight"]


def test_default_seats_are_compare_to_random_layout():
    from citadels_self_play_b200 import arena
    from citadels_self_play_b200.layout import SEAT_DEEP, SEAT_PURE, SEAT_RANDOM
    seats = arena.default_seats()
    assert seats[0] == (SEAT_DEEP, 200, 10, 5.0)
    assert seats[1] == (SEAT_PURE, 2000, 0, 0.0)
    assert seats[2:] == [(SEAT_RANDOM, 0, 0, 0.0)] * 4


@pytest.mark.parametrize("world", [1, 2, 3])
@pytest.mark.parametrize("n_games", [0, 1, 2, 7, 64, 10000])
def test_rank_blocks_cover_every_game_once(n_games, world):
    from citadels_self_play_b200 import arena
    blocks = [arena.rank_block(n_games, r, world) for r in range(world)]
    covered = [g for first, count in blocks for g in range(first, first + count)]
    assert covered == list(range(n_games))
    assert all(count >= 0 for _, count in blocks)
