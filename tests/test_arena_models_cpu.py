"""Value-model slots and head-to-head evaluation, the parts that need no GPU: the header constants and their Python mirror, the
seat encoding of arena.deep(model=), play_arena's and head_to_head's argument checks, and the pair counting."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_value_model_slots_match_the_header():
    from citadels_self_play_b200 import layout
    src = open(os.path.join(ROOT, "include", "citadels_b200.h")).read()
    assert int(re.search(r"#define CTD_MAX_VALUE_MODELS (\d+)", src).group(1)) == layout.MAX_VALUE_MODELS
    shift = re.search(r"#define CTD_SEAT_DEEP_MODEL\(slot\) \(CTD_SEAT_DEEP \| \(\(slot\) << (\d+)\)\)", src)
    assert shift and int(shift.group(1)) == layout.SEAT_MODEL_SHIFT


def test_deep_seat_carries_its_model_slot():
    from citadels_self_play_b200 import arena
    from citadels_self_play_b200.layout import SEAT_DEEP
    assert arena.deep(200, 10, 5.0) == (SEAT_DEEP, 200, 10, 5.0) == arena.deep(200, 10, 5.0, model=0)
    for k in range(6):
        kind, its, depth, weight = arena.deep(30, 7, 2.5, model=k)
        assert kind == SEAT_DEEP | (k << 8) and (its, depth, weight) == (30, 7, 2.5)
        assert arena._seat_kind(kind) == SEAT_DEEP and arena._seat_model(kind) == k


def test_play_arena_argument_errors_come_before_any_engine():
    """Raised on the host before an engine exists (this test also passes where no GPU is present)."""
    from citadels_self_play_b200 import arena
    from citadels_self_play_b200.value_model import ValueOnlyNN
    m = ValueOnlyNN(418, 512).eval()
    rnd = [arena.random_seat()] * 5
    with pytest.raises(ValueError, match="not both"):
        arena.play_arena(2, [arena.deep(10)] + rnd, model=m, models=[m])
    with pytest.raises(ValueError, match="slots \\[0\\]"):
        arena.play_arena(2, [arena.deep(10)] + rnd)
    with pytest.raises(ValueError, match="slots \\[2\\]"):
        arena.play_arena(2, [arena.deep(10, model=2), arena.deep(10, model=1)] + rnd[1:], models=[m, m])
    with pytest.raises(ValueError, match="slots \\[1\\]"):
        arena.play_arena(2, [arena.deep(10), arena.deep(10, model=1)] + rnd[1:], model=m)
    with pytest.raises(ValueError, match="holds 6"):
        arena.play_arena(2, [arena.deep(10)] + rnd, models=[m] * 7)


def test_head_to_head_argument_errors():
    from citadels_self_play_b200 import arena
    from citadels_self_play_b200.value_model import ValueOnlyNN
    m = ValueOnlyNN(418, 512).eval()
    for pattern in ("AAAAAA", "BBRRRR", "ABABA", "ABABABA", "ABCABC", "abab ab"):
        with pytest.raises(ValueError, match="pattern"):
            arena.head_to_head(2, m, m, pattern=pattern)
    with pytest.raises(ValueError, match="deep"):
        arena.head_to_head(2, m, m, player=arena.pure(10))


def test_swap_pattern():
    from citadels_self_play_b200 import arena
    assert arena.swap_pattern("ABABAB") == "BABABA"
    assert arena.swap_pattern("AARBBR") == "BBRAAR"


def test_pair_counts_on_made_up_winners():
    from citadels_self_play_b200 import arena
    # pattern A B R A B R; the second pass plays B A R B A R
    w_ab = [0, 0, 1, 3, 2, -1, 0, 5, 4, 2, 1]
    w_ba = [1, 0, 0, 4, 2, 0, -1, 3, 3, 5, 4]
    # game:  0 A/A  1 A/B  2 B/B  3 A/A  4 R/R  5 E  6 E  7 R/B  8 B/B  9 R/R  10 B/A
    got = arena.pair_counts("ABRABR", w_ab, w_ba)
    assert got == dict(a_both=2, b_both=2, split=2, random=3, error=2)
    assert sum(got.values()) == len(w_ab)
    assert arena.pair_counts("ABABAB", np.array([], dtype=np.int8), np.array([], dtype=np.int8)) == dict.fromkeys(arena.PAIR_KEYS, 0)
    # identical winners seat for seat with no random seat: every decided pair is split
    w = np.array([0, 1, 2, 3, 4, 5, -1], dtype=np.int8)
    assert arena.pair_counts("ABABAB", w, w) == dict(a_both=0, b_both=0, split=6, random=0, error=1)
    with pytest.raises(ValueError):
        arena.pair_counts("ABABAB", [0, 1], [0])
