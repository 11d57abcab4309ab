"""Byte layout of the packed game record and bit layout of option descriptors
(mirror of include/citadels_b200.h; kept in Python so the facade can decode without the oracle)."""
import numpy as np

STATE_BYTES = 256
STATE_VISIBLE_BYTES = 228

STATE_DTYPE = np.dtype([
    ("arena", np.uint8, 128), ("off", np.uint8, 28), ("gold", np.int8, 6), ("role", np.uint8, 6),
    ("replicas", np.int8, 6), ("pflags", np.uint8, 6), ("rprops", np.uint8, 8), ("variant", np.uint8, 8),
    ("order", np.uint8, 6), ("used_roles", np.uint8, 6), ("used_len", np.uint8), ("rtc_mask", np.uint8),
    ("state", np.uint8), ("player", np.uint8), ("done", np.uint8), ("done_builds", np.uint8),
    ("next_player", np.uint8), ("next_mode", np.uint8), ("crown", np.uint8), ("gflags", np.uint8),
    ("winner", np.int8), ("wiz_target", np.uint8), ("points", np.int8, 6), ("warrant_building", np.uint8),
    ("ruleset", np.uint8), ("err", np.uint8), ("seer_mask", np.uint8), ("seven_n", np.uint8), ("gold_hi03", np.uint8),
    ("rng_draws", np.uint32), ("tape_pos", np.uint16), ("steps", np.uint16), ("seven", np.uint8, 7), ("gold_hi45", np.uint8),
    ("gid", np.uint64)])
assert STATE_DTYPE.itemsize == STATE_BYTES

# option kinds: index in the reference's action list (game/option.py:34-45)
KIND_NAMES = [
    "role_pick", "gold_or_card", "which_card_to_keep", "blackmail_response",
    "reveal_blackmail_as_blackmailer", "reveal_warrant_as_magistrate", "build", "empty_option",
    "finish_round", "ghost_town_color_choice", "smithy_choice", "laboratory_choice",
    "magic_school_choice", "weapon_storage_choice", "lighthouse_choice", "museum_choice",
    "graveyard", "take_gold_for_war", "assassination", "magistrate_warrant", "bewitching",
    "steal", "blackmail", "spy", "magic_hand_change", "discard_and_draw", "look_at_hand",
    "take_from_hand", "seer", "give_back_card", "take_crown_king", "give_crown",
    "take_crown_pat", "bishop", "cardinal_exchange", "abbot_gold_or_card", "abbot_beg",
    "merchant", "alchemist", "trader", "architect", "navigator_gold_card", "scholar",
    "scholar_card_pick", "warlord_desctruction", "marshal_steal", "diplomat_exchange"]
KIND = {n: i for i, n in enumerate(KIND_NAMES)}
# named choices (game/option.py:69-83)
NAMED_NAMES = ["gold", "card", "pay", "not_pay", "reveal", "not_reveal", "4gold", "4card", "trade", "war",
               "religion", "lord", "unique"]
SUIT_NAMES = ["trade", "war", "religion", "lord", "unique"]
# role names by rank and variant (game/config.py:83-91)
ROLES = [["Assassin", "Witch", "Magistrate"], ["Thief", "Spy", "Blackmailer"], ["Magician", "Wizard", "Seer"],
         ["King", "Emperor", "Patrician"], ["Bishop", "Abbot", "Cardinal"], ["Merchant", "Alchemist", "Trader"],
         ["Architect", "Navigator", "Scholar"], ["Warlord", "Diplomat", "Marshal"]]
COST_OF_TYPE = [1, 2, 4, 2, 5, 3, 2, 3, 5, 1, 2, 3, 1, 4, 3, 5,
                5, 3, 6, 2, 6, 5, 5, 6, 5, 6, 6, 3, 6, 3, 5, 5, 6, 5, 4, 6, 5, 4, 0, 5]
SUIT_OF_TYPE = [0] * 6 + [1] * 4 + [2] * 3 + [3] * 3 + [4] * 24


def record_gold(rec, seat):
    """Agent.gold of `seat` from a packed record: signed low byte + 256 * signed 2-bit page (gold_hi03 / gold_hi45)."""
    page = (int(rec["gold_hi03"]) >> (2 * seat)) & 3 if seat < 4 else (int(rec["gold_hi45"]) >> (2 * (seat - 4))) & 3
    return int(rec["gold"][seat]) + 256 * ((page ^ 2) - 2)


def opt_fields(d):
    d = int(d)
    rep = (d >> 32) & 0xF
    return dict(kind=d & 0x3F, perp=(d >> 6) & 7, target=((d >> 9) & 7) - 1, a=((d >> 12) & 0x3F) - 1,
                b=((d >> 18) & 0x3F) - 1, rank=((d >> 24) & 0xF) - 1, named=((d >> 28) & 0xF) - 1,
                replica=rep - 16 if rep >= 8 else rep, build=(d >> 36) & 1, next_witch=(d >> 37) & 1,
                crown=(d >> 38) & 1, count=(d >> 39) & 0x3F, r=(d >> 45) & 0x3F, j=(d >> 51) & 0x3FF)


# ---- MCCFR tree export block (csrc/ctd_mccfr.cuh: CtdTreeHdrOut | CtdNodeOut[] | CtdChild[] | double[]) ----
KNOW_BYTES = 592
# one HandKnowledge entry is a 32-bit word (csrc/ctd_engine.cuh CtdHK): bits 0-3 pid (signed, -1 = the deck), 4-6 confidence,
# 7-8 flags (1 wizard, 2 believed in this determinisation), 9-16 number of cards, 17-25 offset into the card pool
KNOW_HK_MAX = 64
KNOW_DTYPE = np.dtype([("viewer", np.uint8), ("conf_mask", np.uint8), ("n_hk", np.uint8), ("wiz_n", np.uint8),
                       ("kr", np.uint16, 6), ("hk", np.uint32, KNOW_HK_MAX), ("wiz_cards", np.uint8, 48), ("pool", np.uint8, 256),
                       ("pool_used", np.uint16), ("err", np.uint8), ("pad", np.uint8, 13)])


def hk_pack(pid, conf, flags, n, off):
    return (pid & 0xF) | (conf & 7) << 4 | (flags & 3) << 7 | (n & 0xFF) << 9 | (off & 0x1FF) << 17


def hk_unpack(word):
    word = int(word)
    pid = word & 0xF
    return dict(pid=pid - 16 if pid >= 8 else pid, conf=(word >> 4) & 7, flags=(word >> 7) & 3, n=(word >> 9) & 0xFF, off=(word >> 17) & 0x1FF)


# Knowledge blocks written by a round-1 build (and the CFR fixtures under tests/golden/, which pin the reference's knowledge in that
# form) hold at most 32 entries of 8 bytes (int8 pid, u8 conf, u8 flags, u8 n, u16 off, u16 pad) in the same 256 bytes.
_HK_V1 = np.dtype([("pid", np.int8), ("conf", np.uint8), ("flags", np.uint8), ("n", np.uint8), ("off", np.uint16), ("pad", np.uint16)])


def know_from_v1(blob):
    """592-byte knowledge block(s) in the round-1 entry format -> the current one.  Accepts [592] or [n, 592] uint8."""
    a = np.array(blob, dtype=np.uint8, copy=True)
    flat = a.reshape(-1, KNOW_BYTES)
    for row in flat:
        old = row[16:272].copy().view(_HK_V1)
        new = np.zeros(KNOW_HK_MAX, dtype=np.uint32)
        for i in range(int(row[2])):
            e = old[i]
            new[i] = hk_pack(int(e["pid"]), int(e["conf"]), int(e["flags"]), int(e["n"]), int(e["off"]))
        row[16:272] = new.view(np.uint8)
    return a


def know_to_v1(blob):
    """The inverse (blocks with at most 32 entries): what the fixtures' knowledge checksums are taken over."""
    a = np.array(blob, dtype=np.uint8, copy=True)
    flat = a.reshape(-1, KNOW_BYTES)
    for row in flat:
        if int(row[2]) > 32:
            raise ValueError("more than 32 hand-knowledge entries do not fit the round-1 format")
        new = row[16:272].copy().view(np.uint32)
        old = np.zeros(32, dtype=_HK_V1)
        for i in range(int(row[2])):
            f = hk_unpack(new[i])
            old[i] = (f["pid"], f["conf"], f["flags"], f["n"], f["off"], 0)
        row[16:272] = old.view(np.uint8)
    return a


assert KNOW_DTYPE.itemsize == KNOW_BYTES
NODE_DTYPE = np.dtype([("parent", np.int32), ("depth", np.uint16), ("player", np.uint8), ("flags", np.uint8),
                       ("n_children", np.uint32), ("child_cap", np.uint32), ("child_off", np.uint32),
                       ("arr_off", np.uint32), ("visits", np.uint32), ("pad0", np.uint32), ("V", np.float64, 6),
                       ("P", np.float64, 6), ("pred", np.float32, 6), ("order", np.uint8, 6), ("gstate", np.uint8),
                       ("winner", np.int8), ("game", STATE_DTYPE), ("know", KNOW_DTYPE)])
NODE_BYTES = NODE_DTYPE.itemsize
assert NODE_BYTES == 160 + 256 + KNOW_BYTES
CHILD_DTYPE = np.dtype([("desc", np.uint64), ("node", np.uint32), ("pad", np.uint32)])
TREE_HDR_DTYPE = np.dtype([("n_nodes", np.uint32), ("max_nodes", np.uint32), ("child_used", np.uint32),
                           ("child_cap", np.uint32), ("arr_used", np.uint32), ("arr_cap", np.uint32),
                           ("status", np.uint32), ("iterations", np.uint32), ("rng_draws", np.uint32),
                           ("viewer", np.uint8), ("training", np.uint8), ("has_model", np.uint8), ("phase", np.uint8),
                           ("gid", np.uint64), ("used_cards", np.uint8, 76), ("cur_node", np.uint32)])
assert TREE_HDR_DTYPE.itemsize == 128
NF_ROLE_PICK, NF_TERMINAL = 1, 2
# tree status bits (include/citadels_b200.h ctd_mccfr_result.status)
TREE_TERMINAL_ROOT, TREE_EPOOL, TREE_EENGINE, TREE_REF_RAISE = 1, 2, 4, 16
# ctd_arena_seat.kind, and the Philox counter word 1 of the arena's random seats (draw s of game gid: block s >> 2, word s & 3)
SEAT_RANDOM, SEAT_PURE, SEAT_DEEP = 0, 1, 2
ARENA_STREAM = 4
# value-model slots of an engine (CTD_MAX_VALUE_MODELS); a deep seat's slot sits in bits 8..15 of its kind (CTD_SEAT_DEEP_MODEL)
MAX_VALUE_MODELS = 6
SEAT_MODEL_SHIFT = 8


def tree_bytes(n_nodes, child_used, arr_used):
    return 128 + n_nodes * NODE_BYTES + child_used * 16 + arr_used * 8


class TreeView:
    """numpy views over one exported tree block (the sizes are in its header)."""

    def __init__(self, buf):
        buf = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
        self.hdr = buf[:128].view(TREE_HDR_DTYPE)[0]
        nn, nc, na = int(self.hdr["n_nodes"]), int(self.hdr["child_used"]), int(self.hdr["arr_used"])
        o = 128
        self.nodes = buf[o:o + nn * NODE_BYTES].view(NODE_DTYPE)
        o += nn * NODE_BYTES
        self.children = buf[o:o + nc * 16].view(CHILD_DTYPE)
        o += nc * 16
        self.arr = buf[o:o + na * 8].view(np.float64)

    def arrays(self, i):
        """(R, s, C) of node i shaped like the reference's numpy arrays."""
        n = self.nodes[i]
        k = int(n["n_children"])
        a = self.arr[int(n["arr_off"]):]
        if n["flags"] & NF_ROLE_PICK and k:
            return a[0:60].reshape(6, 10), a[60:120].reshape(6, 10), a[120:180].reshape(6, 10)
        cap = int(n["child_cap"])
        return a[0:k], a[cap:cap + k], a[2 * cap:2 * cap + k]

    def child_list(self, i):
        n = self.nodes[i]
        c = self.children[int(n["child_off"]):int(n["child_off"]) + int(n["n_children"])]
        return [(int(x["desc"]), int(x["node"])) for x in c]


MCCFR_RESULT_DTYPE = np.dtype([("status", np.uint32), ("n_nodes", np.uint32), ("iterations", np.uint32),
                               ("rng_draws", np.uint32), ("n_children", np.uint32), ("role_pick", np.uint8),
                               ("viewer", np.uint8), ("player", np.uint8), ("pad", np.uint8),
                               ("live_option", np.uint64), ("node_value", np.float64, 6), ("winning_probabilities", np.float64, 6),
                               ("options", np.uint64, 128), ("cumulative_regrets", np.float64, 180),
                               ("strategy", np.float64, 180), ("cumulative_strategy", np.float64, 180)])

TARGET_META_DTYPE = np.dtype([("tree", np.uint32), ("node", np.uint32), ("n_options", np.uint32), ("option_offset", np.uint32),
                              ("seat", np.uint32), ("role_pick", np.uint32), ("node_value", np.float64, 6)])
assert TARGET_META_DTYPE.itemsize == 72

# ctd_record_origin (ctd_sizeof(9)): where a self-play record came from and how its game ended (winner -1: errored or max_steps)
ORIGIN_DTYPE = np.dtype([("gid", np.uint64), ("search", np.uint32), ("step", np.uint16), ("mover", np.uint8), ("winner", np.int8),
                         ("points", np.int8, 6), ("pad", np.uint8, 2)])
assert ORIGIN_DTYPE.itemsize == 24
# ctd_record_opts.mode and the labels of ctd_train_begin_dataset
RECORD_TREE, RECORD_ROOT = 0, 1
LABEL_NODE_VALUE, LABEL_WINNER = 0, 1


def encode_options(descs):
    """option.encode_option (game/option.py:52-115) for a list of descriptors -> float32[K, 131].
    Bit layout: [0,47) kind, [47,53) perpetrator, [53,59) target, [60,68) role rank, [76,89) named choice,
    [89,129) card type, [129] replica, [130] number of "card" entries (Abbot).  The reference's elif chain means a
    `target` attribute suppresses everything after it, and tuple choices (Library pairs) set no card bits."""
    out = np.zeros((len(descs), 131), dtype=np.float32)
    for i, d in enumerate(descs):
        f = opt_fields(d)
        name = KIND_NAMES[f["kind"]]
        out[i, f["kind"]] = 1
        out[i, f["perp"] + 47] = 1
        if f["target"] >= 0:
            out[i, f["target"] + 53] = 1
        elif name == "role_pick":
            out[i, f["rank"] + 60] = 1
        elif f["named"] >= 0:
            out[i, f["named"] + 76] = 1
        elif name in ("laboratory_choice", "lighthouse_choice", "museum_choice", "build"):
            out[i, f["a"] + 89] = 1
        elif name == "which_card_to_keep":
            if f["b"] < 0:
                out[i, f["a"] + 89] = 1
        elif name == "abbot_gold_or_card":
            out[i, 130] = f["count"]
    return out
