"""ctypes binding of the C ABI (include/citadels_b200.h).  There is no CPU fallback: if the CUDA
library is missing or no device is present, the engine raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTD_LIB", os.path.join(_HERE, "libcitadels_b200.so"))

c_u8p = ctypes.POINTER(ctypes.c_uint8)
c_void = ctypes.c_void_p


class PlayoutStats(ctypes.Structure):
    """ctd_playout_stats"""
    _fields_ = [("games", ctypes.c_uint64), ("steps", ctypes.c_uint64), ("steps_sq", ctypes.c_uint64),
                ("wins", ctypes.c_uint64 * 6), ("points_sum", ctypes.c_int64 * 6), ("points_sq", ctypes.c_uint64 * 6),
                ("errors", ctypes.c_uint64), ("max_steps", ctypes.c_uint64)]


class ArenaSeat(ctypes.Structure):
    """ctd_arena_seat"""
    _fields_ = [("kind", ctypes.c_int32), ("iterations", ctypes.c_uint32), ("max_depth", ctypes.c_uint32),
                ("reward_weight", ctypes.c_float)]


class RecordOpts(ctypes.Structure):
    """ctd_record_opts"""
    _fields_ = [("seat_mask", ctypes.c_uint32), ("mode", ctypes.c_int32), ("threshold", ctypes.c_double)]


# every symbol include/citadels_b200.h declares: name -> (restype, argtypes)
_u32, _u64, _i = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int
SIGNATURES = {
    "ctd_create": (_i, [_i, _u32, ctypes.POINTER(c_void)]),
    "ctd_destroy": (None, [c_void]),
    "ctd_last_error": (ctypes.c_char_p, [c_void]),
    "ctd_sizeof": (_u32, [_i]),
    "ctd_sync": (_i, [c_void]),
    "ctd_set_stream": (_i, [c_void, c_void]),
    "ctd_set_seed": (_i, [c_void, _u64]),
    "ctd_reset": (_i, [c_void, _u32, _u64, _u64, _i]),
    "ctd_load_states": (_i, [c_void, _u32, _u32, c_void]),
    "ctd_store_states": (_i, [c_void, _u32, _u32, c_void]),
    "ctd_states_dev": (_i, [c_void, ctypes.POINTER(c_void)]),
    "ctd_set_tapes": (_i, [c_void, _u32, c_void, c_void]),
    "ctd_enumerate": (_i, [c_void, _u32, c_void, c_void, _u32]),
    "ctd_step": (_i, [c_void, _u32, c_void, c_void]),
    "ctd_choose_check": (_i, [c_void, _u32, c_void]),
    "ctd_playout": (_i, [c_void, _u64, _u64, _u64, _i, _u32, c_void, c_void, c_void, ctypes.POINTER(PlayoutStats)]),
    "ctd_playout_slots": (_i, [c_void, _u32, _u32, c_void, c_void]),
    "ctd_playout_dev": (_i, [c_void, _u64, _u64, _u64, _i, _u32, ctypes.POINTER(PlayoutStats),
                             ctypes.POINTER(ctypes.c_float)]),
    "ctd_arena": (_i, [c_void, _u64, _u64, _u64, _i, ctypes.POINTER(ArenaSeat), _u32, c_void, c_void, c_void, c_void,
                       ctypes.POINTER(PlayoutStats), ctypes.POINTER(ctypes.c_float)]),
    "ctd_arena_record": (_i, [c_void, _u64, _u64, _u64, _i, ctypes.POINTER(ArenaSeat), _u32, c_void, c_void, c_void, c_void,
                              ctypes.POINTER(PlayoutStats), ctypes.POINTER(RecordOpts), ctypes.POINTER(ctypes.c_float)]),
    "ctd_dataset_reserve": (_i, [c_void, _u32, _u32]),
    "ctd_dataset_clear": (_i, [c_void]),
    "ctd_dataset_info": (_i, [c_void, ctypes.POINTER(_u32), ctypes.POINTER(_u32), ctypes.POINTER(_u64), ctypes.POINTER(_u64)]),
    "ctd_dataset_read": (_i, [c_void, _u32, _u32, c_void, c_void, c_void]),
    "ctd_dataset_read_options": (_i, [c_void, _u32, _u32, c_void, c_void]),
    "ctd_dataset_append": (_i, [c_void, _u32, _u32, c_void, c_void, c_void, c_void, c_void]),
    "ctd_train_begin_dataset": (_i, [c_void, _u32, c_void, _u32, c_void, _i, _u32]),
    "ctd_launch_count": (_u64, [c_void]),
    "ctd_make_roots": (_i, [c_void, _u32, _u64, _u64, _i, _u32, _u32, _i, c_void]),
    "ctd_load_roots": (_i, [c_void, _u32, c_void, c_void, c_void, c_void]),
    "ctd_store_roots": (_i, [c_void, _u32, c_void, c_void, c_void, c_void]),
    "ctd_mccfr_tree_shape": (None, [_u32, _i, _u32, ctypes.POINTER(_u32), ctypes.POINTER(_u32), ctypes.POINTER(_u64)]),
    "ctd_mccfr_export": (_i, [c_void, _u32, _u32, c_void, c_void, _u64]),
    "ctd_mccfr_root_children": (_i, [c_void, _u32, _u32, _u32, c_void, c_void, c_void, c_void]),
    "ctd_game_new": (_i, [c_void, _u64, _u64, _i, c_void, c_void, c_void]),
    "ctd_game_options": (_i, [c_void, _u64, c_void, c_void, c_void, _u32, ctypes.POINTER(_u32)]),
    "ctd_game_step": (_i, [c_void, _u64, c_void, c_void, _u64, ctypes.POINTER(ctypes.c_int8)]),
    "ctd_game_sample": (_i, [c_void, _u64, c_void, c_void, c_void, _i, _i]),
    "ctd_set_value_model": (_i, [c_void] + [c_void] * 8),
    "ctd_set_value_model_slot": (_i, [c_void, _i] + [c_void] * 8),
    "ctd_set_value_backend": (_i, [c_void, _i]),
    "ctd_value_eval": (_i, [c_void, _u32, c_void, ctypes.c_float, c_void]),
    "ctd_encode": (_i, [c_void, _u32, _i, c_void]),
    "ctd_mccfr_pred": (_i, [c_void, _u32, _u64, _u32, _u32, _i, ctypes.c_float, c_void,
                            ctypes.POINTER(ctypes.c_float), ctypes.POINTER(_u32)]),
    "ctd_mccfr_targets": (_i, [c_void, _u32, _u64, _u32, _i, ctypes.c_double, ctypes.POINTER(_u32), ctypes.POINTER(_u32),
                               c_void, c_void, c_void, c_void]),
    "ctd_train_begin": (_i, [c_void, _u32, c_void, c_void, _u32, c_void, c_void, _u32]),
    "ctd_train_set_state": (_i, [c_void, c_void]),
    "ctd_train_get_state": (_i, [c_void, c_void]),
    "ctd_train_get_grads": (_i, [c_void, c_void]),
    "ctd_train_epoch": (_i, [c_void, _u64, ctypes.c_float, c_void, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "ctd_train_end": (None, [c_void]),
    "ctd_mccfr_continue": (_i, [c_void, _u32, _u64, _u32, _i, c_void, ctypes.POINTER(ctypes.c_float)]),
    "ctd_mccfr_root_set": (_i, [c_void, _u32, _u32, c_void, c_void, c_void]),
    "ctd_mccfr": (_i, [c_void, _u32, _u64, _u32, _i, c_void, ctypes.POINTER(ctypes.c_float)]),
}

_lib = None


def load():
    """Load libcitadels_b200.so (built in-tree by __graft_entry__.build() / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "citadels_self_play_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
