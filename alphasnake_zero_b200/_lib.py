"""ctypes binding of include/asz_b200.h.  The library is the product: if it cannot be loaded, or no CUDA device is
present, every engine call raises -- there is no CPU fallback."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ASZ_LIB") or os.path.join(HERE, "libasz_b200.so")   # ASZ_LIB: measurement builds (tools/)

ASZ_MAX_SNAKES = 8
STEP_TIC, STEP_ENCODE, STEP_AUTO_RESET, STEP_RANDOM_ACT, STEP_KEYS = 1, 2, 4, 8, 16
SPAWN_NONE, SPAWN_REPLAY, SPAWN_NATIVE = 0, 1, 2
ASZ_ERR_ARG, ASZ_ERR_CUDA, ASZ_ERR_STATE, ASZ_ERR_CAPACITY = -1, -2, -3, -4


class AszError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("side", C.c_int32), ("snakes", C.c_int32), ("health_dec", C.c_int32), ("food_chance", C.c_float),
                ("games", C.c_int32), ("seed", C.c_uint64), ("max_depth", C.c_int32), ("max_breadth", C.c_int32),
                ("softmax_base", C.c_float), ("training", C.c_int32), ("table_log2", C.c_int32),
                ("numpy1_mask", C.c_int32)]


class StepArgs(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("spawn_mode", C.c_int32), ("d_actions", C.c_void_p),
                ("d_spawn_cells", C.c_void_p), ("d_planes", C.c_void_p), ("d_row_ids", C.c_void_p),
                ("d_keys", C.c_void_p), ("max_rows", C.c_int32), ("d_row_count", C.c_void_p), ("d_ended", C.c_void_p),
                ("d_rewards", C.c_void_p), ("row_base", C.c_int32), ("plane_pitch", C.c_int32)]


class NetWeights(C.Structure):
    _fields_ = [("side", C.c_int32), ("w_conv", C.c_void_p * 9), ("scale", C.c_void_p * 9), ("bias", C.c_void_p * 9),
                ("head_w", C.c_void_p), ("head_scale", C.c_float), ("head_bias", C.c_float), ("dense1_w", C.c_void_p),
                ("dense1_b", C.c_void_p), ("dense2_w", C.c_void_p), ("dense2_b", C.c_void_p)]


class NetWeightsFP8(C.Structure):
    _fields_ = [("w", NetWeights), ("act_scale", C.c_float * 9)]


class PitPlayer(C.Structure):
    _fields_ = [("net", C.c_void_p), ("stub_word", C.c_int32)]


_lib = None

# every symbol include/asz_b200.h declares: (name, restype, argtypes)
_vp, _i32, _u32, _u64 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64
SYMBOLS = [
    ("asz_last_error", C.c_char_p, []),
    ("asz_version", C.c_int, []),
    ("asz_engine_create", C.c_int, [C.POINTER(_vp), C.POINTER(Config)]),
    ("asz_engine_destroy", C.c_int, [_vp]),
    ("asz_reset", C.c_int, [_vp, _vp]),
    ("asz_get_state", C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    ("asz_set_state", C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    ("asz_env_step", C.c_int, [_vp, C.POINTER(StepArgs), _vp]),
    ("asz_env_step_host", C.c_int, [_vp, _u32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    ("asz_env_submit_host", C.c_int, [_vp, _u32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    ("asz_env_wait_host", C.c_int, [_vp, _i32, _vp]),
    ("asz_get_totals", C.c_int, [_vp, _vp]),
    ("asz_internal_profile", C.c_int, [_vp, _vp]),
    ("asz_internal_state", C.c_int, [_vp, _vp]),
    ("asz_internal_planes", _vp, [_vp]),
    ("asz_internal_row_ids", _vp, [_vp]),
    ("asz_plane_floats", C.c_size_t, [_vp]),
    ("asz_plane_pitch", C.c_size_t, [_vp]),
    ("asz_search_begin", C.c_int, [_vp, _vp]),
    ("asz_search_epoch_begin", C.c_int, [_vp, _vp]),
    ("asz_search_step_probe", C.c_int, [_vp, _vp, _vp]),
    ("asz_search_step_sample", C.c_int, [_vp, _vp, _vp, _i32, _vp]),
    ("asz_search_finish", C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    ("asz_search_stub_values", C.c_int, [_vp, _vp]),
    ("asz_search_run_stub", C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    ("asz_search_run_net", C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp]),
    ("asz_obstacle_mask", C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    ("asz_debug_policy", C.c_int, [_vp, _vp, _i32, C.c_float, _vp, _vp, _vp, _vp]),
    ("asz_search_clear", C.c_int, [_vp, _vp]),
    ("asz_search_info", C.c_int, [_vp, _vp]),
    ("asz_search_eval_planes", _vp, [_vp]),
    ("asz_search_eval_values", _vp, [_vp]),
    ("asz_search_root_q", _vp, [_vp]),
    ("asz_search_root_moves", _vp, [_vp]),
    ("asz_search_stats", C.c_int, [_vp, _vp]),
    ("asz_search_table_dump", C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    ("asz_records_enable", C.c_int, [_vp, C.c_int64]),
    ("asz_records_append", C.c_int, [_vp, _vp, _vp, _vp]),
    ("asz_records_count", C.c_int, [_vp, _vp]),
    ("asz_records_clear", C.c_int, [_vp]),
    ("asz_records_gather", C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    ("asz_records_planes", _vp, [_vp]),
    ("asz_records_values", _vp, [_vp]),
    ("asz_records_ids", _vp, [_vp]),
    ("asz_records_turns", _vp, [_vp]),
    ("asz_net_create", C.c_int, [C.POINTER(_vp), C.POINTER(NetWeights), _i32]),
    ("asz_net_destroy", C.c_int, [_vp]),
    ("asz_net_update_weights", C.c_int, [_vp, C.POINTER(NetWeights), _vp]),
    ("asz_net_forward", C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    ("asz_net_forward_pitched", C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp]),
    ("asz_net_debug_layer", C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp]),
    ("asz_net_create_fp8", C.c_int, [C.POINTER(_vp), C.POINTER(NetWeightsFP8), _i32]),
    ("asz_net_update_weights_fp8", C.c_int, [_vp, C.POINTER(NetWeightsFP8), _vp]),
    ("asz_pit_begin", C.c_int, [_vp, C.POINTER(PitPlayer), C.POINTER(PitPlayer), _i32, _vp, _vp]),
    ("asz_pit_turn", C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp]),
    ("asz_pit_finish", C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    ("asz_pit_run", C.c_int, [_vp, C.POINTER(PitPlayer), C.POINTER(PitPlayer), _i32, _i32, _vp, _vp, _vp, _vp]),
    ("asz_pit_stats", C.c_int, [_vp, _vp]),
    ("asz_copy_root_games", C.c_int, [_vp, _vp, _vp, _vp]),
    ("asz_pit_set_search", C.c_int, [_vp, _i32, _vp]),
    ("asz_pit_search_stats", C.c_int, [_vp, _vp]),
]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AszError("libasz_b200.so is not built (run `python -m alphasnake_zero_b200.build`); "
                           "the engine has no fallback path")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise AszError("asz error %d: %s" % (rc, lib().asz_last_error().decode()))
