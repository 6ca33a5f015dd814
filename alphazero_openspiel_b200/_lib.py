"""ctypes binding of libaz_b200.so (include/az_b200.h).  There is no fallback: a missing library is an error."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libaz_b200.so")

GAME_CONNECT_FOUR, GAME_BREAKTHROUGH = 0, 1
F_KEEP_TREE, F_AUTO_RESTART, F_MANUAL, F_SAMPLE_MOVES = 1 << 0, 1 << 1, 1 << 2, 1 << 3
F_RECORDS, F_OFFPOLICY, F_PRIORS_F64, F_RANDOM_START = 1 << 4, 1 << 5, 1 << 6, 1 << 7
F_ASYNC_COMPACT = 1 << 8
F_EAGER_COMPACT = 1 << 9
F_UCT = 1 << 10
F_VIRTUAL_LOSS = 1 << 11
F_EVAL_CACHE = 1 << 12
F_RESIGN = 1 << 13
F_PLAYOUT_CAP = 1 << 14
F_FORCED_PLAYOUTS = 1 << 15
EVAL_CACHE_LOG2_SHIFT = 24   # flags bits 24-28: log2 of the F_EVAL_CACHE table's entries (0 = default)
NOISE_NONE, NOISE_DIRICHLET, NOISE_HOST, NOISE_COUNTER = 0, 1, 2, 3
EVAL_EXTERNAL, EVAL_UNIFORM, EVAL_HASH, EVAL_ROLLOUT = 0, 1, 2, 3
OBS_NONE, OBS_F32_NCHW, OBS_BF16_NHWC = 0, 1, 2
PH_IDLE, PH_ROOT_EVAL, PH_LEAF_EVAL, PH_SEARCH_DONE, PH_RUN, PH_ERROR = 0, 1, 2, 3, 4, 5
CTR_NAMES = ["sims", "depth", "children", "expansions", "legal", "terminal", "root_evals", "moves", "games",
             "compact_nodes", "overflow", "idle_slots", "peak_nodes", "cache_hits", "resigns", "resign_samples",
             "resign_false"]


class AzConfig(C.Structure):
    _fields_ = [
        ("game_id", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32),
        ("n_trees", C.c_int32), ("node_capacity", C.c_int32), ("n_playouts", C.c_int32),
        ("c_puct", C.c_double), ("dirichlet_ratio", C.c_double), ("dirichlet_alpha", C.c_double),
        ("noise_weight", C.c_double), ("temperature", C.c_double),
        ("num_probabilistic_actions", C.c_int32), ("noise_mode", C.c_int32), ("eval_mode", C.c_int32),
        ("eval_shift", C.c_int32), ("max_sims_per_step", C.c_int32), ("start_plies_mod", C.c_int32),
        ("record_capacity", C.c_int32), ("max_games", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32),
        ("seed", C.c_uint64), ("leaves_per_tree", C.c_int32), ("step_cycle_budget", C.c_int32),
    ]


class AzRecord(C.Structure):
    _fields_ = [
        ("tree", C.c_int32), ("game_seq", C.c_int32), ("ply", C.c_int32), ("action", C.c_int32),
        ("n_legal", C.c_int32), ("kind", C.c_int32), ("root_n", C.c_int32), ("end", C.c_int32),
        ("bb", C.c_uint64 * 2),
        ("root_q", C.c_double), ("v_a0c", C.c_double), ("v_offpolicy", C.c_double),
    ]


class EngineUnavailable(RuntimeError):
    pass


_VP, _I32P, _U64P, _F64P = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p  # raw addresses (torch data_ptr / ctypes)

NN_F_REVERSE = 1

SIGNATURES = {
    "az_last_error": (C.c_char_p, []),
    "az_version": (C.c_int, []),
    "az_create": (C.c_int, [C.POINTER(AzConfig), C.POINTER(C.c_void_p)]),
    "az_destroy": (C.c_int, [C.c_void_p]),
    "az_config_get": (C.c_int, [C.c_void_p, C.POINTER(AzConfig)]),
    "az_max_children": (C.c_int, [C.c_void_p]),
    "az_num_actions": (C.c_int, [C.c_void_p]),
    "az_record_stride": (C.c_int, [C.c_void_p]),
    "az_device_bytes": (C.c_int64, [C.c_void_p]),
    "az_reset": (C.c_int, [C.c_void_p, _VP]),
    "az_set_positions": (C.c_int, [C.c_void_p, _I32P, _I32P, C.c_int32, _VP]),
    "az_command": (C.c_int, [C.c_void_p, _I32P, _I32P, _I32P, _VP]),
    "az_step": (C.c_int, [C.c_void_p, _VP, _VP, _F64P, _VP, C.c_int32, _VP]),
    "az_compact": (C.c_int, [C.c_void_p, _VP]),
    "az_eval_cache_invalidate": (C.c_int, [C.c_void_p, _VP]),
    "az_set_resign": (C.c_int, [C.c_void_p, C.c_double, C.c_int32, _VP]),
    "az_set_playout_cap": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, _VP]),
    "az_set_forced_playouts": (C.c_int, [C.c_void_p, C.c_double, _VP]),
    "az_debug_timing": (C.c_int, [C.c_void_p, _VP]),
    "az_status": (C.c_int, [C.c_void_p, _I32P, _I32P, _I32P, _I32P, _VP]),
    "az_request_info": (C.c_int, [C.c_void_p, _U64P, _I32P, _I32P, _I32P, C.c_int32, _VP]),
    "az_root_stats": (C.c_int, [C.c_void_p, _I32P, _F64P, _I32P, _I32P, _I32P, _F64P, _F64P, _F64P, _F64P, _VP]),
    "az_positions": (C.c_int, [C.c_void_p, _U64P, _I32P, _I32P, _F64P, _VP]),
    "az_drain_records": (C.c_int, [C.c_void_p, _VP, C.c_int64, C.POINTER(C.c_int64), _VP]),
    "az_counters": (C.c_int, [C.c_void_p, _VP, _VP]),
    "az_game_replay": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _I32P, _I32P, C.c_int32, _U64P, _I32P,
                                 _F64P, _I32P, _I32P, _VP, C.c_int32, _VP]),
    "az_observations": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _U64P, _I32P, _VP, _VP, C.c_int32, _VP]),
    "az_game_random_playouts": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_int32, _I32P,
                                          _I32P, _VP]),
    "az_nn_last_error": (C.c_char_p, []),
    "az_nn_conv3x3": (C.c_int, [_VP] * 8 + [C.c_int32] * 6 + [_VP]),
    "az_nn_block": (C.c_int, [_VP] * 9 + [C.c_int32] * 4 + [_VP]),
    "az_nn_stem": (C.c_int, [_VP] * 5 + [C.c_int32] * 4 + [_VP]),
    "az_nn_head": (C.c_int, [_VP] * 5 + [C.c_int32] * 5 + [_VP]),
    "az_nn_head_large_scratch_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "az_nn_head_large": (C.c_int, [_VP] * 6 + [C.c_int32] * 4 + [_VP]),
}

_lib = None


def load():
    """Load libaz_b200.so; raises EngineUnavailable (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EngineUnavailable(
            "libaz_b200.so is missing (%s). Build it with `python -m alphazero_openspiel_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == the library does not export the header's symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().az_last_error().decode("utf-8", "replace")
        raise RuntimeError("az_b200 error %d: %s" % (rc, msg))
