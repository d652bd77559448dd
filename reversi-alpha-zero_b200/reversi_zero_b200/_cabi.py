"""ctypes binding of librz_engine.so (include/rz_engine.h).  No torch types cross this boundary.

The library is built in-tree by ``__graft_entry__.build()`` (csrc/Makefile).  There is no CPU
fallback: if the shared object is missing every operator raises ``RuntimeError``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "csrc", "librz_engine.so")

u64p, u8p, i8p, f32p, i32p = (C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_int8),
                              C.POINTER(C.c_float), C.POINTER(C.c_int32))
vp, sz = C.c_void_p, C.c_size_t


class RzError(RuntimeError):
    pass


class EnvState(C.Structure):
    _fields_ = [("black", C.c_uint64), ("white", C.c_uint64), ("next_player", C.c_uint8), ("turn", C.c_uint8),
                ("done", C.c_uint8), ("winner", C.c_uint8)]


class NetCfg(C.Structure):
    _fields_ = [("filters", C.c_int32), ("res_blocks", C.c_int32), ("value_fc", C.c_int32), ("kernel_size", C.c_int32)]


class EngineCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "games", "simulation_num_per_move", "parallel_search_num", "virtual_loss", "change_tau_turn", "thinking_loop",
        "required_visit_to_decide_action", "start_rethinking_turn", "allowed_resign_turn", "use_resign_threshold",
        "share_mtcs_info", "eval_mode", "net_impl", "max_plies", "warm_start", "overlap_groups", "max_sims_per_wave", "use_solver_turn", "use_solver_turn_in_simulation",
        "reset_mtcs_info_per_game", "max_searches_per_game", "arena_simulation_num")] + [(n, C.c_float) for n in (
            "c_puct", "noise_eps", "dirichlet_alpha", "resign_threshold", "disable_resignation_rate")] + [
        (n, C.c_uint64) for n in ("seed", "first_game_id", "game_id_stride", "max_games")]


class Ply(C.Structure):
    _fields_ = [("own", C.c_uint64), ("enemy", C.c_uint64), ("n_visit", C.c_int32 * 64), ("action", C.c_int16),
                ("player", C.c_uint8), ("loops", C.c_uint8), ("recorded", C.c_uint8), ("pad", C.c_uint8), ("waves", C.c_uint16),
                ("n", C.c_float), ("q", C.c_float)]


class Game(C.Structure):
    _fields_ = [("game_id", C.c_uint64), ("black", C.c_uint64), ("white", C.c_uint64), ("first_ply", C.c_int32),
                ("n_plies", C.c_int32), ("expansions", C.c_int32), ("simulations", C.c_int32), ("winner", C.c_uint8),
                ("black_z", C.c_int8), ("resign_enabled", C.c_uint8), ("resigned_mask", C.c_uint8), ("turn", C.c_uint8),
                ("black_net", C.c_uint8), ("pad", C.c_uint8 * 2), ("table_nodes", C.c_int32), ("pad2", C.c_int32)]


class PlayRow(C.Structure):
    _fields_ = [("own", C.c_uint64), ("enemy", C.c_uint64), ("n_visit", C.c_int32 * 64), ("z", C.c_int32), ("pad", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("games_started", "games_finished", "expansions", "simulations", "waves",
                                          "plies", "nn_launches", "mcts_launches", "max_nodes_used", "max_edges_used")] + [
        ("nn_ms", C.c_double), ("mcts_ms", C.c_double), ("run_ms", C.c_double)]


# name -> (restype, argtypes); every symbol include/rz_engine.h declares
SIGNATURES = {
    "rz_abi_version": (C.c_int, []),
    "rz_last_error": (C.c_char_p, []),
    "rz_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "rz_bitsliced_host": (C.c_int, [u8p, u64p, u64p, u64p, sz]),
    "rz_find_correct_moves_dev": (C.c_int, [vp, vp, vp, sz, vp]),
    "rz_find_correct_moves": (C.c_int, [u64p, u64p, u64p, sz]),
    "rz_calc_flip_dev": (C.c_int, [vp, vp, vp, vp, sz, vp]),
    "rz_calc_flip": (C.c_int, [u8p, u64p, u64p, u64p, sz]),
    "rz_step_dev": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "rz_step": (C.c_int, [u64p, u64p, u8p, u8p, u8p, u8p, i8p, u64p, sz]),
    "rz_dihedral_dev": (C.c_int, [vp, vp, vp, sz, vp]),
    "rz_solve_dev": (C.c_int, [vp, vp, vp, vp, vp, sz, vp]),
    "rz_solve": (C.c_int, [u64p, u64p, u8p, i8p, i8p, sz]),
    "rz_find_correct_moves_host": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "rz_calc_flip_host": (C.c_uint64, [C.c_int, C.c_uint64, C.c_uint64]),
    "rz_dihedral_host": (C.c_uint64, [C.c_uint64, C.c_int]),
    "rz_env_reset_host": (None, [C.POINTER(EnvState)]),
    "rz_env_update_host": (None, [C.POINTER(EnvState), C.c_uint64, C.c_uint64, C.c_int]),
    "rz_env_step_host": (None, [C.POINTER(EnvState), C.c_int]),
    "rz_net_create": (C.c_int, [C.POINTER(NetCfg), C.c_int, C.POINTER(vp)]),
    "rz_net_destroy": (C.c_int, [vp]),
    "rz_net_blob_size": (C.c_int, [vp, C.POINTER(sz)]),
    "rz_net_load_weights": (C.c_int, [vp, f32p, sz]),
    "rz_net_load_weights_dev": (C.c_int, [vp, vp, sz, vp]),
    "rz_net_predict_dev": (C.c_int, [vp, vp, vp, vp, vp, sz, C.c_int, vp]),
    "rz_net_debug_tower_dev": (C.c_int, [vp, vp, vp, vp, vp, vp, sz, vp]),
    "rz_net_debug_heads_dev": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "rz_net_predict": (C.c_int, [vp, u8p, f32p, f32p, sz, C.c_int]),
    "rz_engine_create": (C.c_int, [C.POINTER(EngineCfg), vp, C.c_int, C.POINTER(vp)]),
    "rz_engine_destroy": (C.c_int, [vp]),
    "rz_engine_run": (C.c_int, [vp, C.c_uint64, C.c_uint64]),
    "rz_engine_poll": (C.c_int, [vp, C.POINTER(Game), sz, C.POINTER(sz), C.POINTER(Ply), sz, C.POINTER(sz)]),
    "rz_engine_stats": (C.c_int, [vp, C.POINTER(Stats)]),
    "rz_engine_set_simulation_num": (C.c_int, [vp, C.c_int32]),
    "rz_engine_set_warm_start_profile": (C.c_int, [vp, f32p, C.c_int]),
    "rz_engine_set_max_games": (C.c_int, [vp, C.c_uint64]),
    "rz_engine_set_second_net": (C.c_int, [vp, vp, C.c_int]),
    "rz_engine_set_resign_threshold": (C.c_int, [vp, C.c_int, C.c_float]),
    "rz_engine_search_root": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, i32p, f32p]),
    "rz_write_play_data": (C.c_int, [C.c_char_p, C.POINTER(Game), sz, C.POINTER(Ply), C.c_int, C.c_int, C.POINTER(sz)]),
    "rz_write_play_rows": (C.c_int, [C.c_char_p, C.POINTER(Game), sz, C.POINTER(Ply), C.c_int, C.c_int, C.POINTER(sz)]),
    "rz_read_play_rows": (C.c_int, [C.c_char_p, vp, sz, C.POINTER(sz), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "rz_ingest_dev": (C.c_int, [vp, sz, C.c_int, C.c_int, vp, vp, vp, vp]),
    "rz_ingest": (C.c_int, [vp, sz, C.c_int, C.c_int, u8p, f32p, f32p]),
}

_lib = None


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RzError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          f"(the CUDA extension is mandatory, there is no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name, None)  # a missing symbol is caught by tests/test_host_mirror.py
            if fn is not None:
                fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().rz_last_error()
        raise RzError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
