"""ctypes binding of libonb.so (include/onb.h). The CUDA library is the product: if it is missing this
module raises -- there is no CPU fallback and nothing here imports the oracle."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libonb.so")

ONB_OK = 0
E_INVALID, E_CUDA, E_NOMEM, E_STATE, E_OVERFLOW = -1, -2, -3, -4, -5
POLICY_UNIFORM, POLICY_AGENT = 0, 1
OUT_MASKS, OUT_PLANES, OUT_ACTIONS = 1, 2, 4
EVAL_UNIFORM, EVAL_HASH, EVAL_NET = 0, 1, 2
(BUF_STATES, BUF_MASKS, BUF_PLANES, BUF_ACTIONS, BUF_LEAF_PLANES, BUF_POLICY, BUF_VALUE, BUF_PI, BUF_BEST,
 BUF_STATS) = range(10)
STAT_STEPS, STAT_RED_WINS, STAT_BLUE_WINS, STAT_PASSES, STAT_RESETS, STAT_BAD_ACTIONS, STAT_COUNT = 0, 1, 2, 3, 4, 5, 8
HOST_MASKS, HOST_DONE, HOST_STATS = 1, 2, 4
NET_F16, NET_TF32, NET_F32 = 0, 1, 2
ACTION_NONE = 0xFFFF

# onb_state (24 bytes)
STATE_DTYPE = np.dtype([("pawns", "<u4", (2,)), ("kings", "<u4", (2,)), ("cards", "u1", (5,)), ("side", "u1"),
                        ("result", "u1"), ("flags", "u1")])
assert STATE_DTYPE.itemsize == 24


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32), ("n_games", C.c_int64), ("game_id_base", C.c_uint64),
                ("seed", C.c_uint64), ("stream", C.c_void_p), ("mcts_max_sims", C.c_uint32), ("mcts_node_cap", C.c_uint32),
                ("alloc_planes", C.c_uint32), ("reserved", C.c_uint32)]


class TreeDump(C.Structure):
    _fields_ = [("visits", C.c_void_p), ("reward", C.c_void_p), ("prior", C.c_void_p), ("action", C.c_void_p),
                ("parent", C.c_void_p), ("first_child", C.c_void_p), ("n_child", C.c_void_p), ("flags", C.c_void_p)]


class ActorView(C.Structure):
    _fields_ = [("first", C.c_int64), ("count", C.c_int64), ("actions", C.c_void_p), ("masks", C.c_void_p), ("done", C.c_void_p),
                ("stats", C.c_void_p)]


# every symbol include/onb.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "onb_version": (C.c_int32, []),
    "onb_create": (C.c_int32, [C.POINTER(Config), C.POINTER(_P)]),
    "onb_destroy": (C.c_int32, [_P]),
    "onb_last_error": (C.c_char_p, [_P]),
    "onb_sync": (C.c_int32, [_P]),
    "onb_get_stream": (C.c_int32, [_P, C.POINTER(_P)]),
    "onb_buffer": (C.c_int32, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "onb_read_buffer": (C.c_int32, [_P, C.c_int32, _P, C.c_int64]),
    "onb_write_buffer": (C.c_int32, [_P, C.c_int32, _P, C.c_int64]),
    "onb_start_states": (C.c_int32, [_P, C.c_int64, _P]),
    "onb_rand_u32": (C.c_uint32, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]),
    "onb_deal": (C.c_int32, [C.c_uint64, C.c_uint64, C.c_uint32, _P]),
    "onb_attack_maps": (C.c_int32, [_P]),
    "onb_env_reset": (C.c_int32, [_P, _P, C.c_int64, C.c_uint32]),
    "onb_env_reset_games": (C.c_int32, [_P, _P, C.c_uint32, _P]),
    "onb_env_set_states": (C.c_int32, [_P, _P, C.c_int64, C.c_int64]),
    "onb_env_get_states": (C.c_int32, [_P, _P, C.c_int64, C.c_int64]),
    "onb_env_legal_moves": (C.c_int32, [_P, _P, _P]),
    "onb_env_legal_masks": (C.c_int32, [_P, _P]),
    "onb_env_encode": (C.c_int32, [_P, _P]),
    "onb_env_step": (C.c_int32, [_P, _P, C.c_uint32, C.c_int32, C.c_uint32]),
    "onb_env_step_random": (C.c_int32, [_P, C.c_uint32, C.c_int32, C.c_int32, C.c_uint32]),
    "onb_env_choose_random": (C.c_int32, [_P, C.c_uint32, C.c_int32]),
    "onb_env_run_random": (C.c_int32, [_P, C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_uint32]),
    "onb_env_playout": (C.c_int32, [_P, C.c_uint32, C.c_uint32, C.c_int32, _P, _P]),
    "onb_env_stats": (C.c_int32, [_P, _P, C.c_int32]),
    "onb_actor_create": (C.c_int32, [_P, C.c_int32, C.c_uint32, C.c_uint32, C.POINTER(_P)]),
    "onb_actor_destroy": (C.c_int32, [_P]),
    "onb_actor_get_view": (C.c_int32, [_P, C.c_int32, C.POINTER(ActorView)]),
    "onb_actor_submit": (C.c_int32, [_P, C.c_int32, _P, C.c_uint32, C.c_int32]),
    "onb_actor_wait": (C.c_int32, [_P, C.c_int32]),
    "onb_actor_join": (C.c_int32, [_P]),
    "onb_actor_replay": (C.c_int32, [_P, _P, C.c_int64, C.c_uint32, C.c_uint32, C.c_int32]),
    "onb_perft": (C.c_int32, [_P, _P, C.c_int64, C.c_int32, _P, _P, _P]),
    "onb_mcts_begin": (C.c_int32, [_P, C.c_double, C.c_uint32]),
    "onb_mcts_set_noise": (C.c_int32, [_P, C.c_int32, C.c_double, C.c_double, C.c_uint64]),
    "onb_mcts_set_reuse": (C.c_int32, [_P, C.c_int32]),
    "onb_mcts_reuse_stats": (C.c_int32, [_P, _P, C.c_int32]),
    "onb_mcts_set_gumbel": (C.c_int32, [_P, _P]),
    "onb_mcts_select": (C.c_int32, [_P]),
    "onb_mcts_expand_backup": (C.c_int32, [_P]),
    "onb_mcts_eval": (C.c_int32, [_P, C.c_int32]),
    "onb_mcts_run": (C.c_int32, [_P, C.c_int32, C.c_uint32]),
    "onb_mcts_finish": (C.c_int32, [_P, _P, _P, _P, _P, _P]),
    "onb_mcts_play_best": (C.c_int32, [_P, C.c_uint32]),
    "onb_mcts_dump_tree": (C.c_int32, [_P, C.c_int64, C.c_int64, C.POINTER(TreeDump), C.POINTER(C.c_int64)]),
    "onb_mcts_tree_info": (C.c_int32, [_P, _P, _P]),
    "onb_selftest": (C.c_int32, [_P, C.c_int32, _P]),
    "onb_self_play": (C.c_int32, [_P, _P, _P]),
    "onb_copy_to_host": (C.c_int32, [_P, _P, _P, C.c_int64]),
    "onb_fight": (C.c_int32, [_P, _P, _P, _P, C.c_uint32, _P, _P]),
    "onb_fight_stats": (C.c_int32, [_P, C.c_double, C.c_double, _P, _P]),
    "onb_comm_unique_id": (C.c_int32, [_P]),
    "onb_comm_create": (C.c_int32, [_P, C.c_int32, C.c_int32, _P, _P, C.POINTER(_P)]),
    "onb_comm_destroy": (C.c_int32, [_P]),
    "onb_selfplay_pack": (C.c_int32, [_P, _P, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int64)]),
    "onb_gather_counts": (C.c_int32, [_P, _P, C.c_int64, _P, C.POINTER(C.c_int64)]),
    "onb_gather_samples": (C.c_int32, [_P, _P, C.c_int32, _P, _P, _P, C.c_int64, _P, _P, _P, C.c_int64, _P, C.POINTER(C.c_int64)]),
    "onb_replay_create": (C.c_int32, [_P, C.c_int64, C.POINTER(_P)]),
    "onb_replay_destroy": (C.c_int32, [_P]),
    "onb_replay_add": (C.c_int32, [_P, _P, _P, _P, C.c_int64]),
    "onb_replay_size": (C.c_int32, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "onb_replay_sample": (C.c_int32, [_P, C.c_int64, C.c_uint64, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_int64)]),
    "onb_replay_indices": (C.c_int32, [C.c_int64, C.c_int64, C.c_uint64, _P]),
    "onb_uct_run": (C.c_int32, [_P, C.c_float, C.c_uint32, C.c_uint32]),
    "onb_alphabeta_run": (C.c_int32, [_P, C.c_int32, _P, _P, _P]),
    "onb_tb_solve": (C.c_int32, [_P, _P, C.c_int32, _P]),
    "onb_tb_free": (C.c_int32, [_P]),
    "onb_tb_table": (C.c_int32, [_P, C.c_int32, C.c_int32, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "onb_tb_probe": (C.c_int32, [_P, _P]),
    "onb_tb_best": (C.c_int32, [_P, _P]),
    "onb_tb_index": (C.c_int32, [_P, _P, C.c_int64, _P, _P]),
    "onb_tb_state": (C.c_int32, [_P, C.c_int32, _P, C.c_int64, _P]),
    "onb_net_precision": (C.c_int32, [_P, C.c_int32]),
    "onb_net_select": (C.c_int32, [_P, C.c_int32]),
    "onb_net_load": (C.c_int32, [_P, C.c_int32, _P, _P, _P]),
    "onb_net_forward": (C.c_int32, [_P, C.c_int32]),
}

class SelfPlayConfig(C.Structure):
    _fields_ = [("c_puct", C.c_double), ("sims", C.c_uint32), ("evaluator", C.c_int32), ("n_games", C.c_int64), ("max_plies", C.c_uint32),
                ("train", C.c_int32), ("noise_seed", C.c_uint64), ("sample_cap", C.c_int64)]


AGENT_RANDOM, AGENT_PUCT, AGENT_UCT, AGENT_ALPHABETA, AGENT_GUMBEL, AGENT_TABLEBASE = 0, 1, 2, 3, 4, 5
ALPHABETA_MAX_DEPTH = 8
ALPHABETA_WIN = 1000000
TB_MAX_PAWNS = 4
TB_NONE = -32768


class TbClass(C.Structure):
    """onb_tb_class (onb_tb_solve): per-class counts of a solved tablebase"""
    _fields_ = [("entries", C.c_int64), ("wins", C.c_int64), ("losses", C.c_int64), ("draws", C.c_int64), ("invalid", C.c_int64),
                ("max_win", C.c_int32), ("max_loss", C.c_int32), ("iterations", C.c_int32), ("solved", C.c_int32), ("examined", C.c_int64)]


class GumbelConfig(C.Structure):
    """onb_gumbel_config (onb_mcts_set_gumbel)"""
    _fields_ = [("enabled", C.c_int32), ("max_considered", C.c_uint32), ("c_visit", C.c_double), ("c_scale", C.c_double),
                ("gumbel_scale", C.c_double), ("seed", C.c_uint64), ("step0", C.c_uint32), ("reserved", C.c_uint32)]


class Agent(C.Structure):
    """onb_agent: kind, evaluator (PUCT), net_slot (ONB_EVAL_NET), sims / playouts / alpha-beta depth, exploration constant,
    min_node_visits (UCT)"""
    _fields_ = [("kind", C.c_int32), ("evaluator", C.c_int32), ("net_slot", C.c_int32), ("sims", C.c_uint32), ("c", C.c_double),
                ("min_node_visits", C.c_uint32), ("reserved", C.c_uint32)]


class FightResult(C.Structure):
    _fields_ = [("a_wins", C.c_int64), ("b_wins", C.c_int64), ("draws", C.c_int64), ("plies_run", C.c_int64), ("results", C.c_void_p),
                ("moves_chosen", C.c_int64)]


class FightStats(C.Structure):
    """onb_fight_statistics (FightStatistics of evaluator.rs:38-110, folded on the device)"""
    _fields_ = [("n_games", C.c_int64), ("wins", C.c_int64), ("loses", C.c_int64), ("draws", C.c_int64), ("color_wins", C.c_int64 * 2),
                ("color_loses", C.c_int64 * 2), ("color_draws", C.c_int64 * 2), ("winrate", C.c_double), ("color_winrate", C.c_double * 2),
                ("rating_a", C.c_double), ("rating_b", C.c_double)]


class SelfPlayResult(C.Structure):
    _fields_ = [("n_samples", C.c_int64), ("n_valid", C.c_int64), ("n_games", C.c_int64), ("plies_run", C.c_int64), ("truncated", C.c_int32),
                ("reserved", C.c_int32), ("planes", C.c_void_p), ("pi", C.c_void_p), ("z", C.c_void_p), ("color", C.c_void_p),
                ("serial", C.c_void_p), ("valid_idx", C.c_void_p)]


_lib = None


class OnbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libonb error %d: %s" % (code, msg))
        self.code = code


def load():
    """Load libonb.so; raises if the CUDA extension has not been built (python __graft_entry__.py / build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libonb.so is missing at %s: build the CUDA extension first "
                              "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)
