"""onitama_alphazero_b200 -- B200-native (sm_100a) batched Onitama dynamics + batched PUCT MCTS behind a C ABI.

The product is libonb.so (csrc/, include/onb.h); this package is the Python host layer used by tests and bench.py.
Importing it does not touch the oracle. Every compute call requires the built CUDA library and a CUDA device."""
from . import _lib
from ._lib import (ACTION_NONE, BUF_ACTIONS, BUF_BEST, BUF_LEAF_PLANES, BUF_MASKS, BUF_PI, BUF_PLANES, BUF_POLICY, BUF_STATES,
                   BUF_STATS, BUF_VALUE, EVAL_HASH, EVAL_NET, EVAL_UNIFORM, OUT_ACTIONS, OUT_MASKS, OUT_PLANES, POLICY_AGENT, POLICY_UNIFORM,
                   STAT_BLUE_WINS, STAT_PASSES, STAT_RED_WINS, STAT_RESETS, STAT_STEPS, STATE_DTYPE, TB_NONE, BUF_VL_PLANES, BUF_VL_POLICY,
                   BUF_VL_VALUE, BUF_ROOT_M, BUF_ROOT_PROOF, NODE_LOSS, NODE_WIN, OnbError)
from .engine import Context, selfplay_protocol, start_states, tb_index, tb_states
from .selfplay import (EloRating, FightStatistics, NativeReplayBuffer, ReplayBuffer, fight, fight_statistics, resign_threshold, self_play,
                       self_play_continuous)
from .sharding import gather_replay, shard_range

__all__ = ["Context", "start_states", "tb_index", "tb_states", "OnbError", "STATE_DTYPE"]
