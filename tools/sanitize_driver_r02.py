"""Round-2 code paths for compute-sanitizer memcheck, sized to finish quickly: the pipelined actor (slices, done words), the
deterministic compaction + subset searches of onb_self_play / onb_fight, the device Elo fold, the split-operand network kernels
(pipelined, plain), onb_selfplay_pack and the single-rank gather."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np
import torch
import onitama_alphazero_b200 as onb
from onitama_alphazero_b200.engine import Actor
from onitama_alphazero_b200.net import ConvResNet

L = onb._lib
n = 333
torch.manual_seed(0)
model = ConvResNet(64, 21, 1).eval()
with onb.Context(n, seed=3, mcts_max_sims=24) as ctx:
    ctx.reset()
    with Actor(ctx, n_sub=3, out_flags=onb.OUT_PLANES, host_flags=L.HOST_MASKS | L.HOST_DONE | L.HOST_STATS) as act:
        for step in range(5):
            for j, v in enumerate(act.views):
                act.wait(j)
                if v["count"]:
                    v["actions"][:] = 0xFFFF
                act.submit(j, None, step=step, auto_reset=True)
        for j in range(act.n_sub):
            act.wait(j)
        act.join()
    for prec, env in (("f32", {}), ("f32", {"ONB_NET_X3_PIPE": "0"}), ("f16", {})):
        os.environ.pop("ONB_NET_X3_PIPE", None)
        os.environ.update(env)
        ctx.net_load(model, precision=prec)
        ctx.encode(to_host=False)
        ctx.net_forward(onb.BUF_PLANES)
        ctx.sync()
    os.environ.pop("ONB_NET_X3_PIPE", None)
    res = ctx.self_play_native(2.0, 12, 400, max_plies=6, evaluator=onb.EVAL_NET, train=True, noise_seed=4)
    assert res["games"] == 400
    import ctypes as C
    from onitama_alphazero_b200.sharding import Comm
    with Comm(ctx, 1, 0, Comm.unique_id()) as comm:
        got = comm.gather_samples(res["planes"], res["pi"], res["z"], dst=0)
        assert got[0].shape[0] == res["planes"].shape[0]
    ctx.reset()
    a_is_red = (np.arange(n) % 2) == 0
    ctx.fight_native(ctx.agent_puct(12, 2.0), ctx.agent_uct(24), a_is_red, max_plies=8)
    st = ctx.fight_stats(history=True)
    assert st["n_games"] == n
    ctx.reset()
    ctx.search(2.0, 8, evaluator=onb.EVAL_NET)
    ctx.search(2.0, 20)
print("sanitize driver r02 ok")
