"""Times the fused PUCT search (BASELINE config 4: 16 384 trees x 400 simulations, uniform and hash evaluators), by default as built,
or once per value of environment variables, and checks that every variant builds the same trees:
python tools/mcts_time.py [VAR=a,b,c ...]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import onitama_alphazero_b200 as onb

n, sims = 1 << 14, 400
s = torch.cuda.Stream(); torch.cuda.set_stream(s)
ctx = onb.Context(n, seed=20240607, stream=s.cuda_stream, mcts_max_sims=sims, planes=False, mcts_node_cap=int(os.environ.get('ONB_TIME_NODE_CAP', '0')))
ctx.reset()
base = ctx.get_states(); cur = base.copy()
for step in range(16):   # the config-4 roots: positions after (id mod 16) random plies
    ctx.step_random(step)
    nxt = ctx.get_states()
    live = (np.arange(n) % 16) > step
    cur[live] = nxt[live]
    ctx.set_states(cur)
dead = cur["result"] != 0
cur[dead] = base[dead]
ctx.set_states(cur)


def run(label, evaluator=onb.EVAL_UNIFORM, reps=8):
    for _ in range(3):
        ctx.mcts_begin(2.0, sims); ctx.mcts_run(evaluator, sims); ctx.mcts_finish(to_host=False)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(s)
    for _ in range(reps):
        ctx.mcts_begin(2.0, sims); ctx.mcts_run(evaluator, sims); ctx.mcts_finish(to_host=False)
    b.record(s); b.synchronize()
    ms = a.elapsed_time(b) / reps
    out = ctx.mcts_finish()
    print("%-44s %.3f ms  %.4g sims/s" % (label, ms, n * sims / ms * 1e3), flush=True)
    return out["child_visits"].copy(), out["root_q"].copy()


specs = [a.split("=") for a in sys.argv[1:]] or [[None, "default"]]
ref = None
for var, vals in specs:
    for v in vals.split(","):
        if var is not None:
            os.environ[var] = v
        for ev, name in ((onb.EVAL_UNIFORM, "uniform"), (onb.EVAL_HASH, "hash")):
            got = run("%s %s" % (v if var is None else "%s=%s" % (var, v), name), ev)
            key = name
            if ref is None:
                ref = {}
            if key not in ref:
                ref[key] = got
            else:
                assert np.array_equal(ref[key][0], got[0]) and np.array_equal(ref[key][1].view(np.uint64), got[1].view(np.uint64)), "variant changed the trees"
    if var is not None:
        os.environ.pop(var, None)
print("all variants built identical trees")
