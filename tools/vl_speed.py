"""Time per move and strength of leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h).

    python tools/vl_speed.py --out DIR

Reports:
  * time per move: host clock around begin + run + finish, ending in a synchronise; the median over --moves searches of the same
    mid-game roots after --warmup untimed ones. Grid: n = 1 / 16 / 256 / 4 096 trees, 800 and (n <= 256) 5 000 simulations,
    K = 1 (no virtual loss) / 2 / 4 / 8 / 16 / 32 with vl = 1, the reference's trained 3-block weights (tests/golden/net_golden.npz)
    through ONB_EVAL_NET in f16 and in f32-faithful arithmetic;
  * where one round's time goes for one game at 800 simulations (f16, K = 1 and 16): torch.profiler's CUDA time per kernel;
  * strength: onb_fight over --games dealt games with alternating colours, both agents on the trained weights (f16), the reference's
    ply cap of 150: K = 4 / 16 / 32 against K = 1 at 800 simulations each, and K = 16 against K = 1 at equal time per move (K = 16
    gets the simulations that take it as long as 800 take K = 1 for one game, from the timings above).
Writes vl_speed.json and vl_speed.txt into DIR; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def move_ms(onb, ctx, roots, sims, leaves, moves, warmup):
    """median ms of begin + run + finish over `moves` searches of the same roots, host clock, ending in a synchronise"""
    ctx.set_virtual_loss(leaves, 1.0)
    times = []
    for r in range(warmup + moves):
        ctx.set_states(roots)
        ctx.sync()
        t0 = time.perf_counter()
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(onb.EVAL_NET, sims)
        ctx.mcts_finish(to_host=False)
        ctx.sync()
        if r >= warmup:
            times.append((time.perf_counter() - t0) * 1e3)
    ctx.set_virtual_loss(1)
    return float(np.median(times))


def profile_round(onb, torch, ctx, roots, sims, leaves, out_dir):
    """CUDA time per kernel of one search (torch.profiler, in a run of its own after the timings)"""
    from torch.profiler import ProfilerActivity, profile
    ctx.set_virtual_loss(leaves, 1.0)
    ctx.set_states(roots)
    ctx.search_device(2.0, sims, evaluator=onb.EVAL_NET)  # warm-up
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.set_states(roots)
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(onb.EVAL_NET, sims)
        ctx.mcts_finish(to_host=False)
        ctx.sync()
    ctx.set_virtual_loss(1)
    rows = []
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            rows.append(dict(kernel=e.key[:90], calls=int(e.count), total_us=float(t), mean_us=float(t) / max(1, int(e.count))))
    rows.sort(key=lambda r: -r["total_us"])
    return rows[:12]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for vl_speed.json and vl_speed.txt")
    ap.add_argument("--trees", default="1,16,256,4096")
    ap.add_argument("--leaves", default="1,2,4,8,16,32")
    ap.add_argument("--moves", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--skip-fight", action="store_true")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    import oracle_lib as O
    import onitama_alphazero_b200 as onb
    from test_net_cpu import golden_tensors
    if not torch.cuda.is_available():
        raise SystemExit("vl_speed.py measures on the GPU; no CUDA device found")
    card = card_info()
    weights = golden_tensors()
    trees = [int(x) for x in a.trees.split(",")]
    leaves = [int(x) for x in a.leaves.split(",")]
    g = O.new_games(2 * max(trees), seed=3)  # mid-game roots: 12 random plies
    for step in range(12):
        O.env_step_random(g, 3, step)
    live = np.ascontiguousarray(g[g["result"] == 0])
    res = dict(card=card, grid=[], profile={}, fights=[])
    lines = ["# leaf parallelism with virtual loss (DESIGN.md §5h), card: %s" % card,
             "# ms per move: median of %d (begin + run + finish + synchronise), trained 3-block weights through ONB_EVAL_NET, vl = 1" % a.moves,
             "%-10s %6s %6s" % ("precision", "trees", "sims") + "".join("%10s" % ("K=%d" % k) for k in leaves)]
    for precision in ("f16", "f32"):
        for n in trees:
            for sims in (800, 5000):
                if sims == 5000 and n > 256:
                    continue
                roots = live[:n]
                with onb.Context(n, seed=1, mcts_max_sims=sims, planes=False) as ctx:
                    ctx.net_load(weights, precision=precision)
                    row = {}
                    for k in leaves:
                        row[k] = move_ms(onb, ctx, roots, sims, k, a.moves, a.warmup)
                        res["grid"].append(dict(precision=precision, trees=n, sims=sims, leaves=k, ms_per_move=row[k]))
                lines.append("%-10s %6d %6d" % (precision, n, sims) + "".join("%10.2f" % row[k] for k in leaves))
                print(lines[-1], flush=True)
    ms = {(r["precision"], r["trees"], r["sims"], r["leaves"]): r["ms_per_move"] for r in res["grid"]}
    if ("f16", 1, 800, 1) in ms and ("f16", 1, 800, 16) in ms:
        ratio = ms[("f16", 1, 800, 16)] / ms[("f16", 1, 800, 1)]
        res["floor_ratio_k16_over_k1_one_game_800_f16"] = ratio
        lines.append("one game, 800 simulations, f16: K=16 takes %.3f of K=1's time per move (floor: at most 0.5)" % ratio)
    with onb.Context(1, seed=1, mcts_max_sims=800, planes=False) as ctx:
        ctx.net_load(weights, precision="f16")
        for k in (1, 16):
            prof = profile_round(onb, torch, ctx, live[:1], 800, k, a.out)
            res["profile"][k] = prof
            lines.append("# CUDA time per kernel, one game, 800 simulations, f16, K=%d (torch.profiler)" % k)
            lines += ["  %-90s %6d calls %10.1f us total %8.2f us mean" % (r["kernel"], r["calls"], r["total_us"], r["mean_us"]) for r in prof]
    if not a.skip_fight:
        n = a.games
        a_is_red = (np.arange(n) % 2 == 0)
        equal = 800
        if ("f16", 1, 800, 16) in ms:
            equal = int(min(5000, round(800 * ms[("f16", 1, 800, 1)] / ms[("f16", 1, 800, 16)])))
        with onb.Context(n, seed=5, mcts_max_sims=max(800, equal), planes=False) as ctx:
            ctx.net_load(weights, precision="f16")
            for k, sims_k in ((4, 800), (16, 800), (32, 800), (16, equal)):
                ctx.reset()
                t0 = time.perf_counter()
                w, l, d, _ = ctx.fight_native(ctx.agent_puct(sims_k, 2.0, onb.EVAL_NET, leaves=k), ctx.agent_puct(800, 2.0, onb.EVAL_NET), a_is_red, 150)
                dt = time.perf_counter() - t0
                res["fights"].append(dict(leaves=k, sims=sims_k, opponent="K=1 at 800", games=n, wins=w, losses=l, draws=d, seconds=dt))
                lines.append("arena: K=%d at %d sims vs K=1 at 800 sims, %d games: W/L/D %d/%d/%d (%.1f s)" % (k, sims_k, n, w, l, d, dt))
                print(lines[-1], flush=True)
    with open(os.path.join(a.out, "vl_speed.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(a.out, "vl_speed.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
