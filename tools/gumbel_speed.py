"""Cost and strength of the Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f) against PUCT.

    python tools/gumbel_speed.py --out DIR

Reports:
  * the cost of the root step: ms per search of 16 384 trees (CUDA events around begin + run + finish, the same roots every time,
    mean of --reps after one warm-up), Gumbel (m = 16) against PUCT, at 2 / 16 / 32 / 64 / 200 / 800 simulations, with the hash
    evaluator (fused kernel) and with the reference's trained 3-block weights (tests/golden/net_golden.npz) in the f16 network;
  * onb_self_play games/s (4 096 slots, 4 096 games, f16, trained weights) at 32 Gumbel simulations against 800 PUCT simulations;
  * the arena: W/L/D of Gumbel(n) against PUCT(n) for n = 8, 16, 32, 64 and of Gumbel(32) against PUCT(800), onb_fight on 4 096 dealt
    games with alternating colours, both agents on the trained weights (f16), the reference's ply cap of 150.
Writes gumbel_speed.json and gumbel_speed.txt into DIR; the card's name and power limit are read in the same run."""
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


def search_ms(onb, torch, ctx, roots, sims, evaluator, gumbel, reps):
    """mean ms of begin + run + finish on the same roots (one untimed warm-up search first)"""
    if gumbel:
        ctx.set_gumbel(True, m=16, seed=1)
    else:
        ctx.set_gumbel(False)
    stream = ctx.torch_stream()
    times = []
    for r in range(reps + 1):
        ctx.set_states(roots)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            ctx.mcts_begin(2.0, sims)
            ctx.mcts_run(evaluator, sims)
            ctx.mcts_finish(to_host=False)
            e1.record(stream)
        e1.synchronize()
        if r:
            times.append(e0.elapsed_time(e1))
    ctx.set_gumbel(False)
    return float(np.mean(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for gumbel_speed.json and gumbel_speed.txt")
    ap.add_argument("--trees", type=int, default=16384)
    ap.add_argument("--sims", default="2,16,32,64,200,800")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sp-slots", type=int, default=4096)
    ap.add_argument("--arena-games", type=int, default=4096)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch

    import __graft_entry__ as ge
    ge.build()
    import oracle_lib as O
    import onitama_alphazero_b200 as onb
    from test_net_cpu import golden_tensors

    sims_list = [int(s) for s in a.sims.split(",")]
    res = dict(card=card_info(), torch_device=torch.cuda.get_device_name(0), trees=a.trees, m=16, c_visit=50.0, c_scale=0.1, search={})
    lines = ["GPU: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (res["torch_device"], res["card"])]
    weights = golden_tensors()

    # ---- cost of the root step: mid-game roots (12 random plies), the same for both modes
    g = O.new_games(2 * a.trees, seed=3)
    for step in range(12):
        live = (np.arange(2 * a.trees) % 12) > step
        h = g.copy()
        O.env_step_random(h, 3, step)
        g[live] = h[live]
    roots = np.ascontiguousarray(g[g["result"] == 0][:a.trees])
    with onb.Context(len(roots), seed=1, mcts_max_sims=max(sims_list), planes=False) as ctx:
        ctx.net_load(weights, precision="f16")
        for ev_name, ev in (("hash", onb.EVAL_HASH), ("net_f16", onb.EVAL_NET)):
            for sims in sims_list:
                puct = search_ms(onb, torch, ctx, roots, sims, ev, False, a.reps)
                gum = search_ms(onb, torch, ctx, roots, sims, ev, True, a.reps)
                res["search"]["%s_%d" % (ev_name, sims)] = dict(puct_ms=puct, gumbel_ms=gum)
                lines.append("search %-7s %5d trees x %3d sims: PUCT %8.2f ms, Gumbel %8.2f ms (%.2fx)" % (
                    ev_name, len(roots), sims, puct, gum, gum / puct))
                print(lines[-1], flush=True)

    # ---- self-play games/s: 32 Gumbel simulations against 800 PUCT simulations
    res["self_play"] = {}
    with onb.Context(a.sp_slots, seed=2, mcts_max_sims=800) as ctx:
        ctx.net_load(weights, precision="f16")
        for name, sims, gumbel in (("gumbel_32", 32, dict(m=16, seed=1)), ("puct_800", 800, False)):
            ctx.self_play_native(2.0, sims, a.sp_slots, max_plies=2, evaluator=onb.EVAL_NET, gumbel=gumbel)   # warm-up
            ctx.sync()
            t0 = time.perf_counter()
            r = ctx.self_play_native(2.0, sims, a.sp_slots, evaluator=onb.EVAL_NET, gumbel=gumbel)
            ctx.sync()
            dt = time.perf_counter() - t0
            res["self_play"][name] = dict(seconds=dt, games=r["games"], games_per_s=r["games"] / dt, plies=r["plies_run"],
                                          samples=int(r["z"].numel()))
            lines.append("self-play %-9s: %d slots, %d games: %.2f s, %.1f games/s, %d plies, %d samples" % (
                name, a.sp_slots, r["games"], dt, r["games"] / dt, r["plies_run"], int(r["z"].numel())))
            print(lines[-1], flush=True)
        ctx.set_gumbel(False)

    # ---- the arena: Gumbel(n) against PUCT(n') on the trained weights
    res["arena"] = {}
    n = a.arena_games
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=5, mcts_max_sims=800, planes=False) as ctx:
        ctx.net_load(weights, precision="f16")
        for ng, npc in ((8, 8), (16, 16), (32, 32), (64, 64), (32, 800)):
            ctx.reset()
            t0 = time.perf_counter()
            w, l, d, _ = ctx.fight_native(ctx.agent_gumbel(ng, m=16, c_scale=0.1, evaluator=onb.EVAL_NET, net_slot=0),
                                          ctx.agent_puct(npc, 2.0, onb.EVAL_NET, 0), a_is_red, max_plies=150)
            dt = time.perf_counter() - t0
            st = ctx.fight_stats()
            res["arena"]["gumbel%d_vs_puct%d" % (ng, npc)] = dict(wins=w, losses=l, draws=d, seconds=dt, plies=ctx.last_fight_plies,
                                                                  as_red=st["color"][0], as_blue=st["color"][1])
            lines.append("arena Gumbel(%d) vs PUCT(%d), %d games: Gumbel W/L/D %d/%d/%d (as Red %d/%d/%d, as Blue %d/%d/%d), %d plies, %.1f s" % (
                ng, npc, n, w, l, d, st["color"][0]["wins"], st["color"][0]["loses"], st["color"][0]["draws"], st["color"][1]["wins"],
                st["color"][1]["loses"], st["color"][1]["draws"], ctx.last_fight_plies, dt))
            print(lines[-1], flush=True)
    with open(os.path.join(a.out, "gumbel_speed.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    with open(os.path.join(a.out, "gumbel_speed.txt"), "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
