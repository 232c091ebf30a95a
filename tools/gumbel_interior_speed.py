"""Cost and strength of Gumbel MuZero's interior selection (onb_gumbel_config.interior, DESIGN.md §5f) against the root-only Gumbel
search and PUCT.

    python tools/gumbel_interior_speed.py --out DIR

Reports:
  * ms per search of 16 384 mid-game trees (CUDA events around begin + run + finish, the same roots every time, mean of --reps after
    one warm-up), root-only Gumbel against interior selection (m = 16): the hash evaluator (fused kernel) at 16 / 32 / 800 simulations,
    the reference's trained 3-block weights (tests/golden/net_golden.npz) in the f16 and the f32-faithful network (split kernels) at 32
    and 800;
  * onb_self_play games/s (4 096 slots, 4 096 games, f16, trained weights) at 32 simulations, root-only against interior;
  * the arena, onb_fight on 4 096 dealt games with alternating colours, the trained weights (f16), ply cap 150: Gumbel MuZero(n) against
    root-only Gumbel(n) and against PUCT(n) for n = 16, 32, 64, and Gumbel MuZero(32) against PUCT(800).
Writes gumbel_interior_speed.json and gumbel_interior_speed.txt into DIR; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def search_ms(torch, ctx, roots, sims, evaluator, interior, reps):
    """mean ms of begin + run + finish on the same roots (one untimed warm-up search first)"""
    ctx.set_gumbel(True, m=16, seed=1, interior=interior)
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
    ap.add_argument("--out", required=True, help="directory for gumbel_interior_speed.json and gumbel_interior_speed.txt")
    ap.add_argument("--trees", type=int, default=16384)
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
    from gumbel_speed import card_info
    from test_net_cpu import golden_tensors

    res = dict(card=card_info(), torch_device=torch.cuda.get_device_name(0), trees=a.trees, m=16, c_visit=50.0, c_scale=0.1, search={})
    lines = ["GPU: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (res["torch_device"], res["card"])]
    weights = golden_tensors()

    g = O.new_games(2 * a.trees, seed=3)
    for step in range(12):
        live = (np.arange(2 * a.trees) % 12) > step
        h = g.copy()
        O.env_step_random(h, 3, step)
        g[live] = h[live]
    roots = np.ascontiguousarray(g[g["result"] == 0][:a.trees])
    with onb.Context(len(roots), seed=1, mcts_max_sims=800, planes=False) as ctx:
        for ev_name, ev, precision, sims_list in (("hash", onb.EVAL_HASH, None, (16, 32, 800)), ("net_f16", onb.EVAL_NET, "f16", (32, 800)),
                                                  ("net_f32", onb.EVAL_NET, "f32", (32, 800))):
            if precision:
                ctx.net_load(weights, precision=precision)
            for sims in sims_list:
                root_only = search_ms(torch, ctx, roots, sims, ev, False, a.reps)
                interior = search_ms(torch, ctx, roots, sims, ev, True, a.reps)
                res["search"]["%s_%d" % (ev_name, sims)] = dict(root_only_ms=root_only, interior_ms=interior)
                lines.append("search %-7s %5d trees x %3d sims: root-only Gumbel %8.2f ms, interior %8.2f ms (%.2fx)" % (
                    ev_name, len(roots), sims, root_only, interior, interior / root_only))
                print(lines[-1], flush=True)

    res["self_play"] = {}
    with onb.Context(a.sp_slots, seed=2, mcts_max_sims=32) as ctx:
        ctx.net_load(weights, precision="f16")
        for name, interior in (("root_only_32", False), ("interior_32", True)):
            gumbel = dict(m=16, seed=1, interior=interior)
            ctx.self_play_native(2.0, 32, a.sp_slots, max_plies=2, evaluator=onb.EVAL_NET, gumbel=gumbel)   # warm-up
            ctx.sync()
            t0 = time.perf_counter()
            r = ctx.self_play_native(2.0, 32, a.sp_slots, evaluator=onb.EVAL_NET, gumbel=gumbel)
            ctx.sync()
            dt = time.perf_counter() - t0
            res["self_play"][name] = dict(seconds=dt, games=r["games"], games_per_s=r["games"] / dt, plies=r["plies_run"],
                                          samples=int(r["z"].numel()))
            lines.append("self-play %-12s: %d slots, %d games: %.2f s, %.1f games/s, %d plies, %d samples" % (
                name, a.sp_slots, r["games"], dt, r["games"] / dt, r["plies_run"], int(r["z"].numel())))
            print(lines[-1], flush=True)
        ctx.set_gumbel(False)

    res["arena"] = {}
    n = a.arena_games
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=5, mcts_max_sims=800, planes=False) as ctx:
        ctx.net_load(weights, precision="f16")
        mz = lambda s: ctx.agent_gumbel(s, m=16, c_scale=0.1, evaluator=onb.EVAL_NET, net_slot=0, interior=True)  # noqa: E731
        games = [("gumbel_root_only", s, s, ctx.agent_gumbel(s, m=16, c_scale=0.1, evaluator=onb.EVAL_NET, net_slot=0)) for s in (16, 32, 64)]
        games += [("puct", s, s, ctx.agent_puct(s, 2.0, onb.EVAL_NET, 0)) for s in (16, 32, 64)]
        games += [("puct", 32, 800, ctx.agent_puct(800, 2.0, onb.EVAL_NET, 0))]
        for opp, sa, sb, agent_b in games:
            ctx.reset()
            t0 = time.perf_counter()
            w, l, d, _ = ctx.fight_native(mz(sa), agent_b, a_is_red, max_plies=150)
            dt = time.perf_counter() - t0
            st = ctx.fight_stats()
            res["arena"]["muzero%d_vs_%s%d" % (sa, opp, sb)] = dict(wins=w, losses=l, draws=d, seconds=dt, plies=ctx.last_fight_plies,
                                                                   as_red=st["color"][0], as_blue=st["color"][1])
            lines.append("arena Gumbel MuZero(%d) vs %s(%d), %d games: MuZero W/L/D %d/%d/%d (as Red %d/%d/%d, as Blue %d/%d/%d), %d plies, %.1f s" % (
                sa, opp, sb, n, w, l, d, st["color"][0]["wins"], st["color"][0]["loses"], st["color"][0]["draws"], st["color"][1]["wins"],
                st["color"][1]["loses"], st["color"][1]["draws"], ctx.last_fight_plies, dt))
            print(lines[-1], flush=True)
    with open(os.path.join(a.out, "gumbel_interior_speed.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    with open(os.path.join(a.out, "gumbel_interior_speed.txt"), "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
