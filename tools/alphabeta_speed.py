"""Speed of the alpha-beta arena opponent (onb_alphabeta_run / ONB_AGENT_ALPHABETA, DESIGN.md §5d).

    python tools/alphabeta_speed.py --out DIR

Reports, on 16 384 seeded mid-game roots (undecided positions after 4..19 random plies):
  * the kernel at depths 4, 6 and 8: time per call (host clock around the call and a device synchronise, median of 3 after a
    warm-up), nodes per search (mean, max, max/mean), nodes/s, and the warp efficiency of the one-game-per-thread layout
    (sum of a warp's nodes over 32 x its largest tree: the share of lane-iterations that do work, since a warp runs until its
    largest search ends);
  * the CPU oracle (tests/alphabeta_oracle.cpp, recursive, all host cores) on the same roots -- on a prefix of them at depths 6
    and 8, where the whole set would take minutes -- and the per-root speed-up;
  * one onb_fight of 16 384 games: alpha-beta at depth 4 against Random and against PUCT (uniform evaluator, 64 simulations),
    in ms per ply.
Writes alphabeta_speed.json and alphabeta_speed.txt into DIR; the card's name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_ROOTS = 16384
ORACLE_ROOTS = {4: N_ROOTS, 6: 2048, 8: 256}


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def midgame_roots(n, seed):
    import oracle_lib as O
    out = []
    have = 0
    batch = 0
    while have < n:
        m = 2 * n
        g = O.new_games(m, seed=seed + batch, game0=batch * m)
        plies = 4 + (np.arange(m) % 16)
        snap = g.copy()
        for step in range(20):
            take = plies == step
            snap[take] = g[take]
            O.env_step_random(g, seed + batch, step, game0=batch * m)
        live = snap[snap["result"] == 0]
        out.append(live)
        have += len(live)
        batch += 1
    return np.concatenate(out)[:n]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for alphabeta_speed.json and alphabeta_speed.txt")
    ap.add_argument("--depths", default="4,6,8")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import __graft_entry__ as ge
    ge.build()
    import alphabeta_oracle as A
    import onitama_alphazero_b200 as onb

    res = dict(card=card_info(), n_roots=N_ROOTS, kernel={}, oracle={}, fight={})
    roots = midgame_roots(N_ROOTS, seed=2026)
    lines = ["alpha-beta arena opponent, %d mid-game roots; card: %s" % (N_ROOTS, res["card"])]
    with onb.Context(N_ROOTS, planes=False) as ctx:
        ctx.set_states(roots)
        for depth in [int(x) for x in args.depths.split(",")]:
            r = ctx.alphabeta(depth)  # warm-up, and the node counts
            times = []
            for _ in range(3):
                ctx.sync()
                t0 = time.perf_counter()
                ctx.alphabeta(depth, to_host=False)
                ctx.sync()
                times.append(time.perf_counter() - t0)
            t = statistics.median(times)
            nodes = r["nodes"].astype(np.float64)
            warps = nodes.reshape(-1, 32)
            eff = float(warps.sum() / (32 * warps.max(axis=1)).sum())
            k = dict(ms=1e3 * t, ms_all=[1e3 * x for x in times], nodes_mean=float(nodes.mean()), nodes_max=int(nodes.max()),
                     max_over_mean=float(nodes.max() / nodes.mean()), nodes_per_s=float(nodes.sum() / t), warp_efficiency=eff)
            res["kernel"][str(depth)] = k
            lines.append("depth %d: kernel %.2f ms, nodes/search mean %.0f max %d (max/mean %.1f), %.3g nodes/s, warp efficiency %.1f %%"
                         % (depth, k["ms"], k["nodes_mean"], k["nodes_max"], k["max_over_mean"], k["nodes_per_s"], 100 * eff))
            m = ORACLE_ROOTS.get(depth, 256)
            threads = os.cpu_count() or 1
            t0 = time.perf_counter()
            want = A.alphabeta_batch(roots[:m], depth, threads=threads)
            to = time.perf_counter() - t0
            same = bool(np.array_equal(want["best"], r["best"][:m]) and np.array_equal(want["score"], r["score"][:m])
                        and np.array_equal(want["nodes"], r["nodes"][:m]))
            o = dict(roots=m, threads=threads, s=to, us_per_root=1e6 * to / m, nodes_per_s=float(want["nodes"].astype(np.float64).sum() / to),
                     gpu_us_per_root=1e3 * t * 1e3 / N_ROOTS, speedup_per_root=(to / m) / (t / N_ROOTS), bit_exact=same)
            res["oracle"][str(depth)] = o
            lines.append("         oracle (%d threads) on %d roots: %.2f s, %.3g nodes/s; per root %.1f us vs %.3f us on the GPU (x%.0f); "
                         "bit-exact %s" % (threads, m, to, o["nodes_per_s"], o["us_per_root"], o["gpu_us_per_root"], o["speedup_per_root"], same))
    with onb.Context(N_ROOTS, seed=5, mcts_max_sims=64, planes=False) as ctx:
        a_is_red = (np.arange(N_ROOTS) % 2) == 0
        for name, opp in (("random", ctx.agent_random()), ("puct64", ctx.agent_puct(64, 2.0))):
            ctx.reset(epoch=1)
            ctx.fight_native(ctx.agent_alphabeta(4), opp, a_is_red, max_plies=20)  # warm-up
            ctx.reset()
            ctx.sync()
            t0 = time.perf_counter()
            a, b, d, _ = ctx.fight_native(ctx.agent_alphabeta(4), opp, a_is_red)
            t = time.perf_counter() - t0
            plies = ctx.last_fight_plies
            f = dict(s=t, plies=plies, ms_per_ply=1e3 * t / plies, moves_chosen=ctx.last_fight_moves_chosen, ab_wins=a, opp_wins=b, draws=d)
            res["fight"][name] = f
            lines.append("fight alpha-beta(4) vs %s, %d games: %.2f s, %d plies, %.2f ms/ply; W/L/D %d/%d/%d"
                         % (name, N_ROOTS, t, plies, f["ms_per_ply"], a, b, d))
    res["card_after"] = card_info()
    text = "\n".join(lines) + "\n"
    print(text, end="")
    with open(os.path.join(args.out, "alphabeta_speed.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    with open(os.path.join(args.out, "alphabeta_speed.txt"), "w") as fh:
        fh.write(text)


if __name__ == "__main__":
    main()
