"""Speed of search-tree reuse between moves (onb_mcts_set_reuse, DESIGN.md §5e).

    python tools/reuse_speed.py --out DIR

Reports, for the seeded 3-block network (tests/test_net_cpu.py lively_model) and for the reference's trained 3-block weights
(tests/golden/net_golden.npz):
  * config-5-shaped plies: 16 384 games x 800 simulations with ONB_EVAL_NET, f32-faithful and f16, with and without reuse, from the
    same dealt games: ms per ply (CUDA events around begin + run + finish + play_best, mean over plies 2..P: the first ply of a
    reuse run has nothing to keep), network evaluations per ply (leaf evaluations = simulations run) and the kept share (root
    visits carried over / visit target);
  * the reroot: onb_mcts_begin with reuse on (plan, order, compaction, pool swap and the one histogram copy), against
    onb_mcts_begin without reuse, CUDA events around the call;
  * onb_self_play with and without reuse in games/s (4 096 slots, 4 096 games, 200 simulations, f16).
Writes reuse_speed.json and reuse_speed.txt into DIR; the card's name and power limit are read in the same run."""
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


def plies(onb, torch, ctx, n, sims, plies_n, reuse):
    """P plies of search + best move from the same deals; per ply: ms (events), evaluations, kept share, reroot ms"""
    ctx.set_reuse(False)
    if reuse:
        ctx.set_reuse(True)
    ctx.reset()
    stream = ctx.torch_stream()
    out = []
    for _ in range(plies_n):
        ctx.reuse_stats(clear=True)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        with torch.cuda.stream(stream):
            e0.record(stream)
            ctx.mcts_begin(2.0, sims)
            e1.record(stream)
            ctx.mcts_run(onb.EVAL_NET, sims)
            ctx.mcts_finish(to_host=False)
            ctx.mcts_play_best()
            e2.record(stream)
        e2.synchronize()
        st = ctx.reuse_stats()
        evals = st["sims"] if reuse else n * sims
        out.append(dict(ms=e0.elapsed_time(e2), begin_ms=e0.elapsed_time(e1), evals=evals,
                        kept_share=st["kept_visits"] / float(n * sims) if reuse else 0.0, kept_trees=st["kept"] if reuse else 0))
    ctx.set_reuse(False)
    return out


def summarise(rows):
    tail = rows[1:]
    return dict(ms_per_ply=float(np.mean([r["ms"] for r in tail])), evals_per_ply=float(np.mean([r["evals"] for r in tail])),
                kept_share=float(np.mean([r["kept_share"] for r in tail])), begin_ms=float(np.median([r["begin_ms"] for r in tail])),
                plies=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for reuse_speed.json and reuse_speed.txt")
    ap.add_argument("--games", type=int, default=16384)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--plies", type=int, default=6)
    ap.add_argument("--sp-games", type=int, default=4096)
    ap.add_argument("--sp-sims", type=int, default=200)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch

    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as onb
    from test_net_cpu import golden_tensors, lively_model

    res = dict(card=card_info(), torch_device=torch.cuda.get_device_name(0), games=a.games, sims=a.sims, plies=a.plies, nets={})
    nets = dict(seeded=lively_model(3, seed=7).state_dict(), trained=golden_tensors())
    lines = ["GPU: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (res["torch_device"], res["card"])]
    with onb.Context(a.games, seed=1, mcts_max_sims=a.sims, planes=False) as ctx:
        for name, w in nets.items():
            for prec in ("f32", "f16"):
                ctx.net_load(w, precision=prec)
                plies(onb, torch, ctx, a.games, a.sims, 2, False)   # warm-up of every launch shape
                off = summarise(plies(onb, torch, ctx, a.games, a.sims, a.plies, False))
                on = summarise(plies(onb, torch, ctx, a.games, a.sims, a.plies, True))
                res["nets"]["%s_%s" % (name, prec)] = dict(off=off, on=on)
                lines.append("%-8s %s: %d games x %d sims | no reuse %.1f ms/ply, %.3g evals/ply | reuse %.1f ms/ply, %.3g evals/ply, kept share "
                             "%.3f | speed-up %.2fx | begin: %.2f ms without reuse, %.2f ms with (reroot)" % (
                                 name, prec, a.games, a.sims, off["ms_per_ply"], off["evals_per_ply"], on["ms_per_ply"], on["evals_per_ply"],
                                 on["kept_share"], off["ms_per_ply"] / on["ms_per_ply"], off["begin_ms"], on["begin_ms"]))
                print(lines[-1], flush=True)
    res["self_play"] = {}
    with onb.Context(a.sp_games, seed=2, mcts_max_sims=a.sp_sims) as ctx:
        for name, w in nets.items():
            ctx.net_load(w, precision="f16")
            ctx.self_play_native(2.0, a.sp_sims, a.sp_games, max_plies=4, evaluator=onb.EVAL_NET)   # warm-up
            for reuse in (False, True):
                ctx.reuse_stats(clear=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = ctx.self_play_native(2.0, a.sp_sims, a.sp_games, evaluator=onb.EVAL_NET, reuse=reuse)
                ctx.sync()
                dt = time.perf_counter() - t0
                st = ctx.reuse_stats()
                row = dict(seconds=dt, games=r["games"], games_per_s=r["games"] / dt, plies=r["plies_run"], samples=int(r["z"].numel()),
                           evals=st["sims"] if reuse else None, searched_trees=st["trees"] if reuse else None)
                res["self_play"]["%s_%s" % (name, "reuse" if reuse else "plain")] = row
                lines.append("self-play %-8s f16 %s: %d slots, %d games x %d sims: %.2f s, %.1f games/s, %d plies%s" % (
                    name, "reuse   " if reuse else "no reuse", a.sp_games, a.sp_games, a.sp_sims, dt, r["games"] / dt, r["plies_run"],
                    ", %.3g evals for %d searched positions (%.3f of the target)" % (st["sims"], st["trees"], st["sims"] / float(st["trees"] * a.sp_sims))
                    if reuse else ""))
                print(lines[-1], flush=True)
            ctx.set_reuse(False)
    with open(os.path.join(a.out, "reuse_speed.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    with open(os.path.join(a.out, "reuse_speed.txt"), "w") as fh:
        fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
