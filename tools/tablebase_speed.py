"""Solve cost of the endgame tablebase (onb_tb_solve, DESIGN.md §5g) and how often each search keeps the game-theoretic value.

    python tools/tablebase_speed.py --out DIR

Reports:
  * per card set (4 sets at max_pawns 3, 1 set at max_pawns 4): per class the iterations, W/L/D, the longest win and loss and the
    work-list entries examined; per material level p + q the solve time (host clock around onb_tb_solve, which ends in a device
    synchronise: solve(max_pawns = l) - solve(l - 1)) and the entries examined per second;
  * on 16 384 positions with a decided value (win or loss) sampled from the <= 3-pawn table of the first set: the share of moves that
    keep the value (a won position stays won; a lost one cannot be saved, so the won ones are the informative share), for PUCT with
    the uniform evaluator at 64 and 800 simulations, Gumbel (m = 16) at 32, alpha-beta at depths 4 and 6 and PUCT at 800 with the
    seeded 3-block network (tests/test_net_cpu.py lively_model) in f16. Each uses set_states, its search, the move played, then
    tb_probe of the new position.
Writes tablebase_speed.json and tablebase_speed.txt into DIR; the card's name and power limit are read in the same run."""
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

SETS3 = [[0, 1, 2, 3, 11], [4, 5, 6, 7, 8], [9, 10, 12, 13, 14], [15, 0, 5, 10, 3]]
SET4 = [0, 1, 2, 3, 11]


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def solve_levels(ctx, cards, max_pawns, lines):
    """per-level times from solves to max_pawns 0, 1, ..., max_pawns; the classes' counts of the last solve"""
    times, prev = {}, 0.0
    for level in range(max_pawns + 1):
        t0 = time.perf_counter()
        info = ctx.tb_solve(cards, level)
        dt = time.perf_counter() - t0
        times[level] = dt - prev
        prev = dt
    out = dict(cards=cards, max_pawns=max_pawns, total_s=prev, levels={}, classes={})
    lines.append("cards %s, max_pawns %d: %.2f s" % (cards, max_pawns, prev))
    for level in range(max_pawns + 1):
        ex = sum(v["examined"] for (p, q), v in info.items() if p + q == level)
        out["levels"][level] = dict(seconds=times[level], examined=ex, examined_per_s=ex / max(times[level], 1e-9))
        lines.append("  p+q=%d: %8.3f s, %.3e entries examined, %.3e entries/s" % (level, times[level], ex, ex / max(times[level], 1e-9)))
    for (p, q), v in sorted(info.items()):
        out["classes"]["%d,%d" % (p, q)] = v
        live = v["entries"] - v["invalid"]
        lines.append("  (%d,%d) %13d entries: %3d iterations, W %.4f L %.4f D %.4f of the positions, longest win %d, loss %d, examined %.3e"
                     % (p, q, v["entries"], v["iterations"], v["wins"] / live, v["losses"] / live, v["draws"] / live, v["max_win"],
                        v["max_loss"], v["examined"]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for tablebase_speed.json and tablebase_speed.txt")
    ap.add_argument("--positions", type=int, default=16384)
    ap.add_argument("--skip-four", action="store_true", help="leave out the 4-pawn solve")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    import onitama_alphazero_b200 as onb
    from test_net_cpu import lively_model

    res = dict(card=card_info(), torch_device=torch.cuda.get_device_name(0), solves=[], quality={})
    lines = ["GPU: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (res["torch_device"], res["card"])]
    print(lines[0], flush=True)
    with onb.Context(64, planes=False) as ctx:
        for cards in SETS3:
            res["solves"].append(solve_levels(ctx, cards, 3, lines))
            print("\n".join(lines[-25:]), flush=True)
            write(a.out, res, lines)
        if not a.skip_four:
            res["solves"].append(solve_levels(ctx, SET4, 4, lines))
            print("\n".join(lines[-25:]), flush=True)
            write(a.out, res, lines)

    # move quality on positions with a decided value of the first set's <= 3-pawn table
    n = a.positions
    rng = np.random.default_rng(2026)
    with onb.Context(n, seed=1, mcts_max_sims=800, planes=True) as ctx:
        ctx.tb_solve(SETS3[0], 3)
        tables = {(p, q): ctx.tb_table(p, q).cpu().numpy() for p in range(4) for q in range(4) if p + q <= 3}
        pools = {k: np.nonzero((t != onb.TB_NONE) & (t != 0))[0] for k, t in tables.items()}
        keys = sorted(pools)
        weight = np.array([len(pools[k]) for k in keys], np.float64)
        picks = []
        for c in rng.choice(len(keys), n, p=weight / weight.sum()):  # uniform over the entries with a decided value
            k = keys[c]
            picks.append((k, int(pools[k][rng.integers(0, len(pools[k]))])))
        vals = np.array([int(tables[k][i]) for k, i in picks])
        del tables, pools
        st = np.concatenate([onb.tb_states(SETS3[0], 5 * p + q, [i]) for (p, q), i in picks])
        won = vals > 0

        def measure(name, run):
            ctx.set_states(st)
            t0 = time.perf_counter()
            run()
            ctx.sync()
            dt = time.perf_counter() - t0
            after = ctx.get_states()
            child = ctx.tb_probe().astype(np.int32)
            kept_won = (after["result"] != 0) | (child < 0)
            share_won = float(kept_won[won].mean())
            res["quality"][name] = dict(won_kept=share_won, overall_kept=float((kept_won | ~won).mean()), n_won=int(won.sum()),
                                        n=int(n), seconds=dt)
            lines.append("%-28s keeps %.4f of %d won positions (%.4f of all %d), %.2f s" % (name, share_won, int(won.sum()),
                                                                                          float((kept_won | ~won).mean()), n, dt))
            print(lines[-1], flush=True)

        def puct(sims, evaluator=onb.EVAL_UNIFORM):
            def run():
                ctx.mcts_begin(2.0, sims)
                ctx.mcts_run(evaluator, sims)
                ctx.mcts_finish(to_host=False)
                ctx.mcts_play_best()
            return run

        def gumbel(sims):
            def run():
                ctx.set_gumbel(True, m=16, seed=1)
                puct(sims)()
                ctx.set_gumbel(False)
            return run

        def alphabeta(depth):
            def run():
                ctx.alphabeta(depth, to_host=False)
                ctx.step(None)
            return run

        lines.append("move quality on %d positions with a decided value, cards %s, <= 3 pawns (%d won, %d lost)"
                     % (n, SETS3[0], int(won.sum()), int((~won).sum())))
        measure("PUCT uniform 64", puct(64))
        measure("PUCT uniform 800", puct(800))
        measure("Gumbel m=16 uniform 32", gumbel(32))
        measure("alpha-beta depth 4", alphabeta(4))
        measure("alpha-beta depth 6", alphabeta(6))
        ctx.net_load(lively_model(3, seed=7).state_dict(), precision="f16")
        measure("PUCT 800 seeded net f16", puct(800, onb.EVAL_NET))

    write(a.out, res, lines)


def write(out, res, lines):
    """the results so far (written after every part, so a long 4-pawn solve leaves the 3-pawn results behind)"""
    with open(os.path.join(out, "tablebase_speed.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(out, "tablebase_speed.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
