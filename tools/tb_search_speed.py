"""Cost and strength of tablebase leaves (onb_mcts_set_tablebase, ONB_AGENT_PUCT_TB, DESIGN.md §5i).

    python tools/tb_search_speed.py --out DIR

Reports:
  * ms per ply, switch on and off: 16 384 trees x 800 simulations on roots of the set {0,1,2,3,11} one pawn above its 3-pawn table
    (so the searches reach table leaves), the reference's trained 3-block weights (tests/golden/net_golden.npz) through ONB_EVAL_NET
    in f16 and in f32-faithful arithmetic; host clock around begin + run + finish ending in a synchronise, median of --reps;
  * ms per move for one game (the same kind of root, 800 simulations, f16) at K = 1 and K = 16 (virtual loss 1), on and off;
  * the uniform evaluator's cost of leaving the fused kernel (config-4 shape: 16 384 trees x 400 simulations) on dealt mid-game roots
    and on the set's roots; and the probe's cost per round from torch.profiler (expand/backup kernel time with and without the table);
  * strength in onb_fight: --games games per start level, ONB_AGENT_PUCT_TB against ONB_AGENT_PUCT at equal simulations (both on the
    trained weights in f16), every start position played twice with the colours swapped, ply cap 150, from positions one and two
    pawns above the 3-pawn and the 4-pawn table;
  * "won position stays won" on 16 384 positions with a decided value of the <= 3-pawn table (as DESIGN.md §5g measures it) for PUCT
    with the uniform evaluator and tablebase leaves, the search alone (the root is not probed: the move is the search's).
Writes tb_search_speed.json and tb_search_speed.txt into DIR; the card's name and power limit are read in the same run."""
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

CARDS = [0, 1, 2, 3, 11]
RED_TEMPLE_KING, BLUE_TEMPLE_KING = 1 << (31 - 2), 1 << (31 - 22)  # a king on the enemy temple: a decided position


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def above(onb, rng, level, n):
    """n undecided positions of the set with `level` pawns (every split p + q = level), in random order"""
    from tablebase_oracle import entries
    cls = [(p, level - p) for p in range(level + 1) if p <= 4 and level - p <= 4]
    st = np.concatenate([onb.tb_states(CARDS, 5 * p + q, rng.integers(0, entries(p, q), 2 * n // len(cls) + 1)) for p, q in cls])
    st = st[(st["kings"][:, 0] != RED_TEMPLE_KING) & (st["kings"][:, 1] != BLUE_TEMPLE_KING)]
    return np.ascontiguousarray(st[rng.permutation(len(st))[:n]])


def search_ms(ctx, onb, roots, sims, evaluator, tb, reps, warmup, leaves=1):
    """median ms of begin + run + finish over `reps` searches of the same roots, host clock, ending in a synchronise"""
    ctx.set_virtual_loss(leaves, 1.0)
    ctx.set_tablebase(tb)
    times = []
    for r in range(warmup + reps):
        ctx.set_states(roots)
        ctx.sync()
        t0 = time.perf_counter()
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(evaluator, sims)
        ctx.mcts_finish(to_host=False)
        ctx.sync()
        if r >= warmup:
            times.append((time.perf_counter() - t0) * 1e3)
    ctx.set_virtual_loss(1)
    ctx.set_tablebase(False)
    return float(np.median(times))


def kernel_us(onb, ctx, roots, sims, tb):
    """CUDA time per launch of the split-phase kernels over one search (torch.profiler, after the timings)"""
    from torch.profiler import ProfilerActivity, profile
    ctx.set_tablebase(tb)
    ctx.set_states(roots)
    ctx.search_device(2.0, sims, evaluator=onb.EVAL_UNIFORM)  # warm-up
    ctx.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.set_states(roots)
        ctx.mcts_begin(2.0, sims)
        for _ in range(sims):  # the split phase, also with the switch off
            ctx.mcts_select()
            ctx.mcts_eval(onb.EVAL_UNIFORM)
            ctx.mcts_expand_backup()
        ctx.mcts_finish(to_host=False)
        ctx.sync()
    ctx.set_tablebase(False)
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0 and "k_" in e.key:
            out[e.key[:80]] = dict(calls=int(e.count), mean_us=float(t) / max(1, int(e.count)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for tb_search_speed.json and tb_search_speed.txt")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--moves", type=int, default=20)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--fight-sims", type=int, default=200)
    ap.add_argument("--skip-fight", action="store_true")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    import oracle_lib as O
    import onitama_alphazero_b200 as onb
    from test_net_cpu import golden_tensors
    if not torch.cuda.is_available():
        raise SystemExit("tb_search_speed.py measures on the GPU; no CUDA device found")
    card = card_info()
    weights = golden_tensors()
    rng = np.random.default_rng(2026)
    res = dict(card=card, cards=CARDS, ply=[], move=[], uniform=[], kernels={}, fights=[], quality={})
    lines = ["# tablebase leaves (DESIGN.md §5i), card: %s" % card, "# set %s; host clock, median, ending in a synchronise" % CARDS]

    def out(s):
        lines.append(s)
        print(s, flush=True)

    n = 16384
    roots4 = above(onb, rng, 4, n)  # one pawn above the 3-pawn table
    g = O.new_games(2 * n, seed=3)  # dealt mid-game roots: 12 random plies (config 4's kind of root)
    for step in range(12):
        O.env_step_random(g, 3, step)
    dealt = np.ascontiguousarray(g[g["result"] == 0][:n])

    # ms per ply, 16 384 trees x 800 simulations, trained weights
    for precision in ("f16", "f32"):
        with onb.Context(n, seed=1, mcts_max_sims=800, planes=False) as ctx:
            ctx.tb_solve(CARDS, 3)
            ctx.net_load(weights, precision=precision)
            row = {tb: search_ms(ctx, onb, roots4, 800, onb.EVAL_NET, tb, a.reps, a.warmup) for tb in (False, True)}
        res["ply"].append(dict(precision=precision, trees=n, sims=800, off_ms=row[False], on_ms=row[True]))
        out("ms per ply, %d trees x 800 sims, trained weights %s, 4-pawn roots of the set: off %.1f, on %.1f (%.3f x)"
            % (n, precision, row[False], row[True], row[True] / row[False]))

    # ms per move, one game, 800 simulations, f16, K = 1 / 16
    with onb.Context(1, seed=1, mcts_max_sims=800, planes=False) as ctx:
        ctx.tb_solve(CARDS, 3)
        ctx.net_load(weights, precision="f16")
        for k in (1, 16):
            row = {tb: search_ms(ctx, onb, roots4[:1], 800, onb.EVAL_NET, tb, a.moves, 2, leaves=k) for tb in (False, True)}
            res["move"].append(dict(leaves=k, sims=800, off_ms=row[False], on_ms=row[True]))
            out("ms per move, one game, 800 sims, f16, K = %d: off %.2f, on %.2f" % (k, row[False], row[True]))

    # the uniform evaluator: fused kernel (off) against split rounds with table leaves (on), config-4 shape
    with onb.Context(n, seed=1, mcts_max_sims=400, planes=False) as ctx:
        ctx.tb_solve(CARDS, 3)
        for name, roots in (("dealt mid-game roots", dealt), ("4-pawn roots of the set", roots4)):
            row = {tb: search_ms(ctx, onb, roots, 400, onb.EVAL_UNIFORM, tb, a.reps, a.warmup) for tb in (False, True)}
            res["uniform"].append(dict(roots=name, trees=n, sims=400, fused_off_ms=row[False], split_on_ms=row[True]))
            out("uniform evaluator, %d trees x 400 sims, %s: fused (off) %.2f ms, split rounds with table leaves (on) %.2f ms (%.1f x)"
                % (n, name, row[False], row[True], row[True] / row[False]))
        for tb in (False, True):
            ks = kernel_us(onb, ctx, roots4, 64, tb)
            res["kernels"]["on" if tb else "off"] = ks
            out("# split-phase kernels per launch, %d trees, 64 sims, uniform, 4-pawn roots of the set, switch %s (torch.profiler)"
                % (n, "on" if tb else "off"))
            for k, v in sorted(ks.items(), key=lambda kv: -kv[1]["mean_us"]):
                out("  %-80s %6d calls %9.2f us" % (k, v["calls"], v["mean_us"]))

    # won position stays won, the search alone, <= 3-pawn table
    m = 16384
    with onb.Context(m, seed=1, mcts_max_sims=800, planes=False) as ctx:
        ctx.tb_solve(CARDS, 3)
        tables = {(p, q): ctx.tb_table(p, q).cpu().numpy() for p in range(4) for q in range(4) if p + q <= 3}
        pools = {k: np.nonzero((t != onb.TB_NONE) & (t != 0))[0] for k, t in tables.items()}
        keys = sorted(pools)
        weight = np.array([len(pools[k]) for k in keys], np.float64)
        picks = []
        for c in rng.choice(len(keys), m, p=weight / weight.sum()):
            k = keys[c]
            picks.append((k, int(pools[k][rng.integers(0, len(pools[k]))])))
        vals = np.array([int(tables[k][i]) for k, i in picks])
        del tables, pools
        st = np.concatenate([onb.tb_states(CARDS, 5 * p + q, [i]) for (p, q), i in picks])
        won = vals > 0
        for sims in (64, 800):
            for tb in (False, True):
                ctx.set_states(st)
                ctx.set_tablebase(tb)
                ctx.mcts_begin(2.0, sims)
                ctx.mcts_run(onb.EVAL_UNIFORM, sims)
                ctx.mcts_finish(to_host=False)
                ctx.mcts_play_best()
                ctx.set_tablebase(False)
                after = ctx.get_states()
                child = ctx.tb_probe().astype(np.int32)
                kept = float(((after["result"] != 0) | (child < 0))[won].mean())
                res["quality"]["PUCT uniform %d %s" % (sims, "on" if tb else "off")] = dict(won_kept=kept, n_won=int(won.sum()), n=m)
                out("won position stays won, PUCT uniform %d sims, tablebase leaves %s: %.4f of %d won positions"
                    % (sims, "on" if tb else "off", kept, int(won.sum())))

    if not a.skip_fight:
        half = a.games // 2
        a_is_red = np.arange(2 * half) % 2 == 0
        s = a.fight_sims
        for max_pawns in (3, 4):
            with onb.Context(2 * half, seed=5, mcts_max_sims=s, planes=False) as ctx:
                ctx.tb_solve(CARDS, max_pawns)
                ctx.net_load(weights, precision="f16")
                for lvl in (max_pawns + 1, max_pawns + 2):
                    if lvl > 8:
                        continue
                    start = above(onb, rng, lvl, half) if lvl <= 4 else above_many(onb, rng, lvl, half)
                    ctx.set_states(np.repeat(start, 2))
                    t0 = time.perf_counter()
                    w, l, d, _ = ctx.fight_native(ctx.agent_puct(s, 2.0, onb.EVAL_NET, tablebase=True), ctx.agent_puct(s, 2.0, onb.EVAL_NET),
                                                  a_is_red, 150)
                    dt = time.perf_counter() - t0
                    res["fights"].append(dict(max_pawns=max_pawns, start_pawns=lvl, sims=s, games=2 * half, wins=w, losses=l, draws=d, seconds=dt))
                    out("arena, %d-pawn table, starts with %d pawns, %d sims each, %d games: PUCT_TB vs PUCT W/L/D %d/%d/%d (%.1f s)"
                        % (max_pawns, lvl, s, 2 * half, w, l, d, dt))

    with open(os.path.join(a.out, "tb_search_speed.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(a.out, "tb_search_speed.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


def above_many(onb, rng, level, n):
    """n undecided positions of the set with `level` > 4 pawns: a position of the 4-pawn classes' squares is not enough, so pawns are
    added on random free squares of a 4-pawn position (at most four per side)"""
    base = above(onb, rng, 4, 4 * n)
    out = []
    for s in base:
        pr, pb = int(s["pawns"][0]), int(s["pawns"][1])
        occ = pr | pb | int(s["kings"][0]) | int(s["kings"][1])
        free = [1 << (31 - q) for q in range(25) if not occ & (1 << (31 - q))]
        need = level - bin(pr).count("1") - bin(pb).count("1")
        for sq in rng.permutation(free)[:need]:
            if bin(pr).count("1") <= bin(pb).count("1") and bin(pr).count("1") < 4:
                pr |= int(sq)
            elif bin(pb).count("1") < 4:
                pb |= int(sq)
            else:
                pr |= int(sq)
        t = s.copy()
        t["pawns"][0], t["pawns"][1] = pr, pb
        out.append(t)
        if len(out) == n:
            break
    st = np.array(out, dtype=base.dtype)
    keep = (st["kings"][:, 0] != RED_TEMPLE_KING) & (st["kings"][:, 1] != BLUE_TEMPLE_KING)
    return np.ascontiguousarray(st[keep][:n])


if __name__ == "__main__":
    main()
