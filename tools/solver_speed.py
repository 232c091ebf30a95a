"""Cost and strength of the MCTS solver (onb_mcts_set_solver, ONB_AGENT_PUCT_SOLVER, DESIGN.md §5k).

    python tools/solver_speed.py --out DIR

Reports:
  1. the fused search at config 4's shape: 16 384 trees x 400 simulations, uniform evaluator, dealt mid-game roots; solver off and on,
     alternated, host clock around begin + run + finish ending in a synchronise, median of --reps; the fused kernel's own time from
     torch.profiler; and what the two searches do: nodes per tree, levels descended per simulation (the sum of N over the non-root
     nodes of sampled trees over the simulations) and roots proven;
  2. ms per ply, 16 384 trees x 800 simulations, the reference's trained 3-block weights (tests/golden/net_golden.npz) in f16 through
     ONB_EVAL_NET, off and on, alternated;
  3. "won position stays won" on §5i's suite (positions of decided value of the set {0,1,2,3,11}'s <= 3-pawn table, drawn as
     tools/tb_search_speed.py draws them): PUCT with the uniform evaluator at 64 and 800 simulations, table leaves off, solver off and
     on, and the share of roots the solver proves;
  4. the arena: ONB_AGENT_PUCT_SOLVER against ONB_AGENT_PUCT, --games games, colours swapped, trained f16 weights, --fight-sims
     simulations, ply cap 150, from dealt starts and from 5-pawn starts of the set; and ONB_AGENT_PUCT against itself from the same
     starts as a control of the arena's colour swap.
--lib PATH measures another build of libonb.so (for example one compiled with -DONB_SOLVER_MIN_BLOCKS=7); --only-fused runs row 1.
Writes solver_speed.json and solver_speed.txt into DIR; the card's name, power limit and SM clock are read in the same run."""
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

from tb_search_speed import CARDS, above, card_info  # noqa: E402


def timed(ctx, roots, sims, evaluator, solver):
    ctx.set_states(roots)
    ctx.sync()
    t0 = time.perf_counter()
    ctx.set_solver(solver)
    ctx.mcts_begin(2.0, sims)
    ctx.mcts_run(evaluator, sims)
    ctx.mcts_finish(to_host=False)
    ctx.sync()
    dt = (time.perf_counter() - t0) * 1e3
    ctx.set_solver(False)
    return dt


def alternated(ctx, roots, sims, evaluator, reps, warmup):
    """median ms of solver off and on, the two alternated rep by rep after `warmup` rounds of both"""
    for _ in range(warmup):
        timed(ctx, roots, sims, evaluator, False)
        timed(ctx, roots, sims, evaluator, True)
    t = {False: [], True: []}
    for _ in range(reps):
        for s in (False, True):
            t[s].append(timed(ctx, roots, sims, evaluator, s))
    return float(np.median(t[False])), float(np.median(t[True])), t


def kernel_ms(onb, ctx, roots, sims, solver):
    """the fused kernel's device time per search (torch.profiler, CUDA activities), one search after a warm-up"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    timed(ctx, roots, sims, onb.EVAL_UNIFORM, solver)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        timed(ctx, roots, sims, onb.EVAL_UNIFORM, solver)
        torch.cuda.synchronize()
    tot = {}
    for e in prof.key_averages():
        if "k_mcts" in e.key:
            tot[e.key] = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
    return tot


def shape(onb, ctx, roots, sims, solver, sample=256):
    """what one search does: mean nodes per tree, levels descended per simulation (sampled trees) and the share of roots proven"""
    timed(ctx, roots, sims, onb.EVAL_UNIFORM, solver)
    nn, _ = ctx.mcts_tree_info()
    levels = 0
    idx = np.linspace(0, len(roots) - 1, sample).astype(int)
    for t in idx:
        tr = ctx.mcts_dump_tree(int(t))
        levels += int(tr["visits"][1:].sum())
    proof = ctx.root_proof() if solver else np.zeros(len(roots), np.int8)
    return dict(nodes_per_tree=float(nn.mean()), levels_per_sim=levels / float(len(idx) * sims), roots_proven=float((proof != 0).mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for solver_speed.json and solver_speed.txt")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--fight-sims", type=int, default=200)
    ap.add_argument("--skip-ply", action="store_true")
    ap.add_argument("--skip-fight", action="store_true")
    ap.add_argument("--only-fused", action="store_true")
    ap.add_argument("--lib", default=None, help="another build of libonb.so to measure")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if a.lib:
        import onitama_alphazero_b200._lib as L
        L.LIB_PATH = os.path.abspath(a.lib)
    import torch
    import oracle_lib as O
    import onitama_alphazero_b200 as onb
    from test_net_cpu import golden_tensors
    if not torch.cuda.is_available():
        raise SystemExit("solver_speed.py measures on the GPU; no CUDA device found")
    card = card_info()
    res = dict(card=card, lib=a.lib or "libonb.so", fused=None, ply=None, quality={}, fights=[])
    lines = ["# MCTS solver (DESIGN.md §5k), card (name, power limit, max SM clock): %s" % card,
             "# host clock around begin + run + finish ending in a synchronise, median, solver off / on alternated"]

    def out(s):
        lines.append(s)
        print(s, flush=True)

    n = 16384
    g = O.new_games(2 * n, seed=3)  # dealt mid-game roots: 12 random plies (config 4's kind of root)
    for step in range(12):
        O.env_step_random(g, 3, step)
    dealt = np.ascontiguousarray(g[g["result"] == 0][:n])

    # 1. the fused search, config-4 shape
    with onb.Context(n, seed=1, mcts_max_sims=400, planes=False) as ctx:
        off, on, raw = alternated(ctx, dealt, 400, onb.EVAL_UNIFORM, a.reps, a.warmup)
        kern = {s: kernel_ms(onb, ctx, dealt, 400, s) for s in (False, True)}
        shp = {s: shape(onb, ctx, dealt, 400, s) for s in (False, True)}
    res["fused"] = dict(trees=n, sims=400, off_ms=off, on_ms=on, ratio=on / off, off_all=raw[False], on_all=raw[True],
                        kernels_ms={"off": kern[False], "on": kern[True]}, shape={"off": shp[False], "on": shp[True]})
    out("1. fused search, %d trees x 400 sims, uniform, dealt roots (%s): off %.2f ms, on %.2f ms (%.3f x)"
        % (n, res["lib"], off, on, on / off))
    for s in (False, True):
        out("   solver %s: kernels %s; %.1f nodes per tree, %.3f levels per simulation, roots proven %.4f"
            % ("on " if s else "off", ", ".join("%s %.2f ms" % (k.split("(")[0], v) for k, v in kern[s].items()), shp[s]["nodes_per_tree"],
               shp[s]["levels_per_sim"], shp[s]["roots_proven"]))
    if a.only_fused:
        a.skip_ply = a.skip_fight = True

    # 2. per ply with the trained network in f16
    if not a.skip_ply:
        with onb.Context(n, seed=1, mcts_max_sims=800, planes=False) as ctx:
            ctx.net_load(golden_tensors(), precision="f16")
            off, on, raw = alternated(ctx, dealt, 800, onb.EVAL_NET, max(3, a.reps // 2), 1)
        res["ply"] = dict(trees=n, sims=800, off_ms=off, on_ms=on, ratio=on / off)
        out("2. ms per ply, %d trees x 800 sims, trained weights f16: off %.1f, on %.1f (%.3f x)" % (n, off, on, on / off))

    # 3. won position stays won: tools/tb_search_speed.py's suite (same generator, same draws)
    if a.only_fused:
        return finish(a, res, lines)
    rng = np.random.default_rng(2026)
    above(onb, rng, 4, n)  # the draws tb_search_speed.py makes before its suite
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
            for solver in (False, True):
                ctx.set_states(st)
                ctx.set_solver(solver)
                ctx.mcts_begin(2.0, sims)
                ctx.mcts_run(onb.EVAL_UNIFORM, sims)
                ctx.mcts_finish(to_host=False)
                proof = ctx.root_proof() if solver else np.zeros(m, np.int8)
                ctx.mcts_play_best()
                ctx.set_solver(False)
                after = ctx.get_states()
                child = ctx.tb_probe().astype(np.int32)
                kept = float(((after["result"] != 0) | (child < 0))[won].mean())
                proven = float((proof[won] == 1).mean())
                wrong = int(((proof != 0) & (np.sign(vals) != proof)).sum())
                res["quality"]["PUCT uniform %d solver %s" % (sims, "on" if solver else "off")] = dict(
                    won_kept=kept, won_proven=proven, proofs_against_table=wrong, n_won=int(won.sum()), n=m)
                out("3. won position stays won, PUCT uniform %d sims, solver %s: %.4f of %d won positions; proven +1: %.4f; proofs against "
                    "the table: %d" % (sims, "on" if solver else "off", kept, int(won.sum()), proven, wrong))

    # 4. arena
    if not a.skip_fight:
        half = a.games // 2
        a_is_red = np.arange(2 * half) % 2 == 0
        s = a.fight_sims
        gd = O.new_games(half, seed=9)
        starts = (("dealt", np.ascontiguousarray(gd)), ("5-pawn starts of the set", None))
        with onb.Context(2 * half, seed=5, mcts_max_sims=s, planes=False) as ctx:
            ctx.net_load(golden_tensors(), precision="f16")
            for name, start in starts:
                if start is None:
                    from tb_search_speed import above_many
                    start = above_many(onb, np.random.default_rng(7), 5, half)
                ctx.set_states(np.repeat(start, 2))
                t0 = time.perf_counter()
                w, l, d, _ = ctx.fight_native(ctx.agent_puct(s, 2.0, onb.EVAL_NET, solver=True), ctx.agent_puct(s, 2.0, onb.EVAL_NET), a_is_red, 150)
                dt = time.perf_counter() - t0
                res["fights"].append(dict(starts=name, sims=s, games=2 * half, wins=w, losses=l, draws=d, seconds=dt))
                out("4. arena, %s, %d sims each, %d games: PUCT_SOLVER vs PUCT W/L/D %d/%d/%d (%.1f s)" % (name, s, 2 * half, w, l, d, dt))
                ctx.set_states(np.repeat(start, 2))
                w, l, d, _ = ctx.fight_native(ctx.agent_puct(s, 2.0, onb.EVAL_NET), ctx.agent_puct(s, 2.0, onb.EVAL_NET), a_is_red, 150)
                res["fights"].append(dict(starts=name, control=True, sims=s, games=2 * half, wins=w, losses=l, draws=d))
                out("4. control, %s, %d sims each, %d games: PUCT vs PUCT W/L/D %d/%d/%d" % (name, s, 2 * half, w, l, d))

    finish(a, res, lines)


def finish(a, res, lines):
    with open(os.path.join(a.out, "solver_speed.json"), "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.join(a.out, "solver_speed.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
