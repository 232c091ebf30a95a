"""Games per second and plies per game of native self-play with AlphaZero's move protocol (onb_self_play_set_protocol, DESIGN.md §5j).

    python tools/selfplay_protocol_speed.py --out DIR [--slots 2048] [--sims 800] [--games 4096]

onb_self_play over --slots slots at --sims simulations, train-mode root noise, the reference's trained 3-block weights
(tests/golden/net_golden.npz) through ONB_EVAL_NET in f16, the reference's ply cap of 150. Settings, each one timed run (host clock
around onb_self_play, which ends in a synchronise) after an untimed warm-up:
  * off: the protocol off (the most visited move, no resignation);
  * temp: T = 30, tau = 1, resignation off;
  * calibrate: T = 30, tau = 1, resignation on with every game held out (h = 1), so nothing resigns and every game leaves a record:
    these records calibrate v_resign for a 5 % false-positive rate (selfplay.resign_threshold);
  * resign_only: resignation below that v_resign with h = 0, no temperature (T = 0), to separate the two effects;
  * resign: T = 30, tau = 1 and resignation below that v_resign with h = 0;
  * resign_h10: the same with h = 0.1; the false-positive rate observed among its held-out games (a side that did not lose had
    min m < v_resign) is reported.
Then, in a run of its own, torch.profiler's CUDA time per ply of the protocol's kernels (k_mcts_choose, k_sp_resign, k_sp_over_pr,
k_sp_records, k_sp_finish_pr) over a few plies of the same setting. Writes selfplay_protocol_speed.json and .txt into DIR; the card's
name, power limit and maximum SM clock are read in the same run."""
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

KERNELS = ("k_mcts_choose", "k_sp_resign", "k_sp_over_pr", "k_sp_records", "k_sp_finish_pr", "k_sp_proto_init")


def card_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def run(onb, ctx, args, protocol):
    ctx.sync()
    t0 = time.perf_counter()
    r = ctx.self_play_native(2.0, args.sims, args.games, max_plies=150, evaluator=onb.EVAL_NET, train=True, noise_seed=args.seed, protocol=protocol)
    ctx.sync()
    dt = time.perf_counter() - t0
    assert not r["truncated"]
    out = dict(seconds=dt, games=r["games"], samples=int(r["z"].shape[0]), plies_run=r["plies_run"], games_per_s=r["games"] / dt,
               plies_per_game=int(r["z"].shape[0]) / r["games"])
    if protocol:
        out.update(resigned=r["resigned"], held_out=int(r["held_out"]["result"].shape[0]))
    return out, r


def false_positives(held, v):
    """held-out games in which a side that did not lose had min m < v"""
    res, mm = held["result"].cpu().numpy(), held["min_m"].cpu().numpy()
    return int((((res != 2) & (mm[:, 0] < v)) | ((res != 1) & (mm[:, 1] < v))).sum())


def profile_plies(onb, torch, ctx, args, protocol):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = ctx.self_play_native(2.0, args.sims, ctx.n, max_plies=args.profile_plies - 2, evaluator=onb.EVAL_NET, train=True, noise_seed=args.seed,
                                 protocol=protocol)
        ctx.sync()
    plies = r["plies_run"]
    per = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key and "DeviceToHost" not in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                per[k] = dict(calls=int(e.count), us_total=float(t), us_per_ply=float(t) / plies, us_per_call=float(t) / max(1, e.count))
    total = sum(getattr(e, "device_time_total", 0.0) or 0.0 for e in prof.key_averages())
    return dict(plies=plies, kernels=per, all_kernels_us_per_ply=total / plies)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--slots", type=int, default=2048)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--fp", type=float, default=0.05)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--profile-plies", type=int, default=6)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import torch

    import onitama_alphazero_b200 as onb
    from test_net_cpu import load_net_golden
    card = card_info()
    weights = load_net_golden()[0]
    res = dict(card=card, slots=args.slots, sims=args.sims, games=args.games, evaluator="ONB_EVAL_NET f16, reference's trained 3-block weights",
               train_noise=True, max_plies=150, fp=args.fp, settings={})
    with onb.Context(args.slots, seed=args.seed, mcts_max_sims=args.sims) as ctx:
        ctx.net_load(weights, precision="f16")
        ctx.self_play_native(2.0, args.sims, args.slots, max_plies=4, evaluator=onb.EVAL_NET, train=True, noise_seed=99)   # warm-up
        temp = dict(temp_plies=30, temperature=1.0, seed=args.seed)
        res["settings"]["off"], _ = run(onb, ctx, args, False)
        res["settings"]["temp"], _ = run(onb, ctx, args, temp)
        res["settings"]["calibrate"], r = run(onb, ctx, args, dict(temp, resign=True, resign_below=-1.0, resign_holdout=1.0))
        v = onb.resign_threshold(r["held_out"], args.fp)
        res["v_resign"] = v
        res["calibration_false_positives_at_v"] = false_positives(r["held_out"], v)
        if np.isfinite(v):
            res["settings"]["resign_only"], _ = run(onb, ctx, args, dict(resign=True, resign_below=v, resign_holdout=0.0, seed=args.seed))
            res["settings"]["resign"], _ = run(onb, ctx, args, dict(temp, resign=True, resign_below=v, resign_holdout=0.0))
            res["settings"]["resign_h10"], r = run(onb, ctx, args, dict(temp, resign=True, resign_below=v, resign_holdout=0.1))
            g = int(r["held_out"]["result"].shape[0])
            fp = false_positives(r["held_out"], v)
            res["settings"]["resign_h10"].update(false_positives=fp, false_positive_rate=fp / g if g else float("nan"))
        res["profile"] = profile_plies(onb, torch, ctx, args, dict(temp, resign=True, resign_below=v if np.isfinite(v) else -1.0, resign_holdout=0.1))
    res["card_after"] = card_info()
    with open(os.path.join(args.out, "selfplay_protocol_speed.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = ["self-play move protocol, onb_self_play: %d slots x %d simulations, %d games, f16 trained 3-block net, train-mode noise" %
             (args.slots, args.sims, args.games), "card (name, power limit, max SM clock): " + card, ""]
    lines.append("%-12s %10s %10s %12s %10s %9s %9s" % ("setting", "games/s", "plies/game", "seconds", "resigned", "held out", "FP rate"))
    for k, s in res["settings"].items():
        lines.append("%-12s %10.2f %10.2f %12.2f %10s %9s %9s" % (k, s["games_per_s"], s["plies_per_game"], s["seconds"], s.get("resigned", "-"),
                                                                 s.get("held_out", "-"), "%.3f" % s["false_positive_rate"] if "false_positive_rate" in s else "-"))
    lines += ["", "v_resign (calibrated at %.2f on the calibrate run's held-out games): %r" % (args.fp, v), "",
              "torch.profiler, CUDA time per ply over %d plies (T = 30, resignation, h = 0.1):" % res["profile"]["plies"]]
    for k, d in res["profile"]["kernels"].items():
        lines.append("  %-16s %9.2f us/ply  (%d calls, %.2f us/call)" % (k, d["us_per_ply"], d["calls"], d["us_per_call"]))
    lines.append("  all kernels      %9.1f us/ply" % res["profile"]["all_kernels_us_per_ply"])
    open(os.path.join(args.out, "selfplay_protocol_speed.txt"), "w").write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
