#!/usr/bin/env python3
"""One AlphaZero iteration on the GPU hot path, shaped like the reference's train() (alphazero-training/src/train.rs:158-412):

    self-play (train-mode noise, network-guided PUCT, every slot kept busy)  ->  replay ring buffer
    ->  a few SGD minibatches with alphaloss  ->  arena: the trained network against the `Random` and `Mcts` agents.

Everything game-, search- and inference-related runs in libonb.so: the current weights are handed to the library with
onb_net_load after every update and evaluated by the tensor-core kernel between select and expand. The optimiser, the
backward pass and the bookkeeping are plain PyTorch / Python (out of scope of the hot path).
Usage: python examples/selfplay_train_loop.py [--slots 256] [--games 512] [--sims 64] [--iters 2] [--hidden {64,128}] [--torch-net]
       [--temp-plies 30 --temperature 1 --resign-fp 0.05]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import onitama_alphazero_b200 as onb
from onitama_alphazero_b200.net import ConvResNet, alphaloss, make_evaluator


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, default=256, help="concurrent games on the device")
    ap.add_argument("--games", type=int, default=512, help="self-play games per iteration")
    ap.add_argument("--sims", type=int, default=64)
    ap.add_argument("--iters", type=int, default=2)
    ap.add_argument("--max-plies", type=int, default=40)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--sgd-steps", type=int, default=20)
    ap.add_argument("--eval-games", type=int, default=64)
    ap.add_argument("--mcts-playouts", type=int, default=200, help="playouts of the plain-UCT arena opponent")
    ap.add_argument("--ab-depth", type=int, default=4, help="search depth in plies (1..8) of the alpha-beta arena opponent")
    ap.add_argument("--torch-net", action="store_true", help="evaluate with the PyTorch module as a black box instead of onb_net_load")
    ap.add_argument("--reuse", action="store_true", help="keep the played child's subtree between moves in self-play (onb_mcts_set_reuse; "
                                                         "--sims then counts root visits, kept ones included; not with --torch-net)")
    ap.add_argument("--gumbel", type=int, default=0, metavar="M",
                    help="self-play with the Gumbel root search over M considered actions (onb_mcts_set_gumbel) and train on its improved "
                         "policy instead of PUCT with root noise; the arena adds Gumbel(--sims) against PUCT(--sims)")
    ap.add_argument("--gumbel-interior", action="store_true",
                    help="with --gumbel: Gumbel MuZero, interior selection below the root instead of PUCT (onb_gumbel_config.interior)")
    ap.add_argument("--temp-plies", type=int, default=0, help="AlphaZero's opening temperature: the first N plies of a self-play game sample "
                                                               "their move in proportion to N^(1/temperature) (onb_self_play_set_protocol)")
    ap.add_argument("--temperature", type=float, default=1.0)
    ap.add_argument("--resign-fp", type=float, default=None, metavar="F",
                    help="AlphaGo Zero's resignation: the first iteration holds out every game, each later one resigns below the threshold "
                         "calibrated on the previous iteration's held-out games for a false-positive rate F, holding out 10%% of its games")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="directory for the reference's on-disk artefacts: loss_stats JSON (stats.rs) and .ot checkpoints (train.rs:414-430)")
    ap.add_argument("--hidden", type=int, default=64, choices=[64, 128], help="hidden channels of the ConvResNet (both run on the tensor cores)")
    ap.add_argument("--net-precision", default="f32", choices=["f32", "f16", "tf32"], help="arithmetic of the on-device network (f32 = the reference's)")
    args = ap.parse_args(argv)

    torch.manual_seed(args.seed)
    model = ConvResNet(args.hidden, 21, 3).cuda().eval()
    opt = torch.optim.SGD(model.parameters(), lr=1e-2, weight_decay=1e-4)  # train.rs:181-186
    replay = onb.ReplayBuffer(200_000, device="cuda")
    log = []
    from onitama_alphazero_b200.stats import Stats
    stats_log = Stats(root=os.path.join(args.out, "loss_stats")) if args.out else None

    def evaluator_for(ctx):
        """(evaluator id, torch callable) for Context.search_device"""
        if args.torch_net:
            return onb.EVAL_UNIFORM, make_evaluator(model)
        ctx.net_load(model, precision=args.net_precision)   # BatchNorm folded, weights laid out for the tensor cores
        return onb.EVAL_NET, None

    if args.gumbel and args.reuse:
        ap.error("--gumbel does not combine with --reuse")
    if args.gumbel_interior and not args.gumbel:
        ap.error("--gumbel-interior needs --gumbel M")
    gumbel = dict(m=args.gumbel, seed=args.seed, interior=args.gumbel_interior) if args.gumbel else None
    if args.reuse and args.torch_net:
        ap.error("--reuse needs the on-device network (a PyTorch module drives the split phase, which tree reuse does not support)")
    if args.temp_plies and args.gumbel:
        ap.error("--temp-plies does not combine with --gumbel (Gumbel plays its sequential-halving winner)")
    resign_below = None   # the threshold calibrated on the previous iteration's held-out games
    for it in range(args.iters):
        protocol = None
        if args.temp_plies or args.resign_fp is not None:
            protocol = dict(temp_plies=args.temp_plies, temperature=args.temperature, seed=args.seed + 7 * it)
            if args.resign_fp is not None:   # the first iteration (no threshold yet) holds out every game
                protocol.update(resign=True, resign_below=resign_below if resign_below is not None else -1.0,
                                resign_holdout=0.1 if resign_below is not None else 1.0)
        # ---- self-play (train.rs:218-245): train-mode root noise, the current network as evaluator, finished slots restart at once
        with onb.Context(args.slots, seed=args.seed + it, mcts_max_sims=args.sims) as ctx:
            ev, net = evaluator_for(ctx)
            if net is None:   # the whole loop inside the library (onb_self_play)
                data = ctx.self_play_native(2.0, args.sims, args.games, max_plies=args.max_plies, evaluator=ev, train=not gumbel,
                                            noise_seed=args.seed + 1000 * it, reuse=args.reuse, gumbel=gumbel, protocol=protocol or False)
            else:             # the same loop driven from Python, the PyTorch module between select and expand
                data = onb.self_play_continuous(ctx, 2.0, args.sims, n_games=args.games, max_plies=args.max_plies, evaluator=ev, net=net,
                                                train=not gumbel, noise_seed=args.seed + 1000 * it, gumbel=gumbel, protocol=protocol)
        if args.resign_fp is not None:
            v = onb.resign_threshold(data["held_out"], args.resign_fp)
            if np.isfinite(v):   # +inf: too few held-out games to bound the false positives; keep holding out every game
                resign_below = v
        replay.add(data["planes"], data["pi"], data["z"])
        # ---- training (train.rs:264-339)
        model.train()
        losses = []
        for _ in range(args.sgd_steps):
            x, pi, z = replay.sample(args.batch)
            p, v = model(x)
            vl, pl = alphaloss(v, p, pi, z)
            opt.zero_grad()
            (vl + pl).backward()
            opt.step()
            losses.append((float(vl.detach()), float(pl.detach())))
        model.eval()
        # ---- evaluation (evaluator.rs:195-353): the network-guided search against the Random, the Mcts and the AlphaBeta agent,
        #      colours alternate
        a_is_red = (np.arange(args.eval_games) % 2) == 0
        counter = {"i": 0}
        results = {}
        with onb.Context(args.eval_games, seed=10_000 + it, mcts_max_sims=max(args.sims, args.mcts_playouts), planes=False) as ctx:
            ev, net = evaluator_for(ctx)

            def az(cx):
                cx.search_device(2.0, args.sims, evaluator=ev, net=net)
                cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

            def rnd(cx):
                cx.choose_random(counter["i"], policy=onb.POLICY_AGENT)
                counter["i"] += 1

            def plain_mcts(cx):
                cx.uct_search(2.0 ** 0.5, 5, args.mcts_playouts, to_host=False)
                cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

            def alphabeta(cx):
                cx.alphabeta(args.ab_depth, to_host=False)   # leaves the chosen actions in BUF_ACTIONS

            def gumbel_az(cx):   # the Gumbel agent of onb_fight: step = ply (one search per ply and agent)
                cx.set_gumbel(True, m=args.gumbel, seed=cx.seed, step0=counter["ply"], interior=args.gumbel_interior)
                cx.search_device(2.0, args.sims, evaluator=ev, net=net)
                cx.set_gumbel(False)
                cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))
                counter["ply"] += 1

            fights = [("random", az, rnd, ctx.agent_puct(args.sims, 2.0, ev, 0), ctx.agent_random()),
                      ("mcts", az, plain_mcts, ctx.agent_puct(args.sims, 2.0, ev, 0), ctx.agent_uct(args.mcts_playouts)),
                      ("alphabeta", az, alphabeta, ctx.agent_puct(args.sims, 2.0, ev, 0), ctx.agent_alphabeta(args.ab_depth))]
            if args.gumbel:
                fights.append(("gumbel_vs_puct", gumbel_az, az, ctx.agent_gumbel(args.sims, args.gumbel, 0.1, ev, 0, args.gumbel_interior),
                               ctx.agent_puct(args.sims, 2.0, ev, 0)))
            for name, mine, opponent, native_a, native in fights:
                ctx.reset()
                counter["ply"] = 0
                if net is None:   # the arena loop inside the library (onb_fight)
                    w, l, d, _ = ctx.fight_native(native_a, native, a_is_red, max_plies=150)
                else:
                    w, l, d = onb.fight(ctx, mine, opponent, a_is_red, max_plies=150)
                # FightStatistics incl. the Elo fold: on the device for the native arena (onb_fight_stats), on the host otherwise
                stats = ctx.fight_stats(history=True) if net is None else onb.fight_statistics(ctx.last_fight_results, a_is_red)
                elo = stats["rating_a"] if isinstance(stats, dict) else stats.rating_a
                results[name] = dict(wins=w, losses=l, draws=d, elo=elo, stats=stats)
        if stats_log is not None:   # what train() leaves on disk: the loss / arena log and the checkpoint of the iteration
            stats_log.push(it, losses[-1][0] + losses[-1][1], losses[-1][0], losses[-1][1])
            stats_log.push_games_played(int(data["games"]), int(data["planes"].shape[0]))
            stats_log.push_fight(False, random_fight=results["random"]["stats"], mcts_fight=results["mcts"]["stats"],
                                 alphabeta_fight=results["alphabeta"]["stats"])
            stats_log.save()
            model.save_ot(os.path.join(args.out, "model_%d.ot" % it))
        for r in results.values():
            r.pop("stats")
        log.append(dict(iteration=it, games=int(data["games"]), samples=int(data["planes"].shape[0]), replay=replay.size,
                        value_loss=losses[-1][0], policy_loss=losses[-1][1], wins=results["random"]["wins"],
                        losses=results["random"]["losses"], draws=results["random"]["draws"], elo=results["random"]["elo"],
                        vs_mcts=results["mcts"], vs_alphabeta=results["alphabeta"],
                        **({"gumbel_vs_puct": results["gumbel_vs_puct"]} if args.gumbel else {}),
                        **({"resigned": data["resigned"], "held_out": int(data["held_out"]["result"].shape[0]), "resign_below": resign_below}
                           if args.resign_fp is not None else {})))
        print(log[-1], flush=True)
    return log


if __name__ == "__main__":
    main()
