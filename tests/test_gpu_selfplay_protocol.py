"""AlphaZero's self-play move protocol (onb_self_play_set_protocol, onb_mcts_choose, DESIGN.md §5j) on the GPU: the switch off changes
nothing, k_mcts_choose against the restatement (tests/selfplay_protocol_oracle.py) bit for bit, the native loop against the Python
driver, the resignation rules and records, the temperature's effect, the refusals, the C++ mirror and the example."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import selfplay_protocol_oracle as SP
from test_gpu_parity import G
from test_gpu_vl import _roots

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def _same_run(a, b, keys=("planes", "pi", "z", "color", "serial")):
    import torch
    assert a["games"] == b["games"]
    for k in keys:
        assert torch.equal(a[k], b[k]), k


def _net_ctx(onb, ctx):
    from test_net_cpu import lively_model
    ctx.net_load(lively_model(1, seed=4))


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [0, 1, 2])
def test_off_means_unchanged(onb, evaluator):
    n, sims, games = 48, 12, 80
    runs = []
    for clear in (False, True):
        with onb.Context(n, seed=3, mcts_max_sims=sims) as ctx:
            if evaluator == 2:
                _net_ctx(onb, ctx)
            if clear:
                ctx.set_selfplay_protocol(dict(temp_plies=30, resign=True, resign_below=0.5, resign_holdout=0.5, seed=9))
                ctx.set_selfplay_protocol(None)
            runs.append([ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=evaluator, train=train, noise_seed=4)
                         for train in (False, True)])
    for a, b in zip(*runs):
        _same_run(a, b)
        assert "resigned" not in a and "resigned" not in b


def _tree_roots(ctx, n, cap=None):
    """per game: root (W, N) and the root children's visits, rewards and actions in child order"""
    out = []
    for t in range(n):
        d = ctx.mcts_dump_tree(t, cap)
        fc, k = int(d["first_child"][0]), int(d["n_child"][0])
        out.append((float(d["reward"][0]), int(d["visits"][0]), d["visits"][fc:fc + k].astype(np.int64), d["reward"][fc:fc + k],
                    d["action"][fc:fc + k].astype(np.int64), d["flags"][fc:fc + k]))
    return out


def _check_choose(onb, ctx, n, best, seed, step, tau, mask, cap=None):
    ctx.mcts_choose(seed, step, tau, mask)
    acts = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,))
    m = ctx.read(onb.BUF_ROOT_M, np.float64, (n,))
    roots = _tree_roots(ctx, n, cap)
    for g, (rw, rn, vis, rew, act, _) in enumerate(roots):
        mv, mm = SP.choose(rw, rn, vis, rew, act, int(best[g]), bool(mask[g]), tau, seed, ctx.game_id_base + g, step)
        assert int(acts[g]) == mv, (g, tau)
        assert m[g].tobytes() == np.float64(mm).tobytes(), (g, m[g], mm)
        if not mask[g]:
            assert int(acts[g]) == int(best[g])
    return roots, acts, m


@pytest.mark.gpu
@pytest.mark.parametrize("sims", [1, 2, 33, 400])
@pytest.mark.parametrize("evaluator", [0, 1])
def test_choose_equals_the_restatement(onb, evaluator, sims):
    n = 4096
    roots = _roots(n, 70 + sims + evaluator)
    case = G["reference_tests"]["no_moves"][1]   # a side to move without legal moves: its root has pass children
    roots[-8:] = O.make_state(case["deck"], pawns=case["pawns"], kings=case["kings"], side=case["color"])
    with onb.Context(n, mcts_max_sims=sims, planes=False, game_id_base=11) as ctx:
        ctx.set_states(roots)
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(evaluator, sims)
        best = ctx.mcts_finish()["best"].copy()
        rng = np.random.default_rng(sims)
        for tau in (0.5, 1.0, 2.0):
            mask = (rng.random(n) < 0.7).astype(np.uint8)
            tr, acts, m = _check_choose(onb, ctx, n, best, 5 + sims, 3, tau, mask)
        assert max(len(t[2]) for t in tr) > 32                               # roots with more than 32 children
        assert all((t[5] & 4).any() for t in tr[-8:])                          # pass children
        if sims >= 33:
            assert (acts[mask == 1] != best[mask == 1]).any()                  # sampling does change moves
        if sims == 400:   # roots with an immediate win: v_root is positive from the side to move's view
            win = [g for g, t in enumerate(tr) if (t[5] & 2).any()]
            assert win
            for g in win:
                assert -(tr[g][0] / tr[g][1]) > 0 and m[g] > 0, g


@pytest.mark.gpu
def test_choose_on_fabricated_eight_piece_roots(onb):
    # eight pieces of the side to move (a state onb_env_set_states takes as given, and the kind of root for which the expansion may
    # write more than the 40 children of a legal position; k_mcts_choose holds up to kGbStride = 64)
    rng = np.random.default_rng(0)
    red = sum(1 << (sq + 7) for sq in (5, 7, 9, 10, 14, 16, 18))
    roots = np.concatenate([O.make_state(list(rng.choice(16, 5, replace=False)), pawns=[red, 3623878656], kings=[1 << (12 + 7), 536870912], side=0)
                            for _ in range(256)])
    n, sims = len(roots), 33
    cap = 1 + 64 * (sims + 1)
    with onb.Context(n, mcts_max_sims=sims, mcts_node_cap=cap, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(1, sims)
        best = ctx.mcts_finish()["best"].copy()
        for tau in (0.5, 1.0, 2.0):
            tr, _, _ = _check_choose(onb, ctx, n, best, 4, 1, tau, np.ones(n, np.uint8), cap)
        assert max(len(t[2]) for t in tr) >= 20


@pytest.mark.gpu
def test_choose_after_a_reuse_search_follows_the_budget_order(onb):
    # tree reuse lays the trees out by remaining budget (a subset order): choose reads them through the search's game list
    n, sims = 512, 64
    roots = _roots(n, 5)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_reuse(True)
        for ply in range(3):
            ctx.mcts_begin(2.0, sims)
            ctx.mcts_run(1, sims)
            best = ctx.mcts_finish()["best"].copy()
            mask = (np.arange(n) % 3 != 0).astype(np.uint8)
            _check_choose(onb, ctx, n, best, 2, ply, 1.0, mask)
            ctx.mcts_play_best()


def _threshold(onb, ctx, sims, games, ev, **kw):
    """a v_resign that resigns some games: calibrated at fp = 0.5 on an h = 1 run"""
    cal = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=ev, protocol=dict(resign=True, resign_below=-1.0, resign_holdout=1.0, seed=1), **kw)
    assert cal["resigned"] == 0 and cal["held_out"]["result"].shape[0] == cal["games"]
    return onb.resign_threshold(cal["held_out"], 0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator,reuse", [(0, False), (0, True), (1, True), (2, False)])
def test_native_equals_the_python_driver(onb, evaluator, reuse):
    import torch
    n, sims, games = 40, 12, 100
    with onb.Context(n, seed=17, mcts_max_sims=sims) as ctx:
        if evaluator == 2:
            _net_ctx(onb, ctx)
        v = _threshold(onb, ctx, sims, games, evaluator)
        proto = dict(temp_plies=8, temperature=1.0, resign=True, resign_below=v, resign_holdout=0.25, seed=23)
        for train in (False, True):
            nat = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=evaluator, train=train, noise_seed=5, reuse=reuse, protocol=proto)
            ctx.set_selfplay_protocol(None)
            py = onb.self_play_continuous(ctx, 2.0, sims, games, max_plies=30, evaluator=evaluator, train=train, noise_seed=5, reuse=reuse,
                                          protocol=proto)
            assert ctx.selfplay_protocol is None   # the driver does not use or change the context's setting
            _same_run(nat, py)
            assert nat["games"] == games and nat["resigned"] == py["resigned"] > 0
            for k in ("serial", "result", "min_m"):
                assert torch.equal(nat["held_out"][k], py["held_out"][k]), k
            assert nat["held_out"]["result"].shape[0] > 0
            # every held-out record's minima are the minima of its game's m over each side's searches
            for i, s in enumerate(py["held_out"]["serial"].tolist()):
                sel = py["serial"] == s
                for side in (0, 1):
                    ms = py["m"][sel & (py["color"] == side)]
                    want = float(ms.min()) if ms.numel() else float("inf")
                    assert float(nat["held_out"]["min_m"][i, side]) == want


@pytest.mark.gpu
def test_resignation_semantics(onb):
    import torch
    n, sims, games = 64, 16, 128
    with onb.Context(n, seed=8, mcts_max_sims=sims) as ctx:
        off = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=1, protocol=False)
        # v_resign above every m, nothing held out: every game resigns at its first search
        r = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=1, protocol=dict(resign=True, resign_below=1.01, resign_holdout=0.0))
        assert r["resigned"] == r["games"] == games and r["z"].shape[0] == games and bool((r["z"] == -1).all())
        assert r["serial"].unique().numel() == games and r["held_out"]["result"].shape[0] == 0
        # every game held out: none resigns, the samples are those of the protocol off, and each game has a record
        h = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=1, protocol=dict(resign=True, resign_below=1.01, resign_holdout=1.0))
        _same_run(h, off)
        assert h["resigned"] == 0 and h["held_out"]["result"].shape[0] == games
        ser = h["held_out"]["serial"]
        assert ser.unique().numel() == games and set(ser.tolist()) == set(off["serial"].tolist())
        # v_resign = -1: m >= -1 and the test is strict, so the run is the protocol off
        lo = ctx.self_play_native(2.0, sims, games, max_plies=30, evaluator=1, protocol=dict(resign=True, resign_below=-1.0, resign_holdout=0.1))
        _same_run(lo, off)
        assert lo["resigned"] == 0 and 0 < lo["held_out"]["result"].shape[0] < games
        # results of the records: the final z of the game's samples (Red's view)
        for s, res in zip(h["held_out"]["serial"].tolist(), h["held_out"]["result"].tolist()):
            sel = (off["serial"] == s) & (off["color"] == 0)
            if sel.any():
                z = float(off["z"][sel][0])
                assert res == (0 if z == 0 else (1 if z > 0 else 2))


@pytest.mark.gpu
def test_temperature_varies_the_games_and_only_in_the_opening(onb):
    import torch
    n, sims, games = 48, 16, 96
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx:
        off = ctx.self_play_native(2.0, sims, games, max_plies=40, evaluator=1, protocol=False)
        zero = ctx.self_play_native(2.0, sims, games, max_plies=40, evaluator=1, protocol=dict(temp_plies=0, temperature=1.0, seed=5))
        _same_run(zero, off)
        a = ctx.self_play_native(2.0, sims, games, max_plies=40, evaluator=1, protocol=dict(temp_plies=30, seed=5))
        b = ctx.self_play_native(2.0, sims, games, max_plies=40, evaluator=1, protocol=dict(temp_plies=30, seed=6))
        assert a["planes"].shape != b["planes"].shape or not torch.equal(a["planes"], b["planes"])   # two seeds, two sets of games
        assert a["planes"].shape != off["planes"].shape or not torch.equal(a["planes"], off["planes"])
    # the loop's rule applied from Python: a game plays a move other than best only at plies p < T
    n, t_plies = 256, 4
    with onb.Context(n, seed=4, mcts_max_sims=sims) as ctx:
        ctx.reset()
        plies = np.zeros(n, np.int64)
        differ_early = 0
        for tick in range(12):
            live = ctx.get_states()["result"] == 0
            ctx.search_device(2.0, sims, evaluator=1)
            best = ctx.read(onb.BUF_BEST, np.uint16, (n,)).copy()
            mask = (live & (plies < t_plies)).astype(np.uint8)
            ctx.mcts_choose(9, tick, 1.0, mask)
            acts = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)).copy()
            assert (acts[mask == 0] == best[mask == 0]).all()
            differ_early += int((acts[mask == 1] != best[mask == 1]).sum())
            acts[~live] = onb.ACTION_NONE
            ctx.step(acts)
            plies += live
        assert differ_early > 0


@pytest.mark.gpu
@pytest.mark.parametrize("t_plies", [1, 3])
def test_native_loop_samples_only_before_ply_t(onb, t_plies):
    # onb_self_play's own gate (plies < temp_plies): eval mode, one game per slot dealt alike in every run, so two runs whose game
    # reaches the same position at ply T must play the rest alike (every later move is the search's best), while the same position
    # at ply T - 1 may still lead to different positions at ply T (the move of ply T - 1 is sampled)
    n, sims, seeds = 512, 16, 4
    runs = []
    with onb.Context(n, seed=6, mcts_max_sims=sims) as ctx:
        for seed in range(seeds):
            r = ctx.self_play_native(2.0, sims, n, max_plies=60, evaluator=1, protocol=dict(temp_plies=t_plies, seed=seed))
            ser, pl = r["serial"].cpu().numpy(), r["planes"].cpu().numpy()
            runs.append([pl[ser == s] for s in range(n)])   # a game's samples in ply order
    # The planes show the pieces and the side to move's hand only. Equal planes up to ply p and equal hand planes (4 .. 19) at ply p + 1
    # (the hand the side that moved at ply p - 1 kept: it reveals the card played there and does not depend on ply p's move) mean the
    # same state at ply p, card slots included, since every game of a slot starts from the same deal.
    def same_state(x, y, p):
        return len(x) > p + 1 and len(y) > p + 1 and np.array_equal(x[:p + 1], y[:p + 1]) and np.array_equal(x[p + 1, 4:20], y[p + 1, 4:20])
    t = t_plies
    same_after = diverge_at_t = 0
    for a in range(seeds):
        for b in range(a + 1, seeds):
            for s in range(n):
                x, y = runs[a][s], runs[b][s]
                if same_state(x, y, t):
                    assert x.shape == y.shape and np.array_equal(x, y), (t, s)
                    same_after += 1
                elif same_state(x, y, t - 1) and not np.array_equal(x[t, :4], y[t, :4]):
                    diverge_at_t += 1
    assert same_after > 0 and diverge_at_t > 0, (same_after, diverge_at_t)


@pytest.mark.gpu
def test_tau_one_frequencies_on_fixed_trees(onb):
    import torch
    from scipy import stats
    n, sims, steps = 64, 200, 2000
    roots = _roots(n, 31)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.mcts_begin(2.0, sims)
        ctx.mcts_run(1, sims)
        ctx.mcts_finish()
        trees = _tree_roots(ctx, n)
        mask = np.ones(n, np.uint8)
        acts = []
        with torch.cuda.stream(ctx.torch_stream()):
            a_t = ctx.tensor(onb.BUF_ACTIONS)
            for step in range(steps):
                ctx.mcts_choose(13, step, 1.0, mask)
                acts.append(a_t.clone())
            acts = torch.stack(acts).cpu().numpy().astype(np.int64) & 0xFFFF
    bad = 0
    for g in range(0, n, 8):
        _, _, vis, _, act, _ = trees[g]
        counts = np.array([(acts[:, g] == a).sum() for a in act])
        assert counts.sum() == steps and counts[vis == 0].sum() == 0
        exp = vis / vis.sum() * steps
        keep = exp >= 5
        obs, e = list(counts[keep]), list(exp[keep])
        if (~keep).any():
            obs.append(counts[~keep].sum()); e.append(exp[~keep].sum())
        bad += stats.chisquare(obs, np.array(e) * sum(obs) / sum(e)).pvalue < 1e-3
    assert bad <= 1


@pytest.mark.gpu
def test_refusals(onb):
    n = 16
    with onb.Context(n, mcts_max_sims=8) as ctx:
        for bad in (dict(temp_plies=3, temperature=0.0), dict(temp_plies=3, temperature=-1.0), dict(temp_plies=3, temperature=float("inf")),
                    dict(temp_plies=3, temperature=float("nan")), dict(resign=True, resign_below=float("nan")),
                    dict(resign=True, resign_below=float("inf")), dict(resign=True, resign_holdout=1.5), dict(resign=True, resign_holdout=-0.1)):
            with pytest.raises(onb.OnbError) as e:
                ctx.set_selfplay_protocol(bad)
            assert e.value.code == -1, bad
        with pytest.raises(onb.OnbError) as e:   # before any self-play run
            ctx.selfplay_protocol_stats()
        assert e.value.code == -4
        with pytest.raises(onb.OnbError) as e:   # no finished search
            ctx.mcts_choose(0, 0, 1.0)
        assert e.value.code == -4
        ctx.reset()
        ctx.search_device(2.0, 8)
        for tau in (0.0, -2.0, float("inf")):
            with pytest.raises(onb.OnbError) as e:
                ctx.mcts_choose(0, 0, tau)
            assert e.value.code == -1
        ctx.set_selfplay_protocol(dict(temp_plies=4, seed=1))
        with pytest.raises(onb.OnbError) as e:   # Gumbel plays its sequential-halving winner
            ctx.self_play_native(2.0, 8, 16, max_plies=10, gumbel=dict(m=4))
        assert e.value.code == -4
        # resignation combines with Gumbel
        ctx.set_selfplay_protocol(dict(resign=True, resign_below=-0.5, resign_holdout=0.5, seed=1))
        r = ctx.self_play_native(2.0, 8, 16, max_plies=10, gumbel=dict(m=4))
        assert r["games"] == 16
        ctx.set_gumbel(False)


@pytest.mark.gpu
def test_mirror_equals_the_context(onb, tmp_path):
    exe = str(tmp_path / "test_selfplay_protocol_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "cpp", "test_selfplay_protocol_mirror.cpp"), "-o", exe,
                           "-L" + os.path.join(ROOT, "onitama_alphazero_b200"), "-lonb", "-Wl,-rpath," + os.path.join(ROOT, "onitama_alphazero_b200")])
    slots, games, sims, t_plies, tau, v, h, seed = 32, 64, 16, 8, 1.0, -0.2, 0.25, 3
    p = subprocess.run([exe], input="%d %d %d %d %r %r %r %d\n" % (slots, games, sims, t_plies, tau, v, h, seed), capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    lines = p.stdout.split("\n")
    m = int(lines[0])
    got = np.array([[float(x) for x in ln.split()] for ln in lines[1:1 + m]]).reshape(-1, 2)
    with onb.Context(slots, seed=seed, mcts_max_sims=sims) as ctx:
        r = ctx.self_play_native(2.0, sims, games, max_plies=150, evaluator=0,
                                 protocol=dict(temp_plies=t_plies, temperature=tau, resign=True, resign_below=v, resign_holdout=h, seed=seed))
    assert m == r["z"].shape[0]
    assert np.array_equal(got[:, 0], r["z"].cpu().numpy()) and np.array_equal(got[:, 1], r["color"].cpu().numpy())


@pytest.mark.gpu
def test_example_runs_with_temperature_and_resignation(onb):
    import importlib.util
    spec = importlib.util.spec_from_file_location("selfplay_train_loop", os.path.join(ROOT, "examples", "selfplay_train_loop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for extra in ([], ["--torch-net"]):
        log = mod.main(["--slots", "48", "--games", "96", "--sims", "16", "--iters", "2", "--max-plies", "40", "--batch", "64", "--sgd-steps", "3",
                        "--eval-games", "16", "--mcts-playouts", "60", "--temp-plies", "30", "--resign-fp", "0.05"] + extra)
        assert len(log) == 2 and all(x["games"] == 96 and x["samples"] > 0 for x in log)
        assert log[0]["resigned"] == 0 and log[0]["held_out"] == 96          # the first iteration holds out every game
        assert log[1]["held_out"] < 96 and np.isfinite(log[1]["policy_loss"])
