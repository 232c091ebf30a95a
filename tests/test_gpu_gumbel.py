"""The Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f) on the GPU against the CPU restatement (tests/gumbel_oracle.cpp): child
visits, actions, pi' bits and node counts on 4 096 roots, whole trees on a sample, continued plies with the fused network; the split
phase, CUDA graphs, batch / subset / shard invariance, native self-play and the arena against their Python drivers, the switch and
the refusals."""
import numpy as np
import pytest

import gumbel_oracle as GO
import oracle_lib as O

KEYS = ("visits", "reward", "prior", "action", "parent", "first_child", "n_child", "flags")


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def _undecided(n, seed, plies=12):
    g = O.new_games(2 * n, seed=seed)
    for step in range(plies):
        live = (np.arange(2 * n) % plies) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return np.ascontiguousarray(g[g["result"] == 0][:n])


def _same(got, want, keys=("best", "pi", "root_visits", "child_visits")):
    for k in keys:
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pi"].view(np.uint32), want["pi"].view(np.uint32))


CASES = [(16, 1), (16, 2), (16, 17), (4, 50), (16, 200), (40, 400)]


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.0, 1.0])
@pytest.mark.parametrize("m,sims", CASES)
@pytest.mark.parametrize("evaluator", [0, 1])
def test_equals_the_oracle(onb, evaluator, m, sims, scale):
    n, c, seed, step = 4096, 2.0, 17, 5
    roots = _undecided(n, 40 + sims + evaluator)
    assert len(roots) == n
    want = GO.search(roots, c, sims, evaluator=evaluator, m=m, gumbel_scale=scale, seed=seed, step=step)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=m, gumbel_scale=scale, seed=seed, step0=step)
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(evaluator, sims)
        got = ctx.mcts_finish()
        _same(got, want)
        assert np.array_equal(got["root_q"], want["root_q"])
        nn, _ = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"])
        for t in range(0, n, 997):
            tree = GO.search(roots[t:t + 1], c, sims, evaluator=evaluator, m=m, gumbel_scale=scale, seed=seed, step=step, game0=t, dump_tree=0)["tree"]
            mine = ctx.mcts_dump_tree(t)
            for k in KEYS:
                assert np.array_equal(mine[k], tree[k].astype(mine[k].dtype)), (t, k)


@pytest.mark.gpu
def test_three_plies_with_the_fused_network(onb):
    from test_net_cpu import lively_model
    model = lively_model(3, seed=21)
    n, sims, c, seed = 8, 48, 2.0, 4
    states = _undecided(n, 77)
    with onb.Context(1, mcts_max_sims=2, planes=False) as one, onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        one.net_load(model)
        ctx.net_load(model)

        def eval_one(planes525):
            one.write(onb.BUF_LEAF_PLANES, np.asarray(planes525, dtype=np.float32).reshape(1, 525))
            one.net_forward(onb.BUF_LEAF_PLANES)
            return one.read(onb.BUF_POLICY, np.float32, (50,)), float(one.read(onb.BUF_VALUE, np.float32, (1,))[0])

        ctx.set_gumbel(True, m=16, seed=seed)
        ctx.set_states(states)
        for ply in range(3):
            live = states["result"] == 0
            want = GO.search(states, c, sims, m=16, seed=seed, step=ply, callback=eval_one)
            ctx.mcts_begin(c, sims)
            ctx.mcts_run(onb.EVAL_NET, sims)
            got = ctx.mcts_finish()
            for k in ("best", "pi", "child_visits"):
                assert np.array_equal(got[k][live], want[k][live]), (ply, k)
            ctx.mcts_play_best()
            for i in np.nonzero(live)[0]:
                O.make_move(states[i:i + 1], int(want["best"][i]))


@pytest.mark.gpu
def test_split_phase_and_graphs_equal_the_fused_search(onb):
    import torch
    from onitama_alphazero_b200.net import ConvResNet, make_evaluator
    n, sims, c = 256, 24, 2.0
    roots = _undecided(n, 9)
    with onb.Context(n, seed=1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=8, seed=3, step0=2)
        fused = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(True, m=8, seed=3, step0=2)
        split = ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=False)
        _same(split, fused)
        torch.manual_seed(7)
        net = make_evaluator(ConvResNet(64, 21, 3).cuda())
        res = {}
        for graph in (False, True):
            ctx.set_gumbel(True, m=8, seed=3, step0=0)
            res[graph] = []
            for _ in range(2):  # consecutive searches take steps 0 and 1: a replayed graph must read the new step
                ctx.search_device(c, sims, net=net, use_graph=graph)
                res[graph].append(ctx.mcts_finish())
        for a, b in zip(res[False], res[True]):
            _same(b, a)
        assert not np.array_equal(res[False][0]["pi"], res[False][1]["pi"])


@pytest.mark.gpu
def test_batch_subset_and_shard_invariance(onb):
    n, sims, c = 600, 40, 2.0
    roots = _undecided(n, 13)
    with onb.Context(n, seed=1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=16, seed=8, step0=3)
        full = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
    for first, count in ((0, 1), (123, 200), (599, 1)):
        with onb.Context(count, seed=1, game_id_base=first, mcts_max_sims=sims, planes=False) as ctx:
            ctx.set_states(roots[first:first + count])
            ctx.set_gumbel(True, m=16, seed=8, step0=3)
            part = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
            for k in ("best", "pi", "child_visits"):
                assert np.array_equal(part[k], full[k][first:first + count]), (first, k)


@pytest.mark.gpu
def test_native_self_play_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import self_play_continuous
    n, sims, c = 64, 16, 2.0
    cfg = dict(m=8, seed=6)
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx:
        nat = ctx.self_play_native(c, sims, 96, max_plies=30, evaluator=onb.EVAL_HASH, gumbel=cfg)
        ctx.set_gumbel(False)
        py = self_play_continuous(ctx, c, sims, 96, max_plies=30, evaluator=onb.EVAL_HASH, gumbel=cfg)
        assert getattr(ctx, "gumbel", None) is None  # the driver leaves the switch as it was
    assert nat["games"] == py["games"] >= 96
    for k in ("planes", "pi", "z", "color", "serial"):
        assert bool((nat[k] == py[k]).all()), k
    # pi is the improved policy, not the visit shares: with 16 simulations over up to 40 children it is never a multiple of 1/15
    assert not bool(((nat["pi"] * 15).round() == nat["pi"] * 15).all())


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import fight
    n, sims, max_plies = 128, 24, 40
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=11, mcts_max_sims=sims) as ctx:
        ctx.set_gumbel(True, m=4, seed=99, step0=7)
        ctx.reset()
        nat = ctx.fight_native(ctx.agent_gumbel(sims, m=8, c_scale=0.1, evaluator=onb.EVAL_HASH), ctx.agent_puct(sims, 2.0, onb.EVAL_HASH), a_is_red,
                               max_plies)
        # onb_fight left the context's setting (and its step) as it found it
        ctx.reset()
        after = ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(True, m=4, seed=99, step0=7)
        ctx.reset()
        _same(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH), after)
        ply = [0]

        def gumbel_move(x):
            x.set_gumbel(True, m=8, c_scale=0.1, seed=x.seed, step0=ply[0])
            x.search_device(2.0, sims, evaluator=onb.EVAL_HASH)  # PUCT below the root with the agents' c_puct 2
            x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))

        def puct_move(x):
            x.set_gumbel(False)
            x.search_device(2.0, sims, evaluator=onb.EVAL_HASH)
            x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))
            ply[0] += 1

        ctx.reset()
        py = fight(ctx, gumbel_move, puct_move, a_is_red, max_plies)
    assert nat[:3] == tuple(py[:3])


@pytest.mark.gpu
def test_switching_off_restores_puct_and_the_gumbel_refusals(onb):
    n, sims, c = 128, 32, 2.0
    roots = _undecided(n, 3)
    # ctx has room for more simulations than a search asks for, so that running past the begin's sims meets the Gumbel check
    with onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=True) as ctx, onb.Context(n, seed=1, mcts_max_sims=sims, planes=True) as ref:
        for x in (ctx, ref):
            x.set_states(roots)
        ctx.set_gumbel(True)
        ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(False)
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH), ref.search(c, sims, evaluator=onb.EVAL_HASH), keys=("best", "pi", "root_q", "child_visits"))

        def code(fn, *a, **kw):
            with pytest.raises(onb.OnbError) as e:
                fn(*a, **kw)
            return e.value.code

        for bad in (dict(m=0), dict(m=41), dict(c_visit=-1.0), dict(c_scale=float("nan")), dict(gumbel_scale=float("inf"))):
            assert code(ctx.set_gumbel, True, **bad) == onb._lib.E_INVALID
        ctx.set_gumbel(True)
        ctx.set_reuse(True)
        assert code(ctx.mcts_begin, c, sims) == onb._lib.E_STATE
        ctx.set_reuse(False)
        ctx.mcts_set_noise(True)
        assert code(ctx.mcts_begin, c, sims) == onb._lib.E_STATE
        assert code(ctx.self_play_native, c, sims, 4, 10, onb.EVAL_HASH, True) == onb._lib.E_INVALID
        ctx.mcts_set_noise(False)
        ctx.mcts_begin(c, sims)
        assert code(lambda: ctx._ck(ctx._lib.onb_uct_run(ctx._h, 1.4, 5, sims))) == onb._lib.E_STATE
        ctx.mcts_run(onb.EVAL_HASH, sims)
        assert code(ctx.mcts_run, onb.EVAL_HASH, 1) == onb._lib.E_STATE
        assert code(ctx.mcts_select) == onb._lib.E_STATE


@pytest.mark.gpu
def test_subset_searches_equal_the_full_batch(onb):
    """onb_fight searches each agent's games as a list (non-contiguous subsets of the context's trees); two identical Gumbel agents
    over two plies must play what one full-batch search per ply plays"""
    n, sims = 300, 24
    roots = _undecided(n, 23)
    a_is_red = np.random.default_rng(4).random(n) < 0.5
    ag = onb.Context.agent_gumbel(sims, m=8, c_scale=0.2, evaluator=onb.EVAL_HASH)
    with onb.Context(n, seed=31, mcts_max_sims=sims, planes=False) as ctx, onb.Context(n, seed=31, mcts_max_sims=sims, planes=False) as ref:
        ctx.set_states(roots)
        ctx.fight_native(ag, ag, a_is_red, max_plies=0)  # two plies
        assert ctx.last_fight_plies == 2
        ref.set_states(roots)
        ref.set_gumbel(True, m=8, c_scale=0.2, seed=31, step0=0)
        for _ in range(2):
            ref.search_device(2.0, sims, evaluator=onb.EVAL_HASH)
            ref.mcts_play_best()
        assert np.array_equal(ctx.get_states(), ref.get_states())


@pytest.mark.gpu
def test_a_search_begun_with_the_switch_off_is_puct_everywhere(onb):
    """after a Gumbel search and the switch turned off, native self-play with tree reuse is the plain reuse self-play"""
    n, sims, c = 64, 16, 2.0
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx, onb.Context(n, seed=2, mcts_max_sims=sims) as ref:
        ctx.reset()
        ctx.set_gumbel(True, m=8, seed=6)
        ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(False)
        got = ctx.self_play_native(c, sims, 80, max_plies=30, evaluator=onb.EVAL_HASH, reuse=True)
        want = ref.self_play_native(c, sims, 80, max_plies=30, evaluator=onb.EVAL_HASH, reuse=True)
    assert got["games"] == want["games"]
    for k in ("planes", "pi", "z", "color", "serial"):
        assert bool((got[k] == want[k]).all()), k


@pytest.mark.gpu
def test_reuse_switch_with_gumbel(onb):
    """native self-play refuses Gumbel with tree reuse (as onb_mcts_begin and the Python driver do); onb_fight, which never reuses
    trees, plays its Gumbel agents whatever the switch says"""
    n, sims = 64, 16
    a_is_red = np.arange(n) % 2 == 0
    with onb.Context(n, seed=5, mcts_max_sims=sims) as ctx, onb.Context(n, seed=5, mcts_max_sims=sims) as ref:
        ctx.set_gumbel(True, m=8, seed=6)
        ctx.set_reuse(True)
        with pytest.raises(onb.OnbError) as e:
            ctx.self_play_native(2.0, sims, 8, max_plies=10, evaluator=onb.EVAL_HASH)
        assert e.value.code == onb._lib.E_STATE
        from onitama_alphazero_b200.selfplay import self_play_continuous
        with pytest.raises(onb.OnbError) as e:
            self_play_continuous(ctx, 2.0, sims, 8, max_plies=10, evaluator=onb.EVAL_HASH, reuse=True, gumbel=dict(m=8, seed=6))
        assert e.value.code == onb._lib.E_STATE
        for x in (ctx, ref):
            x.reset()
        agents = (onb.Context.agent_gumbel(sims, m=8, evaluator=onb.EVAL_HASH), onb.Context.agent_puct(sims, 2.0, onb.EVAL_HASH))
        got = ctx.fight_native(*agents, a_is_red, max_plies=30)
        want = ref.fight_native(*agents, a_is_red, max_plies=30)
        assert np.array_equal(got[3], want[3]) and got[:3] == want[:3]


@pytest.mark.gpu
def test_python_driver_keeps_the_step(onb):
    n, sims, c = 32, 8, 2.0
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx:
        ctx.set_gumbel(True, m=3, seed=1, step0=5)
        from onitama_alphazero_b200.selfplay import self_play_continuous
        self_play_continuous(ctx, c, sims, 8, max_plies=10, evaluator=onb.EVAL_HASH, gumbel=dict(m=8, seed=6))
        assert ctx.gumbel == (3, 50.0, 0.1, 1.0, 1) and ctx.gumbel_step == 5
        ctx.reset()
        after = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(True, m=3, seed=1, step0=5)
        ctx.reset()
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH), after)


@pytest.mark.gpu
def test_cpp_mirror_moves_equal_the_context(onb, tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_gumbel_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_gumbel_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    start = _undecided(1, 51)
    plies, sims, m, seed = 8, 100, 8, 12
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d %d %d\n%s\n" % (plies, sims, m, seed, line), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = [int(x) for x in p.stdout.split()[:-2]]
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_gumbel(True, m=m, seed=seed)
        ctx.set_states(start)
        for _ in range(len(got)):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)["best"][0]))
            ctx.mcts_play_best()
    assert got == want and len(got) >= 2


@pytest.mark.gpu
def test_example_trains_on_the_gumbel_policy(onb):
    """examples/selfplay_train_loop.py --gumbel M: Gumbel self-play, training on pi', and the Gumbel-against-PUCT arena (native and
    Python-driven)"""
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("selfplay_train_loop", os.path.join(root, "examples", "selfplay_train_loop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for extra in ([], ["--torch-net"]):
        log = mod.main(["--slots", "48", "--games", "64", "--sims", "16", "--iters", "1", "--max-plies", "12", "--batch", "64", "--sgd-steps", "3",
                        "--eval-games", "16", "--mcts-playouts", "60", "--gumbel", "8"] + extra)
        assert len(log) == 1 and log[0]["games"] == 64 and log[0]["samples"] > 0
        assert sum(log[0]["gumbel_vs_puct"][k] for k in ("wins", "losses", "draws")) == 16
        assert np.isfinite(log[0]["policy_loss"])
