"""Gumbel MuZero's interior selection (onb_gumbel_config.interior, DESIGN.md §5f) on the GPU against the CPU restatement
(tests/gumbel_oracle.cpp with interior selection): child visits, actions, pi' bits and node counts on 4 096 roots, whole trees on a sample,
continued plies with the fused network (the split kernels); the split phase, CUDA graphs, batch / subset / shard invariance, native
self-play and the arena against their Python drivers, the C++ mirror, the example, the switch and the refusals, and a strength check."""
import numpy as np
import pytest

import gumbel_interior_oracle as GIO
from test_gpu_gumbel import CASES, KEYS, _same, _undecided


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [0.0, 1.0])
@pytest.mark.parametrize("m,sims", CASES)
@pytest.mark.parametrize("evaluator", [0, 1])
def test_equals_the_oracle(onb, evaluator, m, sims, scale):
    n, c, seed, step = 4096, 2.0, 17, 5
    roots = _undecided(n, 40 + sims + evaluator)
    assert len(roots) == n
    want = GIO.search(roots, c, sims, evaluator=evaluator, m=m, gumbel_scale=scale, seed=seed, step=step)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=m, gumbel_scale=scale, seed=seed, step0=step, interior=True)
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(evaluator, sims)
        got = ctx.mcts_finish()
        _same(got, want)
        assert np.array_equal(got["root_q"], want["root_q"])
        nn, _ = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"])
        for t in range(0, n, 997):
            tree = GIO.search(roots[t:t + 1], c, sims, evaluator=evaluator, m=m, gumbel_scale=scale, seed=seed, step=step, game0=t, dump_tree=0)["tree"]
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

        ctx.set_gumbel(True, m=16, seed=seed, interior=True)
        ctx.set_states(states)
        for ply in range(3):
            live = states["result"] == 0
            want = GIO.search(states, c, sims, m=16, seed=seed, step=ply, callback=eval_one)
            ctx.mcts_begin(c, sims)
            ctx.mcts_run(onb.EVAL_NET, sims)
            got = ctx.mcts_finish()
            for k in ("best", "pi", "child_visits"):
                assert np.array_equal(got[k][live], want[k][live]), (ply, k)
            ctx.mcts_play_best()
            import oracle_lib as O
            for i in np.nonzero(live)[0]:
                O.make_move(states[i:i + 1], int(want["best"][i]))


@pytest.mark.gpu
def test_split_phase_and_graphs_equal_the_fused_search(onb):
    from onitama_alphazero_b200.net import ConvResNet, make_evaluator
    import torch
    n, sims, c = 256, 24, 2.0
    roots = _undecided(n, 9)
    with onb.Context(n, seed=1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=8, seed=3, step0=2, interior=True)
        fused = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        ctx.set_gumbel(True, m=8, seed=3, step0=2, interior=True)
        split = ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=False)
        _same(split, fused)
        ctx.set_gumbel(True, m=8, seed=3, step0=2)
        assert not np.array_equal(ctx.search(c, sims, evaluator=onb.EVAL_HASH)["child_visits"], fused["child_visits"])
        torch.manual_seed(7)
        net = make_evaluator(ConvResNet(64, 21, 3).cuda())
        res = {}
        for graph in (False, True):
            ctx.set_gumbel(True, m=8, seed=3, step0=0, interior=True)
            res[graph] = []
            for _ in range(2):
                ctx.search_device(c, sims, net=net, use_graph=graph)
                res[graph].append(ctx.mcts_finish())
        for a, b in zip(res[False], res[True]):
            _same(b, a)
        # a graph captured for the interior setting is not replayed for the root-only one (the graph key holds the setting)
        ctx.set_gumbel(True, m=8, seed=3, step0=0)
        ctx.search_device(c, sims, net=net, use_graph=True)
        root_only = ctx.mcts_finish()
        ctx.set_gumbel(True, m=8, seed=3, step0=0)
        ctx.search_device(c, sims, net=net, use_graph=False)
        _same(ctx.mcts_finish(), root_only)


@pytest.mark.gpu
def test_batch_subset_and_shard_invariance(onb):
    n, sims, c = 600, 40, 2.0
    roots = _undecided(n, 13)
    with onb.Context(n, seed=1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.set_gumbel(True, m=16, seed=8, step0=3, interior=True)
        full = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
    for first, count in ((0, 1), (123, 200), (599, 1)):
        with onb.Context(count, seed=1, game_id_base=first, mcts_max_sims=sims, planes=False) as ctx:
            ctx.set_states(roots[first:first + count])
            ctx.set_gumbel(True, m=16, seed=8, step0=3, interior=True)
            part = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
            for k in ("best", "pi", "child_visits"):
                assert np.array_equal(part[k], full[k][first:first + count]), (first, k)
    # two identical Gumbel MuZero agents over two plies search the games as lists: equal to one full-batch search per ply
    a_is_red = np.random.default_rng(4).random(n) < 0.5
    ag = onb.Context.agent_gumbel(24, m=8, c_scale=0.2, evaluator=onb.EVAL_HASH, interior=True)
    with onb.Context(n, seed=31, mcts_max_sims=24, planes=False) as ctx, onb.Context(n, seed=31, mcts_max_sims=24, planes=False) as ref:
        ctx.set_states(roots)
        ctx.fight_native(ag, ag, a_is_red, max_plies=0)
        ref.set_states(roots)
        ref.set_gumbel(True, m=8, c_scale=0.2, seed=31, step0=0, interior=True)
        for _ in range(2):
            ref.search_device(2.0, 24, evaluator=onb.EVAL_HASH)
            ref.mcts_play_best()
        assert np.array_equal(ctx.get_states(), ref.get_states())


@pytest.mark.gpu
def test_native_self_play_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import self_play_continuous
    n, sims, c = 64, 16, 2.0
    cfg = dict(m=8, seed=6, interior=True)
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx:
        nat = ctx.self_play_native(c, sims, 96, max_plies=30, evaluator=onb.EVAL_HASH, gumbel=cfg)
        assert ctx.gumbel == (8, 50.0, 0.1, 1.0, 6, True)
        ctx.set_gumbel(False)
        py = self_play_continuous(ctx, c, sims, 96, max_plies=30, evaluator=onb.EVAL_HASH, gumbel=cfg)
        assert getattr(ctx, "gumbel", None) is None
        root_only = ctx.self_play_native(c, sims, 96, max_plies=30, evaluator=onb.EVAL_HASH, gumbel=dict(m=8, seed=6))
    assert nat["games"] == py["games"] >= 96
    for k in ("planes", "pi", "z", "color", "serial"):
        assert bool((nat[k] == py[k]).all()), k
    assert nat["pi"].shape != root_only["pi"].shape or not bool((nat["pi"] == root_only["pi"]).all())


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import fight
    n, sims, max_plies = 128, 24, 40
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=11, mcts_max_sims=sims) as ctx:
        ctx.set_gumbel(True, m=4, seed=99, step0=7)
        ctx.reset()
        nat = ctx.fight_native(ctx.agent_gumbel(sims, m=8, c_scale=0.1, evaluator=onb.EVAL_HASH, interior=True),
                               ctx.agent_gumbel(sims, m=8, c_scale=0.1, evaluator=onb.EVAL_HASH), a_is_red, max_plies)
        ctx.reset()
        after = ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)  # onb_fight left the context's setting and step as it found them
        ctx.set_gumbel(True, m=4, seed=99, step0=7)
        ctx.reset()
        _same(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH), after)
        ply = [0]

        def move(interior):
            def f(x):
                x.set_gumbel(True, m=8, c_scale=0.1, seed=x.seed, step0=ply[0], interior=interior)
                x.search_device(2.0, sims, evaluator=onb.EVAL_HASH)
                x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))
                if not interior:
                    ply[0] += 1
            return f

        ctx.reset()
        py = fight(ctx, move(True), move(False), a_is_red, max_plies)
    assert nat[:3] == tuple(py[:3])


@pytest.mark.gpu
def test_root_only_agent_ignores_the_context_interior_setting(onb):
    n, sims = 96, 24
    a_is_red = (np.arange(n) % 2 == 0)
    ag = (onb.Context.agent_gumbel(sims, m=8, evaluator=onb.EVAL_HASH), onb.Context.agent_puct(sims, 2.0, onb.EVAL_HASH))
    res = []
    for interior in (None, False, True):
        with onb.Context(n, seed=3, mcts_max_sims=sims) as ctx:
            if interior is not None:
                ctx.set_gumbel(True, m=4, seed=1, interior=interior)
            ctx.reset()
            res.append(ctx.fight_native(*ag, a_is_red, 40))
            res[-1] = (res[-1][:3], ctx.get_states().tobytes())
    assert res[0] == res[1] == res[2]


@pytest.mark.gpu
def test_mirror_moves_equal_the_context(onb, tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_gumbel_interior_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"),
                           os.path.join(root, "tests", "cpp", "test_gumbel_interior_mirror.cpp"), "-o", exe,
                           "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb", "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    start = _undecided(1, 51)
    plies, sims, m, seed = 8, 100, 8, 12
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d %d %d\n%s\n" % (plies, sims, m, seed, line), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = [int(x) for x in p.stdout.split()[:-2]]
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_gumbel(True, m=m, seed=seed, interior=True)
        ctx.set_states(start)
        for _ in range(len(got)):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)["best"][0]))
            ctx.mcts_play_best()
    assert got == want and len(got) >= 2


@pytest.mark.gpu
def test_example_runs_with_gumbel_interior(onb):
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("selfplay_train_loop", os.path.join(root, "examples", "selfplay_train_loop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for extra in ([], ["--torch-net"]):
        log = mod.main(["--slots", "48", "--games", "64", "--sims", "16", "--iters", "1", "--max-plies", "12", "--batch", "64", "--sgd-steps", "3",
                        "--eval-games", "16", "--mcts-playouts", "60", "--gumbel", "8", "--gumbel-interior"] + extra)
        assert len(log) == 1 and log[0]["games"] == 64 and log[0]["samples"] > 0
        assert sum(log[0]["gumbel_vs_puct"][k] for k in ("wins", "losses", "draws")) == 16
        assert np.isfinite(log[0]["policy_loss"])


@pytest.mark.gpu
def test_the_switch_and_the_refusals(onb):
    n, sims, c = 128, 32, 2.0
    roots = _undecided(n, 3)
    with onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=True) as ctx, onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=True) as ref:
        for x in (ctx, ref):
            x.set_states(roots)
        ctx.set_gumbel(True, m=8, seed=2, interior=True)
        ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        for x in (ctx, ref):  # root-only Gumbel, then PUCT: as in a context that never enabled interior selection
            x.set_gumbel(True, m=8, seed=2, step0=4)
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH), ref.search(c, sims, evaluator=onb.EVAL_HASH), keys=("best", "pi", "root_q", "child_visits"))
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=False), ref.search(c, sims, evaluator=onb.EVAL_HASH, fused=False))
        for x in (ctx, ref):
            x.set_gumbel(False)
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH), ref.search(c, sims, evaluator=onb.EVAL_HASH), keys=("best", "pi", "root_q", "child_visits"))
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=False), ref.search(c, sims, evaluator=onb.EVAL_HASH, fused=False))

        def code(fn, *a, **kw):
            with pytest.raises(onb.OnbError) as e:
                fn(*a, **kw)
            return e.value.code

        import ctypes as C
        cfg = onb._lib.GumbelConfig(1, 16, 50.0, 0.1, 1.0, 0, 0, 2)
        assert code(lambda: ctx._ck(ctx._lib.onb_mcts_set_gumbel(ctx._h, C.byref(cfg)))) == onb._lib.E_INVALID
        ctx.set_gumbel(True, interior=True)
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
        bad = onb.Context.agent_gumbel(sims, m=41, interior=True)
        assert code(ctx.fight_native, bad, onb.Context.agent_random(), np.ones(n, bool), 4) == onb._lib.E_INVALID


@pytest.mark.gpu
def test_beats_the_random_agent(onb):
    n, sims = 256, 64
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=8, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()
        w, l, d, _ = ctx.fight_native(ctx.agent_gumbel(sims, m=16, evaluator=onb.EVAL_UNIFORM, interior=True), ctx.agent_random(), a_is_red, 150)
    assert w >= 0.8 * n, (w, l, d)
