"""Leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h) on the GPU against the CPU restatement
(tests/vl_oracle.cpp): actions, pi, visits, root Q, node counts and whole trees on 4 096 roots (roots with more than 32 children and
paths deeper than the register path included); onb_mcts_run against the split phase, torch networks with and without CUDA graphs
against ONB_EVAL_NET, the switch, the refusals, the arena agent against the Python driver, the C++ mirror and a strength check."""
import numpy as np
import pytest

import oracle_lib as O
import vl_oracle as VO
from test_gpu_gumbel import KEYS, _same, _undecided


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


_WIDE = []


def _roots(n, seed):
    """n undecided roots; the first ones have more than 32 children (found among 10^5 longer random games)"""
    if not _WIDE:
        for plies in (20, 30):
            r = _undecided(100000, 5, plies=plies)
            k = O.mcts_search_batch(r, 2.0, 1, evaluator=0, threads=8)["n_nodes"] - 1
            _WIDE.append(r[k > 32])
    wide = np.concatenate(_WIDE)
    assert len(wide) >= 8
    return np.ascontiguousarray(np.concatenate([wide, _undecided(n - len(wide), seed)]))


def _search(ctx, c, sims, evaluator, leaves, vl):
    ctx.set_virtual_loss(leaves, vl)
    ctx.mcts_begin(c, sims)
    ctx.mcts_run(evaluator, sims)
    return ctx.mcts_finish()


@pytest.mark.gpu
@pytest.mark.parametrize("sims", [1, 2, 33, 400])
@pytest.mark.parametrize("vl", [0.0, 1.0, 3.0])
@pytest.mark.parametrize("leaves", [2, 8, 32])
@pytest.mark.parametrize("evaluator", [0, 1])
def test_equals_the_oracle(onb, evaluator, leaves, vl, sims):
    n, c = 4096, 2.0
    roots = _roots(n, 40 + sims + evaluator)
    want = VO.search(roots, c, sims, leaves, vl, evaluator=evaluator)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        got = _search(ctx, c, sims, evaluator, leaves, vl)
        _same(got, want)
        assert np.array_equal(got["root_q"], want["root_q"])
        assert (got["root_visits"] == sims).all()
        nn, fl = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"]) and not (fl & 2).any()
        for t in list(range(0, n, 997)) + [0, 1]:
            tree = VO.search(roots[t:t + 1], c, sims, leaves, vl, evaluator=evaluator, dump_tree=0)["tree"]
            mine = ctx.mcts_dump_tree(t)
            for k in KEYS:
                assert np.array_equal(mine[k], tree[k].astype(mine[k].dtype)), (t, k)


@pytest.mark.gpu
@pytest.mark.parametrize("leaves,vl", [(2, 0.0), (8, 0.0), (8, 1.0)])
def test_paths_deeper_than_the_register_path(onb, leaves, vl):
    # c_puct = 0 and value 0: the descents follow one line to the game's end, far below kMaxDepth = 32 levels
    n, c, sims = 256, 0.0, 400
    roots = _undecided(n, 3)
    want = VO.search(roots, c, sims, leaves, vl, evaluator=0)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        got = _search(ctx, c, sims, 0, leaves, vl)
        _same(got, want)
        nn, _ = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"])
        deep = 0
        for t in range(0, n, 16):
            tree = VO.search(roots[t:t + 1], c, sims, leaves, vl, evaluator=0, dump_tree=0)["tree"]
            mine = ctx.mcts_dump_tree(t)
            for k in KEYS:
                assert np.array_equal(mine[k], tree[k].astype(mine[k].dtype)), (t, k)
            d = np.zeros(len(tree["parent"]), int)
            for i in range(1, len(d)):
                d[i] = d[tree["parent"][i]] + 1
            deep += int(d.max() > 32)
        assert deep >= 4


def _split(ctx, onb, c, sims, evaluator):
    ctx.mcts_begin(c, sims)
    for _ in range(ctx.vl_rounds(sims)):
        ctx.mcts_select()
        ctx.mcts_eval(evaluator)
        ctx.mcts_expand_backup()
    out = ctx.mcts_finish()
    with pytest.raises(onb.OnbError) as e:  # the search has run its sims
        ctx.mcts_select()
    assert e.value.code == onb._lib.E_STATE
    return out


@pytest.mark.gpu
def test_run_equals_the_split_phase(onb):
    from test_net_cpu import lively_model
    n, sims, c, leaves = 300, 61, 2.0, 8
    roots = _roots(n, 9)
    with onb.Context(n, mcts_max_sims=2 * sims, planes=False) as ctx:  # room beyond sims: the refusal below is the search's own
        ctx.set_states(roots)
        ctx.set_virtual_loss(leaves, 1.0)
        for ev in (onb.EVAL_UNIFORM, onb.EVAL_HASH):
            fused = ctx.search(c, sims, evaluator=ev)
            _same(_split(ctx, onb, c, sims, ev), fused, keys=("best", "pi", "root_visits", "root_q", "child_visits"))
        ctx.net_load(lively_model(3, seed=5))
        net = ctx.search(c, sims, evaluator=onb.EVAL_NET)
        _same(_split(ctx, onb, c, sims, onb.EVAL_NET), net, keys=("best", "pi", "root_visits", "root_q", "child_visits"))
        assert (net["root_visits"] == sims).all()
        # two onb_mcts_run calls: each counts its rounds against its own end, as one onb_mcts_run per piece in the oracle's schedule
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(onb.EVAL_HASH, 20)
        ctx.mcts_run(onb.EVAL_HASH, sims - 20)
        assert (ctx.mcts_finish()["root_visits"] == sims).all()
        with pytest.raises(onb.OnbError) as e:
            ctx.mcts_run(onb.EVAL_HASH, 1)
        assert e.value.code == onb._lib.E_STATE


@pytest.mark.gpu
def test_torch_net_and_graphs_equal_eval_net(onb):
    from test_net_cpu import lively_model
    import torch
    n, sims, c, leaves = 64, 77, 2.0, 16
    roots = _roots(n, 19)
    model = lively_model(3, seed=8)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        # the library's own network on the K rows through a second context on the same stream: the torch callable sees the rows
        with onb.Context(n * leaves, stream=ctx.stream_handle(), mcts_max_sims=1, planes=True) as aux:  # (policy / value buffers)
            ctx.net_load(model)
            aux.net_load(model)
            ctx.set_states(roots)
            want = ctx.search(c, sims, evaluator=onb.EVAL_NET, vl=leaves)
            planes, pol, val = aux.tensor(onb.BUF_PLANES), aux.tensor(onb.BUF_POLICY), aux.tensor(onb.BUF_VALUE)

            def net(x):
                planes.copy_(x)
                aux.net_forward(onb.BUF_PLANES)
                return pol, val

            _same(ctx.search(c, sims, net=net), want, keys=("best", "pi", "root_visits", "root_q", "child_visits"))
            for graph in (False, True, True):  # the second graph search replays the cached capture
                ctx.search_device(c, sims, net=net, use_graph=graph)
                _same(ctx.mcts_finish(), want, keys=("best", "pi", "root_visits", "root_q", "child_visits"))
            torch.cuda.synchronize()


@pytest.mark.gpu
def test_switching_off_restores_today_and_the_refusals(onb):
    n, sims, c = 128, 40, 2.0
    roots = _roots(n, 3)
    with onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=True) as ctx, onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=True) as ref:
        for x in (ctx, ref):
            x.set_states(roots)

        def code(fn, *a, **kw):
            with pytest.raises(onb.OnbError) as e:
                fn(*a, **kw)
            return e.value.code

        assert code(ctx.buffer, onb.BUF_VL_PLANES) == onb._lib.E_STATE  # before the first enabling call
        assert code(ctx.set_virtual_loss, 33, 1.0) == onb._lib.E_INVALID
        assert code(ctx.set_virtual_loss, 4, -1.0) == onb._lib.E_INVALID
        assert code(ctx.set_virtual_loss, 4, float("inf")) == onb._lib.E_INVALID
        ctx.search(c, sims, evaluator=onb.EVAL_HASH, vl=8)
        _, nbytes = ctx.buffer(onb.BUF_VL_PLANES)
        assert nbytes == n * 8 * 2100
        # a select whose round is never backed up, then a begin: the next searches must not see its virtual counts
        ctx.mcts_begin(c, sims)
        ctx.mcts_select()
        ctx.set_virtual_loss(1)
        for fused in (True, False):
            _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused), ref.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused),
                  keys=("best", "pi", "root_q", "child_visits"))
        ctx.set_virtual_loss(8, 1.0)
        ctx.mcts_begin(c, sims)
        ctx.mcts_select()
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(onb.EVAL_HASH, sims)
        fresh = ctx.mcts_finish()
        with onb.Context(n, seed=1, mcts_max_sims=2 * sims, planes=False) as other:
            other.set_states(roots)
            _same(fresh, other.search(c, sims, evaluator=onb.EVAL_HASH, vl=8), keys=("best", "pi", "root_q", "child_visits"))
        # the refusals, each followed by a search that is unaffected
        ctx.set_reuse(True)
        assert code(ctx.mcts_begin, c, sims) == onb._lib.E_STATE
        ctx.set_reuse(False)
        ctx.mcts_set_noise(True)
        assert code(ctx.mcts_begin, c, sims) == onb._lib.E_STATE
        ctx.mcts_set_noise(False)
        ctx.set_gumbel(True, m=8)
        assert code(ctx.mcts_begin, c, sims) == onb._lib.E_STATE
        ctx.set_gumbel(False)
        assert code(ctx.self_play_native, c, sims, 4, 10, onb.EVAL_HASH) == onb._lib.E_STATE
        ctx.set_states(roots)
        ctx.mcts_begin(c, sims)
        assert code(lambda: ctx._ck(ctx._lib.onb_uct_run(ctx._h, 1.4, 5, sims))) == onb._lib.E_STATE
        ctx.mcts_run(onb.EVAL_HASH, sims)
        assert code(ctx.mcts_run, onb.EVAL_HASH, 1) == onb._lib.E_STATE
        _same(ctx.mcts_finish(), fresh, keys=("best", "pi", "root_q", "child_visits"))
        bad = onb.Context.agent_puct(sims, 2.0, onb.EVAL_HASH, leaves=33)
        assert code(ctx.fight_native, bad, onb.Context.agent_random(), np.ones(n, bool), 4) == onb._lib.E_INVALID
        # a larger K reallocates the rows
        ctx.set_virtual_loss(32, 1.0)
        assert ctx.buffer(onb.BUF_VL_VALUE)[1] == n * 32 * 4
        ctx.set_states(roots)
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH, vl=(8, 1.0)), fresh, keys=("best", "pi", "root_q", "child_visits"))
        ctx.set_virtual_loss(0)
        ctx.set_states(roots)
        ctx.self_play_native(c, 8, 4, 10, onb.EVAL_HASH)


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import fight
    n, sims, max_plies, leaves = 128, 24, 40, 4
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=11, mcts_max_sims=sims) as ctx:
        ctx.set_virtual_loss(2, 3.0)
        ctx.reset()
        nat = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_HASH, leaves=leaves), ctx.agent_puct(sims, 2.0, onb.EVAL_HASH), a_is_red, max_plies)
        assert ctx.vl == (2, 3.0)  # onb_fight left the switch as it found it
        ctx.reset()
        after = ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)
        ctx.reset()
        _same(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH, vl=(2, 3.0)), after)

        def move(k):
            def f(x):
                x.search_device(2.0, sims, evaluator=onb.EVAL_HASH, vl=k)
                x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))
            return f

        ctx.reset()
        py = fight(ctx, move(leaves), move(1), a_is_red, max_plies)
    assert nat[:3] == tuple(py[:3])
    # the agent searches only the games in which it is to move: one ply of two identical agents equals one full search per ply
    roots = _undecided(n, 13)
    ag = onb.Context.agent_puct(sims, 2.0, onb.EVAL_HASH, leaves=8)
    with onb.Context(n, seed=31, mcts_max_sims=sims, planes=False) as ctx, onb.Context(n, seed=31, mcts_max_sims=sims, planes=False) as ref:
        ctx.set_states(roots)
        ctx.fight_native(ag, ag, np.random.default_rng(4).random(n) < 0.5, max_plies=0)
        ref.set_states(roots)
        for _ in range(2):
            ref.search_device(2.0, sims, evaluator=onb.EVAL_HASH, vl=(8, 1.0))
            ref.mcts_play_best()
        assert np.array_equal(ctx.get_states(), ref.get_states())


@pytest.mark.gpu
def test_mirror_moves_equal_the_context(onb, tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_vl_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_vl_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    start = _undecided(1, 51)
    plies, sims, leaves = 6, 100, 8  # EVAL_UNIFORM on the device, and the same evaluator as a HostEvaluator
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d %d\n%s\n" % (plies, sims, leaves, line), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = [int(x) for x in p.stdout.split()[:-2]]
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(start)
        for _ in range(len(got) // 2):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_UNIFORM, vl=leaves)["best"][0]))
            ctx.mcts_play_best()
    assert got == want + want and len(want) >= 2  # the device evaluator, then the host evaluator


@pytest.mark.gpu
def test_beats_the_random_agent(onb):
    n, sims = 256, 64
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=8, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()
        w, l, d, _ = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM, leaves=8), ctx.agent_random(), a_is_red, 150)
    assert w >= 0.8 * n, (w, l, d)
