"""Tablebase leaves (onb_mcts_set_tablebase, ONB_AGENT_PUCT_TB, DESIGN.md §5i) on the GPU with a table solved on the device at two
pawns: the kernels against the CPU restatement (tests/tb_search_oracle.cpp) bit for bit on 4 096 roots (inside the table, one and
two pawns above it, dealt roots of other sets), with and without virtual loss; onb_mcts_run against the split phase, torch networks
with and without CUDA graphs against ONB_EVAL_NET; Gumbel and train-mode noise; the refusals and the freed table; the arena agent
against the Python driver, the C++ mirror and a strength check against plain PUCT."""
import numpy as np
import pytest

import tablebase_oracle as TBO
import tb_search_oracle as TS
from test_gpu_gumbel import KEYS, _same, _undecided
from test_tb_search_cpu import node_states, py_reward, undecided

CARDS = [0, 1, 2, 3, 11]
NONE = TBO.NONE
MAXP = 2


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


@pytest.fixture(scope="module")
def table(onb):
    """the device's two-pawn table of CARDS, downloaded"""
    with onb.Context(64, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        return {(p, q): ctx.tb_table(p, q).cpu().numpy().copy() for p in range(5) for q in range(5) if p + q <= MAXP}


def _roots(onb, table, n, seed):
    """n roots: a quarter inside the table, a quarter each one and two pawns above it, a quarter dealt (other sets)"""
    rng = np.random.default_rng(seed)
    parts = []
    picks = []
    for (p, q), t in sorted(table.items()):
        pool = np.nonzero(t != NONE)[0]
        picks.append(onb.tb_states(CARDS, 5 * p + q, rng.choice(pool, n // 4 // len(table) + 1)))
    parts.append(np.concatenate(picks)[:n // 4])
    for level in (MAXP + 1, MAXP + 2):
        cls = [(p, level - p) for p in range(level + 1)]
        st = np.concatenate([onb.tb_states(CARDS, 5 * p + q, rng.integers(0, TBO.entries(p, q), n // len(cls))) for p, q in cls])
        st = st[undecided(st)]
        parts.append(st[rng.permutation(len(st))[:n // 4]])
    parts.append(_undecided(n - sum(len(x) for x in parts), seed))
    return np.ascontiguousarray(np.concatenate(parts))


def check_tree(root, tree, table):
    """every node below the root that the table holds is unexpanded with W = N r (tests/test_tb_search_cpu.py at two pawns)"""
    st = node_states(root, tree)
    v = TBO.probe(CARDS, MAXP, table, st).astype(np.int32)
    depth = np.zeros(len(st), int)
    for i in range(1, len(st)):
        depth[i] = depth[tree["parent"][i]] + 1
    hits = 0
    for i in range(1, len(st)):
        if v[i] == NONE or tree["visits"][i] == 0:
            continue
        hits += 1
        assert tree["n_child"][i] == 0 and not (tree["flags"][i] & 1), i
        assert tree["reward"][i] == tree["visits"][i] * py_reward(v[i], depth[i], int(st["side"][i])), i
    return hits


def _search(ctx, c, sims, evaluator, leaves):
    ctx.set_virtual_loss(leaves, 1.0)
    ctx.set_tablebase(True)
    ctx.mcts_begin(c, sims)
    ctx.mcts_run(evaluator, sims)
    return ctx.mcts_finish()


@pytest.mark.gpu
@pytest.mark.parametrize("sims", [1, 2, 33, 400])
@pytest.mark.parametrize("leaves", [1, 2, 8])
@pytest.mark.parametrize("evaluator", [0, 1])
def test_equals_the_oracle(onb, table, evaluator, leaves, sims):
    n, c = 4096, 2.0
    roots = _roots(onb, table, n, 50 + sims + evaluator)
    want = TS.search(roots, c, sims, CARDS, MAXP, table, leaves=leaves, evaluator=evaluator)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_states(roots)
        got = _search(ctx, c, sims, evaluator, leaves)
        _same(got, want)
        assert np.array_equal(got["root_q"], want["root_q"])
        assert (got["root_visits"] == sims).all()
        nn, fl = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"]) and not (fl & 2).any()
        hits = 0
        for t in list(range(0, n, 331)) + [0, 1, n // 4 + 1, n // 2 + 1]:
            tree = TS.search(roots[t:t + 1], c, sims, CARDS, MAXP, table, leaves=leaves, evaluator=evaluator, dump_tree=0)["tree"]
            mine = ctx.mcts_dump_tree(t)
            for k in KEYS:
                assert np.array_equal(mine[k], tree[k].astype(mine[k].dtype)), (t, k)
            hits += check_tree(roots[t], mine, table)
        assert sims < 33 or hits > 0


def _split(ctx, c, sims, evaluator):
    ctx.mcts_begin(c, sims)
    for _ in range(ctx.vl_rounds(sims)):
        ctx.mcts_select()
        ctx.mcts_eval(evaluator)
        ctx.mcts_expand_backup()
    return ctx.mcts_finish()


@pytest.mark.gpu
def test_run_equals_the_split_phase_and_torch_nets(onb, table):
    from test_net_cpu import lively_model
    n, sims, c = 256, 61, 2.0
    roots = _roots(onb, table, n, 9)
    keys = ("best", "pi", "root_visits", "root_q", "child_visits")
    model = lively_model(3, seed=5)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_states(roots)
        ctx.net_load(model)
        for leaves in (1, 8):
            ctx.set_virtual_loss(leaves, 1.0)
            ctx.set_tablebase(True)
            for ev in (onb.EVAL_UNIFORM, onb.EVAL_HASH, onb.EVAL_NET):
                _same(_split(ctx, c, sims, ev), ctx.search(c, sims, evaluator=ev), keys=keys)
        # torch networks over the leaf rows, eagerly and in CUDA graphs, against ONB_EVAL_NET
        for leaves in (1, 16):
            rows = n * leaves
            with onb.Context(rows, stream=ctx.stream_handle(), mcts_max_sims=1, planes=True) as aux:
                aux.net_load(model)
                want = ctx.search(c, sims, evaluator=onb.EVAL_NET, vl=leaves, tb=True)
                planes, pol, val = aux.tensor(onb.BUF_PLANES), aux.tensor(onb.BUF_POLICY), aux.tensor(onb.BUF_VALUE)

                def net(x):
                    planes[:len(x)].copy_(x)
                    aux.net_forward(onb.BUF_PLANES)
                    return pol[:len(x)], val[:len(x)]

                _same(ctx.search(c, sims, net=net), want, keys=keys)
                for graph in (False, True, True):
                    ctx.search_device(c, sims, net=net, use_graph=graph)
                    _same(ctx.mcts_finish(), want, keys=keys)
                # a new solve switches the leaves off and replaces the table a captured round was given: the next graph is new
                ctx.tb_solve(CARDS, MAXP)
                ctx.search_device(c, sims, net=net, use_graph=True, tb=True)
                _same(ctx.mcts_finish(), want, keys=keys)
        import torch
        torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["gumbel", "muzero", "noise"])
def test_gumbel_and_noise(onb, table, mode):
    n, sims, c = 512, 64, 2.0
    roots = _roots(onb, table, n, 23)
    other = np.arange(n) >= 3 * n // 4
    keys = ("best", "pi", "root_visits", "root_q", "child_visits")
    with onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ctx, onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ref:
        ctx.tb_solve(CARDS, MAXP)
        for x in (ctx, ref):
            x.set_states(roots)
            if mode == "noise":
                x.mcts_set_noise(True, seed=5)
            else:
                x.set_gumbel(True, m=8, interior=mode == "muzero")
        ctx.set_tablebase(True)
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(onb.EVAL_HASH, sims)
        got = ctx.mcts_finish()
        ref.mcts_begin(c, sims)
        for _ in range(sims):  # the split phase: with tablebase leaves onb_mcts_run runs its rounds
            ref.mcts_select()
            ref.mcts_eval(onb.EVAL_HASH)
            ref.mcts_expand_backup()
        want = ref.mcts_finish()
        for k in keys:
            assert np.array_equal(got[k][other], want[k][other]), k
        hits = sum(check_tree(roots[t], ctx.mcts_dump_tree(t), table) for t in range(0, 3 * n // 4, 5))
        assert hits > 50


@pytest.mark.gpu
def test_switch_refusals_and_the_freed_table(onb, table):
    n, sims, c = 128, 40, 2.0
    roots = _roots(onb, table, n, 3)

    def code(fn, *a, **kw):
        with pytest.raises(onb.OnbError) as e:
            fn(*a, **kw)
        return e.value.code

    E_STATE = onb._lib.E_STATE
    with onb.Context(n, seed=1, mcts_max_sims=sims, planes=True) as ctx, onb.Context(n, seed=1, mcts_max_sims=sims, planes=True) as ref:
        for x in (ctx, ref):
            x.set_states(roots)
        assert code(ctx.set_tablebase, True) == E_STATE  # no table
        assert code(ctx.fight_native, ctx.agent_puct(sims, tablebase=True), ctx.agent_random(), np.ones(n, bool), 4) == E_STATE
        with pytest.raises(ValueError):
            ctx.agent_puct(sims, leaves=4, tablebase=True)
        ctx.tb_solve(CARDS, MAXP)
        ref.tb_solve(CARDS, MAXP)
        # switched off, every entry point computes what it does without the table
        for fused in (True, False):
            _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused, tb=False), ref.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused),
                  keys=("best", "pi", "root_q", "child_visits"))
        on = ctx.search(c, sims, evaluator=onb.EVAL_HASH, tb=True)
        # refusals
        ctx.set_reuse(True)
        assert code(ctx.mcts_begin, c, sims) == E_STATE
        ctx.set_reuse(False)
        assert code(ctx.self_play_native, c, sims, 4, 10, onb.EVAL_HASH) == E_STATE
        ctx.set_states(roots)
        ctx.mcts_begin(c, sims)
        assert code(lambda: ctx._ck(ctx._lib.onb_uct_run(ctx._h, 1.4, 5, sims))) == E_STATE
        # a search begun with the table, then the table is freed: no further step reads it
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(onb.EVAL_HASH, 5)
        ctx.mcts_select()
        ctx.tb_free()
        assert not ctx.tb_leaves
        assert code(ctx.mcts_expand_backup) == E_STATE
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_tablebase(True)
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(onb.EVAL_HASH, 5)
        ctx.tb_solve(CARDS, MAXP)  # a new solve frees the old table too, and switches the leaves off
        assert code(ctx.mcts_run, onb.EVAL_HASH, 5) == E_STATE
        assert code(ctx.mcts_select) == E_STATE
        ctx.set_tablebase(True)
        _same(ctx.search(c, sims, evaluator=onb.EVAL_HASH), on, keys=("best", "pi", "root_q", "child_visits"))
        ctx.set_tablebase(False)
        ctx.set_states(roots)
        ctx.self_play_native(c, 8, 4, 10, onb.EVAL_HASH)


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import fight, puct_tb_move
    n, sims, max_plies = 128, 24, 60
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=11, mcts_max_sims=sims) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        rng = np.random.default_rng(2)
        st = np.concatenate([onb.tb_states(CARDS, 5 * p + (3 - p), rng.integers(0, TBO.entries(p, 3 - p), n)) for p in range(4)])
        st = np.ascontiguousarray(st[undecided(st)][:n])
        ctx.set_states(st)
        ag = ctx.agent_puct(sims, 2.0, onb.EVAL_HASH, tablebase=True)
        nat = ctx.fight_native(ag, ctx.agent_puct(sims, 2.0, onb.EVAL_HASH), a_is_red, max_plies)
        assert not getattr(ctx, "tb_leaves", False)  # onb_fight left the switch as it found it
        ctx.set_states(st)

        def plain(x):
            x.search_device(2.0, sims, evaluator=onb.EVAL_HASH, tb=False)
            x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))

        py = fight(ctx, puct_tb_move(sims, 2.0, onb.EVAL_HASH), plain, a_is_red, max_plies)
        assert nat[:3] == tuple(py[:3])
        assert np.array_equal(nat[3], ctx.last_fight_results)


@pytest.mark.gpu
def test_won_and_drawn_positions_are_kept(onb, table):
    rng = np.random.default_rng(4)
    n, sims = 512, 64
    picks = []
    for (p, q), t in sorted(table.items()):
        tv = t.astype(np.int32)
        pool = np.nonzero((t != NONE) & (tv >= 0))[0]
        picks.append(onb.tb_states(CARDS, 5 * p + q, rng.choice(pool, n)))
    st = np.concatenate(picks)
    st = np.ascontiguousarray(st[rng.permutation(len(st))[:n]])
    with onb.Context(n, seed=6, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_states(st)
        v = ctx.tb_probe().astype(np.int32)
        a_is_red = st["side"] == 0  # the agent is to move and holds the win or the draw
        _, _, _, res = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM, tablebase=True), ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM),
                                        a_is_red, 150)
        a_lost = np.where(a_is_red, res == 2, res == 1)
        a_won = np.where(a_is_red, res == 1, res == 2)
        assert not a_lost.any()
        assert a_won[v > 0].all()


@pytest.mark.gpu
def test_mirror_equals_the_context(onb, tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_tb_search_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_tb_search_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    rng = np.random.default_rng(51)
    st = onb.tb_states(CARDS, 5 * 2 + 1, rng.integers(0, TBO.entries(2, 1), 64))  # one pawn above the table
    start = np.ascontiguousarray(st[undecided(st)][:1])
    plies, sims, games, fight_plies = 8, 100, 64, 40
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d %d %d %d\n%s\n%s\n" % (plies, sims, MAXP, games, fight_plies, " ".join(map(str, CARDS)), line),
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    lines = p.stdout.split("\n")
    k = next(i for i, x in enumerate(lines) if x.startswith("FIGHT"))
    got = [int(x) for x in lines[:k]]
    wld = tuple(int(x) for x in lines[k].split()[1:])
    results = np.array([int(x) for x in lines[k + 1].split()], np.uint8)
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_states(start)
        for _ in range(len(got) // 2):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_UNIFORM, tb=True)["best"][0]))
            ctx.mcts_play_best()
    assert got == want + want and len(want) >= 2  # the device evaluator, then the host evaluator
    # fight_device with ONB_AGENT_PUCT_TB equals onb_fight from Python on the same deck and seed
    with onb.Context(games, seed=0, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.reset(CARDS)
        a, b, d, res = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM, tablebase=True), ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM),
                                        np.arange(games) % 2 == 0, fight_plies)
    assert wld == (a, b, d)
    assert np.array_equal(results, res)
