"""The MCTS solver (onb_mcts_set_solver, ONB_AGENT_PUCT_SOLVER, DESIGN.md §5k) on the GPU: the kernels against the CPU restatement
(tests/solver_oracle.cpp) bit for bit on 4 096 roots, trees and proof flags included, with and without tablebase leaves, fused against
the split phase; every proof of 4 096 searches against a table solved on the device; the deterministic consequences (immediate wins,
positions lost in two plies); the switch set and cleared; the refusals; and the arena agent against the Python driver."""
import numpy as np
import pytest

import oracle_lib as O
import solver_oracle as SO
import tablebase_oracle as TBO
from test_gpu_gumbel import KEYS, _same, _undecided
from test_gpu_tb_search import CARDS, MAXP, NONE, _roots
from test_tb_search_cpu import node_states, undecided

WIN, LOSS = SO.WIN, SO.LOSS


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


def _five_pawns(onb, n, seed):
    """n undecided positions of the set with five pawns: a pawn added on a free square of a position of the four-pawn classes"""
    rng = np.random.default_rng(seed)
    cls = [(p, 4 - p) for p in range(1, 4)]
    st = np.concatenate([onb.tb_states(CARDS, 5 * p + q, rng.integers(0, TBO.entries(p, q), n)) for p, q in cls])
    out = []
    for s in st[rng.permutation(len(st))]:
        occ = int(s["pawns"][0]) | int(s["pawns"][1]) | int(s["kings"][0]) | int(s["kings"][1])
        free = [q for q in range(25) if not occ & (1 << (31 - q))]
        side = int(bin(int(s["pawns"][0])).count("1") > bin(int(s["pawns"][1])).count("1"))
        t = s.copy()
        t["pawns"][side] = int(t["pawns"][side]) | (1 << (31 - int(rng.choice(free))))
        out.append(t)
    st = np.array(out, dtype=st.dtype)
    return np.ascontiguousarray(st[undecided(st)][:n])


def _roots5(onb, table, n, seed):
    """test_gpu_tb_search's roots (inside the two-pawn table, 3 and 4 pawns, dealt) with an eighth replaced by 5-pawn roots"""
    r5 = _five_pawns(onb, n // 8, seed)
    assert len(r5) == n // 8 and ((np.vectorize(lambda x: bin(int(x)).count("1"))(r5["pawns"])).sum(axis=1) == 5).all()
    return np.ascontiguousarray(np.concatenate([_roots(onb, table, n - n // 8, seed), r5]))


def _search(ctx, c, sims, evaluator, tb, fused=True):
    ctx.set_solver(True)
    ctx.set_tablebase(tb)
    ctx.mcts_begin(c, sims)
    if fused:
        ctx.mcts_run(evaluator, sims)
    else:
        for _ in range(sims):
            ctx.mcts_select()
            ctx.mcts_eval(evaluator)
            ctx.mcts_expand_backup()
    out = ctx.mcts_finish()
    out["proof"] = ctx.root_proof()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("sims", [1, 2, 33, 400])
@pytest.mark.parametrize("tb", [False, True])
@pytest.mark.parametrize("evaluator", [0, 1])
def test_equals_the_oracle(onb, table, evaluator, tb, sims):
    n, c = 4096, 2.0
    roots = _roots5(onb, table, n, 70 + sims + evaluator)
    want = SO.search(roots, c, sims, evaluator=evaluator, table=(CARDS, MAXP, table) if tb else None)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.tb_solve(CARDS, MAXP)
        ctx.set_states(roots)
        got = _search(ctx, c, sims, evaluator, tb)
        _same(got, want)
        assert np.array_equal(got["root_q"], want["root_q"])
        assert np.array_equal(got["proof"], want["proof"])
        nn, fl = ctx.mcts_tree_info()
        assert np.array_equal(nn.astype(np.int64), want["n_nodes"]) and not (fl & 2).any()
        for t in list(range(0, n, 331)) + [1, n // 4 + 1, n // 2 + 1, n - 1]:
            tree = SO.search(roots[t:t + 1], c, sims, evaluator=evaluator, table=(CARDS, MAXP, table) if tb else None, dump_tree=0)["tree"]
            mine = ctx.mcts_dump_tree(t)
            for k in KEYS:
                assert np.array_equal(mine[k], tree[k].astype(mine[k].dtype)), (t, k)
    assert sims < 33 or (want["proof"] != 0).sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [0, 1])
def test_fused_equals_the_split_phase(onb, table, evaluator):
    n, sims, c = 512, 61, 2.0
    roots = _roots(onb, table, n, 5 + evaluator)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        a = _search(ctx, c, sims, evaluator, False, fused=True)
        ta = [ctx.mcts_dump_tree(t) for t in range(0, n, 37)]
        ctx.set_states(roots)
        b = _search(ctx, c, sims, evaluator, False, fused=False)
        tb_ = [ctx.mcts_dump_tree(t) for t in range(0, n, 37)]
    for k in ("best", "pi", "root_visits", "root_q", "child_visits", "proof"):
        assert np.array_equal(a[k], b[k]), k
    for x, y in zip(ta, tb_):
        for k in KEYS:
            assert np.array_equal(x[k], y[k]), k


@pytest.mark.gpu
def test_every_proof_agrees_with_the_table(onb, table):
    """table leaves off: every proven node of 4 096 searches of 800 simulations has the sign the table gives its position"""
    n, sims = 4096, 800
    rng = np.random.default_rng(12)
    picks = []
    for (p, q), t in sorted(table.items()):
        pool = np.nonzero(t != NONE)[0]
        picks.append(onb.tb_states(CARDS, 5 * p + q, rng.choice(pool, n)))
    st = np.concatenate(picks)
    st = st[undecided(st)]
    roots = np.ascontiguousarray(st[rng.permutation(len(st))[:n]])
    v = TBO.probe(CARDS, MAXP, table, roots).astype(np.int32)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        _search(ctx, 2.0, sims, 1, False)
        proof = ctx.root_proof()
        assert ((proof == 0) | (np.sign(v) == proof)).all()
        assert (proof != 0).mean() > 0.5
        checked = 0
        for t in range(0, n, 16):
            tree = ctx.mcts_dump_tree(t)
            fl = tree["flags"]
            assert not ((fl & WIN) & (fl & LOSS)).any()
            idx = np.nonzero(fl & (WIN | LOSS))[0]
            if len(idx) == 0:
                continue
            sub = {k: tree[k] for k in ("parent", "action")}
            vs = TBO.probe(CARDS, MAXP, table, node_states(roots[t], sub)[idx]).astype(np.int32)
            for i, x in zip(idx, vs):
                if x == NONE:
                    assert fl[i] & 2 and fl[i] & WIN
                else:
                    assert x != 0 and (x < 0) == bool(fl[i] & WIN), (t, i, x, fl[i])
                checked += 1
        assert checked > 1000


def _winning_moves(roots):
    out = []
    for r in roots:
        g = r.reshape(1).copy()
        w = set()
        for a in O.gen_moves(g):
            h = g.copy()
            O.make_move(h, int(a))
            if h["result"][0] != 0:
                w.add(int(a))
        out.append(w)
    return out


@pytest.mark.gpu
def test_immediate_wins_are_proven_after_one_simulation(onb):
    n = 4096
    roots = _undecided(n, 23)
    wins = _winning_moves(roots)
    has = np.array([len(w) > 0 for w in wins])
    assert has.sum() > 20
    with onb.Context(n, mcts_max_sims=8, planes=False) as ctx:
        for evaluator in (0, 1):
            ctx.set_states(roots)
            out = _search(ctx, 2.0, 1, evaluator, False)
            assert (out["proof"][has] == 1).all() and (out["proof"][~has] == 0).all()
            assert all(int(b) in w for b, w, h in zip(out["best"], wins, has) if h)


@pytest.mark.gpu
def test_positions_lost_in_two_plies(onb, table):
    """value -2: every move lets the opponent win at once; 1 + (number of children) simulations prove the root WIN (proof -1)"""
    rng = np.random.default_rng(8)
    picks = []
    for (p, q), t in sorted(table.items()):
        pool = np.nonzero(t.astype(np.int32) == -2)[0]
        if len(pool):
            picks.append(onb.tb_states(CARDS, 5 * p + q, rng.choice(pool, 64)))
    roots = np.concatenate(picks)
    roots = np.ascontiguousarray(roots[undecided(roots)][:256])
    assert len(roots) > 16
    kids = np.array([len(O.gen_moves(r.reshape(1).copy())) for r in roots])
    assert (kids > 0).all()
    with onb.Context(len(roots), mcts_max_sims=64, planes=False) as ctx:
        for k in np.unique(kids):
            sel = np.nonzero(kids == k)[0]
            ctx.set_states(roots)
            out = _search(ctx, 2.0, int(1 + k), 1, False)
            assert (out["proof"][sel] == -1).all(), k


@pytest.mark.gpu
def test_switch_set_then_cleared_changes_nothing(onb, table):
    n, sims = 1024, 50
    roots = _roots(onb, table, n, 3)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        a = ctx.search(2.0, sims, onb.EVAL_HASH)
        ta = [ctx.mcts_dump_tree(t) for t in range(0, n, 101)]
        ctx.set_solver(True)
        ctx.set_solver(False)
        ctx.set_states(roots)
        b = ctx.search(2.0, sims, onb.EVAL_HASH)
        tb_ = [ctx.mcts_dump_tree(t) for t in range(0, n, 101)]
        ctx.set_states(roots)
        c = ctx.search(2.0, sims, onb.EVAL_HASH, fused=False)
    want = O.mcts_search_batch(roots, 2.0, sims, evaluator=1, threads=8)
    for k in ("best", "pi", "root_q", "child_visits"):
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), k
    assert np.array_equal(a["best"], want["best"])
    for x, y in zip(ta, tb_):
        for k in KEYS:
            assert np.array_equal(x[k], y[k]), k
        assert not (x["flags"] & (WIN | LOSS)).any()


@pytest.mark.gpu
def test_refusals(onb):
    n = 64
    with onb.Context(n, mcts_max_sims=8, planes=True) as ctx:
        with pytest.raises(onb.OnbError) as e:
            ctx.buffer(onb.BUF_ROOT_PROOF)
        assert e.value.code == onb._lib.E_STATE
        ctx.reset()
        ctx.set_solver(True)
        ctx.buffer(onb.BUF_ROOT_PROOF)
        for setup, undo in ((lambda: ctx.mcts_set_noise(True), lambda: ctx.mcts_set_noise(False)),
                            (lambda: ctx.set_gumbel(True), lambda: ctx.set_gumbel(False)),
                            (lambda: ctx.set_virtual_loss(4), lambda: ctx.set_virtual_loss(1)),
                            (lambda: ctx.set_reuse(True), lambda: ctx.set_reuse(False))):
            setup()
            with pytest.raises(onb.OnbError) as e:
                ctx.mcts_begin(2.0, 8)
            assert e.value.code == onb._lib.E_STATE
            undo()
        ctx.mcts_begin(2.0, 8)
        with pytest.raises(onb.OnbError) as e:
            ctx.uct_search(playouts=4)
        assert e.value.code == onb._lib.E_STATE
        with pytest.raises(onb.OnbError) as e:
            ctx.self_play_native(2.0, 4, 4, 10, onb.EVAL_UNIFORM)
        assert e.value.code == onb._lib.E_STATE
        ctx.set_solver(False)
        ctx.mcts_begin(2.0, 8)
        ctx.mcts_run(onb.EVAL_UNIFORM, 8)
        ctx.mcts_finish()
    with pytest.raises(ValueError):
        onb.Context.agent_puct(8, solver=True, leaves=2)
    with pytest.raises(ValueError):
        onb.Context.agent_puct(8, solver=True, tablebase=True)


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    from onitama_alphazero_b200.selfplay import fight, puct_solver_move
    n, sims, max_plies = 256, 32, 80
    a_is_red = (np.arange(n) % 2 == 0)
    with onb.Context(n, seed=13, mcts_max_sims=sims) as ctx:
        ctx.reset()
        st = ctx.get_states()
        nat = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_HASH, solver=True), ctx.agent_puct(sims, 2.0, onb.EVAL_HASH), a_is_red,
                               max_plies)
        assert not ctx.solver
        ctx.set_states(st)

        def plain(x):
            x.search_device(2.0, sims, evaluator=onb.EVAL_HASH, solver=False)
            x.tensor(onb.BUF_ACTIONS).copy_(x.tensor(onb.BUF_BEST))

        py = fight(ctx, puct_solver_move(sims, 2.0, onb.EVAL_HASH), plain, a_is_red, max_plies)
        assert nat[:3] == tuple(py[:3])
        assert np.array_equal(nat[3], ctx.last_fight_results)
        assert not ctx.solver


@pytest.mark.gpu
def test_mirror_equals_the_context(onb, tmp_path):
    """the C++ mirror (AlphaZeroMctsConfig::solver, puct_solver_agent in fight_device) against the context"""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_solver_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_solver_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    start = _undecided(8, 61)[:1]
    plies, sims, games, fight_plies = 10, 100, 64, 60
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d %d %d\n%s\n" % (plies, sims, games, fight_plies, line), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    lines = p.stdout.split("\n")
    k = next(i for i, x in enumerate(lines) if x.startswith("FIGHT"))
    got = [int(x) for x in lines[:k]]
    wld = tuple(int(x) for x in lines[k].split()[1:])
    results = np.array([int(x) for x in lines[k + 1].split()], np.uint8)
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(start)
        for _ in range(len(got) // 2):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_UNIFORM, solver=True)["best"][0]))
            ctx.mcts_play_best()
    assert got == want + want and len(want) >= 2  # the device evaluator, then the host evaluator
    # fight_device with ONB_AGENT_PUCT_SOLVER equals onb_fight from Python on the same deals
    with onb.Context(games, seed=0, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()
        a, b, d, res = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM, solver=True), ctx.agent_puct(sims, 2.0, onb.EVAL_UNIFORM),
                                        np.arange(games) % 2 == 0, fight_plies)
    assert wld == (a, b, d)
    assert np.array_equal(results, res)
