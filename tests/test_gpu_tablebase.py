"""The endgame tablebase on the GPU (onb_tb_*, ONB_AGENT_TABLEBASE, DESIGN.md §5g): the solved tables bit for bit against the oracle
(tests/tablebase_oracle.cpp), whole-table identities at three pawns, the alpha-beta kernel's win scores, probe, best move, the
tablebase agent in onb_fight and the C++ mirror."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import tablebase_oracle as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NONE = T.NONE
SURVEY = [0, 1, 2, 3, 11]
SETS = [SURVEY, [4, 5, 6, 7, 8], [9, 10, 12, 13, 14], [15, 0, 5, 10, 3], [1, 6, 11, 12, 2], [7, 8, 13, 14, 4], [3, 9, 15, 6, 0],
        [2, 4, 8, 10, 12], [5, 7, 11, 13, 15], [0, 14, 9, 6, 1], [3, 12, 4, 10, 7], [8, 11, 2, 15, 13]]
WIN = 1000000


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def download(ctx, max_pawns):
    return {(p, q): ctx.tb_table(p, q).cpu().numpy().copy() for p in range(5) for q in range(5) if p + q <= max_pawns}


def check_counts(tables, info):
    for k, t in tables.items():
        s = info[k]
        w = int((t > 0).sum())
        inv = int((t == NONE).sum())
        assert s["entries"] == len(t) and s["wins"] == w and s["invalid"] == inv, k
        assert s["losses"] == len(t) - w - inv - int((t == 0).sum()) and s["draws"] == int((t == 0).sum()), k
        live = t[t != NONE].astype(np.int32)
        assert s["max_win"] == max(0, int(live.max(initial=0))) and s["max_loss"] == max(0, -int(live.min(initial=0))), k


@pytest.mark.gpu
def test_small_classes_equal_the_oracle_bit_for_bit(onb):
    with onb.Context(64, planes=False) as ctx:
        for cards in SETS:
            info = ctx.tb_solve(cards, 1)
            got = download(ctx, 1)
            want, winfo = T.solve(cards, 1)
            for k in got:
                assert np.array_equal(got[k], want[k]), (cards, k, np.nonzero(got[k] != want[k])[0][:5])
                assert info[k]["iterations"] == winfo[k]["iterations"], (cards, k)
            check_counts(got, info)
        for cards in SETS[:2]:
            info = ctx.tb_solve(cards, 2)
            got = download(ctx, 2)
            want, _ = T.solve(cards, 2)
            for k in got:
                assert np.array_equal(got[k], want[k]), (cards, k)
            check_counts(got, info)
            again = ctx.tb_solve(list(reversed(cards)), 2)  # any order of the ids; a second solve gives the same bytes
            assert again == info
            for k, t in download(ctx, 2).items():
                assert t.tobytes() == got[k].tobytes(), k


@pytest.fixture(scope="module")
def three(onb):
    """max_pawns 3 of two card sets: (cards, tables, per-class info)"""
    out = []
    with onb.Context(64, planes=False) as ctx:
        for cards in (SURVEY, [4, 5, 6, 7, 8]):
            info = ctx.tb_solve(cards, 3)
            print(cards, info)
            out.append((cards, download(ctx, 3), info))
    return out


@pytest.mark.gpu
def test_three_pawns_identities(onb, three):
    rng = np.random.default_rng(3)
    for cards, tables, info in three:
        check_counts(tables, info)
        for (p, q), t in tables.items():
            assert T.check_swap(cards, 3, tables, p, q) == 0, (cards, p, q)
            idx = rng.choice(len(t), min(len(t), 10 ** 6), replace=False)
            bad, first = T.check_local(cards, 3, tables, p, q, idx=idx)
            assert bad == 0, (cards, p, q, first)


def sample(tables, rng, n_per_class, short_half=True):
    """(class, entry) pairs: per class n_per_class entries of the table, half of them with 0 < |v| <= 6"""
    out = []
    for (p, q), t in sorted(tables.items()):
        v = t.astype(np.int32)
        pools = [np.nonzero((t != NONE) & (v != 0) & (np.abs(v) <= 6))[0], np.nonzero((t != NONE) & ((np.abs(v) > 6) | (v == 0)))[0]]
        if not short_half:
            pools = [np.nonzero(t != NONE)[0]]
        for pool in pools:
            if len(pool):
                k = n_per_class // len(pools)
                out += [(5 * p + q, int(i)) for i in rng.choice(pool, k, replace=len(pool) < k)]
    return out


def states_of(onb, cards, picks):
    if not picks:
        return np.zeros(0, dtype=onb.STATE_DTYPE)
    return np.concatenate([onb.tb_states(cards, c, [i]) for c, i in picks])


def sq(row, col):
    """reference layout: square n = row * 5 + col is bit 31 - n"""
    return 1 << (31 - (row * 5 + col))


@pytest.mark.gpu
def test_alphabeta_win_scores_follow_the_table(onb, three):
    rng = np.random.default_rng(7)
    for cards, tables, _ in three:
        picks = sample(tables, rng, 4096)
        st = states_of(onb, cards, picks)
        v = np.array([tables[(c // 5, c % 5)][i] for c, i in picks], np.int32)
        with onb.Context(len(st), planes=False) as ctx:
            ctx.set_states(st)
            score = ctx.alphabeta(6)["score"]
        short = (v != 0) & (np.abs(v) <= 6)
        assert short.sum() >= len(v) // 3
        assert np.array_equal(score[short], np.sign(v[short]) * (WIN - np.abs(v[short])))
        assert (np.abs(score[~short]) < WIN - 6).all()


@pytest.mark.gpu
def test_probe_and_best(onb, three):
    rng = np.random.default_rng(9)
    cards, tables, _ = three[0]
    picks = sample(tables, rng, 4096, short_half=False)
    st = states_of(onb, cards, picks)
    # other hand orders, other slot contents of the same position
    swap = rng.random(len(st)) < 0.5
    st["cards"][swap] = st["cards"][swap][:, [1, 0, 3, 2, 4]]
    n = len(st)
    with onb.Context(n, planes=False) as ctx:
        ctx.tb_solve(cards, 3)
        ctx.set_states(st)
        got = ctx.tb_probe()
        cls, idx = onb.tb_index(cards, st)
        want = np.array([tables[(c // 5, c % 5)][i] for c, i in zip(cls, idx)], np.int16)
        assert np.array_equal(got, want)
        assert np.array_equal(got, T.probe(cards, 3, tables, st))
        best = ctx.tb_best()
        assert np.array_equal(ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)), best)
        assert np.array_equal(best, T.best(cards, 3, tables, st))
        assert (best != 0xFFFF).all()
        # decided games, a foreign card set and an unsolved class are outside the table
        other = [c for c in range(16) if c not in cards][0]
        odd = np.concatenate([
            O.make_state(cards, kings=[sq(1, 1), sq(3, 3)], pawns=[0, 0], side=0),               # decided below (result = 1)
            O.make_state(cards, kings=[sq(0, 2), sq(3, 3)], pawns=[0, 0], side=1),               # red king on the blue temple
            O.make_state(cards[:4] + [other], kings=[sq(1, 1), sq(3, 3)], pawns=[0, 0], side=0),  # another card set
            O.make_state(cards, kings=[sq(1, 1), sq(3, 3)], pawns=[sq(4, 0) | sq(4, 1), sq(0, 0) | sq(0, 4)], side=0)])  # 4 pawns
        odd["result"][0] = 1
        ctx.set_states(odd)
        got = ctx.tb_probe()[:4]
        assert (got == NONE).all(), got
        assert (ctx.tb_best()[:4] == 0xFFFF).all()


def _start_positions(onb, cards, tables, rng, want, n):
    """n states of the ≤ 3-pawn table whose value satisfies want(v)"""
    picks = []
    for (p, q), t in sorted(tables.items()):
        pool = np.nonzero((t != NONE) & want(t.astype(np.int32)))[0]
        if len(pool):
            picks += [(5 * p + q, int(i)) for i in rng.choice(pool, n // len(tables) + 1)]
    picks = picks[:n]
    st = states_of(onb, cards, picks)
    return st, np.array([tables[(c // 5, c % 5)][i] for c, i in picks], np.int32)


@pytest.mark.gpu
def test_fight(onb, three):
    rng = np.random.default_rng(12)
    cards, tables, _ = three[0]
    n = 512
    with onb.Context(n, seed=5, planes=False) as ctx:
        ctx.tb_solve(cards, 3)
        tb = ctx.agent_tablebase()
        # tablebase against tablebase from wins in n: the game ends at exactly ply n, won by the side to move
        st, v = _start_positions(onb, cards, tables, rng, lambda v: (v > 0) & (v <= 41), n)
        ctx.set_states(st)
        a_is_red = st["side"] == 0  # agent A moves first and holds the win
        a, b, d, res = ctx.fight_native(tb, tb, a_is_red, max_plies=150)
        assert a == n and b == 0 and d == 0
        ctx.set_states(st)
        ends = np.full(n, -1)
        for ply in range(1, 42):
            ctx.tb_best(to_host=False)
            ctx.step(None)
            r = ctx.get_states()["result"]
            ends[(r != 0) & (ends < 0)] = ply
        assert np.array_equal(ends, v)
        # from draws, if the set has any, the game runs to the ply cap
        st, v = _start_positions(onb, cards, tables, rng, lambda v: v == 0, 64)
        if len(st):
            m = len(st)
            full = np.concatenate([st] + [st[:1]] * (n - m))
            ctx.set_states(full)
            a, b, d, res = ctx.fight_native(tb, tb, np.ones(n, bool), max_plies=20)
            assert d == n and ctx.last_fight_plies == 22
        # tablebase against a random legal mover (uniform over the legal moves) never loses a won or drawn position and wins every won
        # one within n plies. (The reference's `Random` agent, ONB_AGENT_RANDOM, also makes moves outside the rules -- a Blue card
        # index without the +2 of random.rs:39, fabricated pieces -- against which the table's values promise nothing.)
        st, v = _start_positions(onb, cards, tables, rng, lambda v: (v >= 0) & (v <= 101), n)
        tb_red = st["side"] == 0
        ctx.set_states(st)
        ends = np.full(n, -1)
        for ply in range(1, 152):
            ctx.tb_best(to_host=False)
            tba = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)).copy()
            ctx.choose_random(ply - 1, policy=onb.POLICY_UNIFORM)
            rnd = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)).copy()
            side = ctx.get_states()["side"]
            ctx.step(np.where((side == 0) == tb_red, tba, rnd))
            r = ctx.get_states()["result"]
            ends[(r != 0) & (ends < 0)] = ply
        r = ctx.get_states()["result"]
        tb_won = np.where(tb_red, r == 1, r == 2)
        assert (tb_won | (r == 0)).all()
        assert tb_won[v > 0].all() and (ends[v > 0] <= v[v > 0]).all()
        # the native fight equals the Python-driven one game for game
        for cap in (150, 3):
            counter = {"i": 0}

            def py_random(cx):
                cx.choose_random(counter["i"], policy=onb.POLICY_AGENT)
                counter["i"] += 1

            ctx.set_states(st)
            want = onb.fight(ctx, lambda cx: cx.tb_best(to_host=False), py_random, tb_red, max_plies=cap)
            want_states = ctx.get_states().tobytes()
            ctx.set_states(st)
            got = ctx.fight_native(tb, ctx.agent_random(), tb_red, max_plies=cap)
            assert got[:3] == want and ctx.get_states().tobytes() == want_states
        # error paths: a start outside the table, no table
        ctx.reset()
        with pytest.raises(onb.OnbError) as e:
            ctx.fight_native(tb, ctx.agent_random(), tb_red)
        assert e.value.code == -1
        ctx.tb_free()
        ctx.set_states(st)
        for call in (lambda: ctx.fight_native(tb, ctx.agent_random(), tb_red), ctx.tb_probe, ctx.tb_best, lambda: ctx.tb_table(0, 0)):
            with pytest.raises(onb.OnbError) as e:
                call()
            assert e.value.code == -4
        for bad in (([0, 1, 2, 3, 3], 1), ([0, 1, 2, 3, 16], 1), (SURVEY, 5), (SURVEY, -1)):
            with pytest.raises(onb.OnbError) as e:
                ctx.tb_solve(*bad)
            assert e.value.code == -1


@pytest.mark.gpu
def test_cpp_mirror_agent_equals_context_tb_best(onb, three, tmp_path):
    exe = str(tmp_path / "test_tablebase_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_tablebase_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(ROOT, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(ROOT, "onitama_alphazero_b200")])
    cards, tables, _ = three[0]
    st = states_of(onb, cards, sample({k: t for k, t in tables.items() if sum(k) <= 1}, np.random.default_rng(4), 40, short_half=False))
    lines = ["%d %s" % (len(st), " ".join(map(str, cards)))]
    for r in st:
        lines.append(" ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"])))
    p = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = np.array([int(x) for x in p.stdout.strip().splitlines()[:len(st)]])
    with onb.Context(len(st), planes=False) as ctx:
        ctx.tb_solve(cards, 1)
        ctx.set_states(st)
        want = ctx.tb_best()
    assert np.array_equal(got, want.astype(np.int64))
