"""The alpha-beta arena opponent (ONB_AGENT_ALPHABETA, DESIGN.md §5d).

CPU (unmarked): the evaluation spec, known answers and the exactness of the pruning, on the oracle restatement
(tests/alphabeta_oracle.cpp). GPU (@pytest.mark.gpu): onb_alphabeta_run bit-exact against the oracle (best action, score, node
count), batching and subsets, the arena inside the library against the Python-driven one, errors, and the C++ mirror's agent."""
import json
import os
import subprocess

import numpy as np
import pytest

import alphabeta_oracle as A
import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
WIN = A.WIN
NONE = 0xFFFF
PASS_BIT = 1 << 13
# card ids (card.rs order)
TIGER, DRAGON, FROG, RABBIT, CRAB, ELEPHANT, GOOSE, ROOSTER, MONKEY, MANTIS, CRANE, HORSE, OX, BOAR, EEL, COBRA = range(16)


def sq(row, col):
    """reference bit layout: square n = row * 5 + col is bit 31 - n"""
    return 1 << (31 - (row * 5 + col))


def midgame_roots(n, seed, plies_mod=24):
    """positions after p random plies (uniform policy), p = game mod plies_mod: some games are already decided"""
    g = O.new_games(n, seed=seed)
    out = g.copy()
    for step in range(plies_mod):
        take = (np.arange(n) % plies_mod) == step
        out[take] = g[take]
        O.env_step_random(g, seed, step)
    return out


def golden_no_move_roots():
    return np.concatenate([O.make_state(c["deck"], pawns=c["pawns"], kings=c["kings"], side=c["color"])
                           for c in G["reference_tests"]["no_moves"]])


def action(card_idx, frm, to, king):
    return to | (frm << 5) | (card_idx << 10) | (king << 12)


# ------------------------------------------------------------------ the evaluation spec
def spec_eval(state):
    """eval from the formula, square by square, from the view of the side to move"""
    def value(color):
        v = 0
        temple = 2 if color == 0 else 22
        for n in range(25):
            row, col = divmod(n, 5)
            ctr = 2 - abs(col - 2)
            if (int(state["pawns"][color]) >> (31 - n)) & 1:
                v += 100 + 4 * ((4 - row) if color == 0 else row) + 2 * ctr
            if (int(state["kings"][color]) >> (31 - n)) & 1:
                v += 6 * (6 - (abs(row - temple // 5) + abs(col - temple % 5)))
        return v
    side = int(state["side"])
    return value(side) - value(1 - side)


def test_eval_of_the_start_position_is_zero():
    decks = [[TIGER, DRAGON, FROG, RABBIT, CRAB], [1, 0, 3, 11, 2], [OX, MONKEY, RABBIT, HORSE, DRAGON]]
    for d in decks:
        s = O.new_games(1, deck=d)
        for side in (0, 1):
            s["side"][0] = side
            assert A.evaluate(s)[0] == 0


def rot180(board):
    """q -> 24 - q on reference-layout boards"""
    out = np.zeros_like(board)
    for n in range(25):
        out |= ((board >> np.uint32(31 - n)) & np.uint32(1)) << np.uint32(31 - (24 - n))
    return out


def test_eval_is_invariant_under_the_colour_swap():
    g = midgame_roots(1200, seed=31)
    g = g[g["result"] == 0]
    assert len(g) >= 1000
    sw = g.copy()
    sw["pawns"][:, 0], sw["pawns"][:, 1] = rot180(g["pawns"][:, 1]), rot180(g["pawns"][:, 0])
    sw["kings"][:, 0], sw["kings"][:, 1] = rot180(g["kings"][:, 1]), rot180(g["kings"][:, 0])
    sw["side"] = 1 - g["side"]
    e = A.evaluate(g)
    assert np.array_equal(e, A.evaluate(sw))
    assert np.abs(e).max() < 1000 and len(np.unique(e)) > 20


def test_eval_of_hand_built_positions():
    cases = [  # (pawns [Red, Blue], kings [Red, Blue], side, value by hand)
        # Red: pawns c3 (row 2, col 2) 100 + 8 + 4 and a4 (row 1, col 0) 100 + 12; king c2 (row 3): 6 (6 - 3) = 18 -> 242
        # Blue: pawn e1 (row 4, col 4) 100 + 16; king c5 (row 0) 6 (6 - 4) = 12 -> 128
        ([sq(2, 2) | sq(1, 0), sq(4, 4)], [sq(3, 2), sq(0, 2)], 0, 242 - 128),
        # the same from Blue's view
        ([sq(2, 2) | sq(1, 0), sq(4, 4)], [sq(3, 2), sq(0, 2)], 1, 128 - 242),
        # kings only: Red king b5 (row 0, col 1) next to Blue's temple: 6 (6 - 1) = 30; Blue king e3 (row 2, col 4): 6 (6 - 4) = 12
        ([0, 0], [sq(0, 1), sq(2, 4)], 1, 12 - 30),
    ]
    for pawns, kings, side, want in cases:
        s = O.make_state([TIGER, DRAGON, FROG, RABBIT, CRAB], pawns=pawns, kings=kings, side=side)
        assert spec_eval(s[0]) == want
        assert A.evaluate(s)[0] == want


# ------------------------------------------------------------------ known answers
def test_an_immediate_win_is_found_at_depth_one():
    # Blue to move can take the Red king on d4 (mcts_arena.rs test_best_move_win)
    s = O.make_state([RABBIT, FROG, TIGER, DRAGON, HORSE], kings=[sq(1, 3), 0x20000000], side=1)
    r = A.alphabeta_batch(s, 1)
    assert r["score"][0] == WIN - 1 and r["nodes"][0] == 1
    first = next(int(a) for a in O.gen_moves(s) if O.make_move(s.copy(), a) in (1, 2))
    assert r["best"][0] == first
    # the king reaching the enemy temple is an immediate win too: Tiger moves the Red king from c3 two rows up onto c5
    t = O.make_state([TIGER, FROG, RABBIT, CRAB, HORSE], kings=[sq(2, 2), sq(0, 0)], pawns=[0, 0], side=0)
    r = A.alphabeta_batch(t, 1)
    assert r["score"][0] == WIN - 1 and r["best"][0] == action(0, 12, 2, 1)


def test_depth_two_finds_the_only_move_that_does_not_lose():
    # mcts_arena.rs test_no_way_to_hide_for_blue: the only move that does not lose at once is Rabbit e5-c5
    s = O.make_state([OX, MONKEY, RABBIT, HORSE, DRAGON], kings=[0x00000200, sq(0, 4)], pawns=[sq(0, 3) | sq(1, 4), 0], side=1)
    safe = []
    for a in O.gen_moves(s):
        c = s.copy()
        O.make_move(c, a)
        if A.alphabeta_batch(c, 1)["score"][0] != WIN - 1:
            safe.append(int(a))
    assert safe == [action(2, 4, 2, 1)]
    r = A.alphabeta_batch(s, 2)
    assert r["best"][0] == action(2, 4, 2, 1) and r["score"][0] > -(WIN - 2)
    assert A.minimax_batch(s, 2)["best"][0] == r["best"][0]


def _wins_at_once(state):
    return any(O.make_move(state.copy(), a) in (1, 2) for a in O.gen_moves(state))


def _replies(state):
    moves = O.gen_moves(state)
    if len(moves):
        return [int(a) for a in moves]
    base = 0 if int(state["side"][0]) == 0 else 2
    return [PASS_BIT | (base << 10), PASS_BIT | ((base + 1) << 10)]


def test_a_forced_win_in_two_moves_is_found_at_depth_three():
    roots = midgame_roots(3000, seed=12)
    roots = roots[roots["result"] == 0]
    d1, d3 = A.alphabeta_batch(roots, 1), A.alphabeta_batch(roots, 3)
    hits = np.nonzero((d3["score"] == WIN - 3) & (d1["score"] < WIN - 1))[0]
    assert len(hits) >= 3
    for i in hits[:3]:
        root = roots[i:i + 1]
        # the chosen move does not win at once, but every reply leaves a move that wins at once
        child = root.copy()
        assert O.make_move(child, int(d3["best"][i])) not in (1, 2)
        for reply in _replies(child):
            grand = child.copy()
            assert O.make_move(grand, reply) not in (1, 2)
            assert _wins_at_once(grand)
        assert A.alphabeta_batch(root, 2)["score"][0] < WIN - 3
        m = A.minimax_batch(root, 3)
        assert m["score"][0] == WIN - 3 and m["best"][0] == d3["best"][i]


def test_the_golden_position_without_legal_moves_passes():
    roots = golden_no_move_roots()
    n_moves = [len(O.gen_moves(roots[i:i + 1])) for i in range(len(roots))]
    # state.rs:852-889 has no legal move at all; state.rs:819-850 has none with Rabbit but four with Horse
    assert n_moves == [4, 0]
    for depth in (1, 2, 3, 4):
        r = A.alphabeta_batch(roots, depth)
        assert r["best"][1] & PASS_BIT and (r["best"][1] >> 10) & 3 in (2, 3)  # Blue passes with hand slot 2 or 3
        assert not r["best"][0] & PASS_BIT and int(r["best"][0]) in O.gen_moves(roots[0:1]).tolist()


def test_decided_roots_are_not_searched():
    roots = midgame_roots(480, seed=5)
    done = roots["result"] != 0
    assert done.any()
    r = A.alphabeta_batch(roots, 2)
    assert (r["best"][done] == NONE).all() and (r["score"][done] == 0).all() and (r["nodes"][done] == 0).all()
    assert (r["best"][~done] != NONE).all() and (r["nodes"][~done] > 0).all()


# ------------------------------------------------------------------ the pruning is exact
def test_alphabeta_equals_minimax_and_prunes():
    roots = np.concatenate([midgame_roots(2400, seed=77), golden_no_move_roots()])
    live = roots["result"] == 0
    assert live.sum() >= 2000
    for depth in (1, 2, 3, 4):
        ab, mm = A.alphabeta_batch(roots, depth), A.minimax_batch(roots, depth)
        assert np.array_equal(ab["best"], mm["best"]), depth
        assert np.array_equal(ab["score"], mm["score"]), depth
        assert (ab["nodes"] <= mm["nodes"]).all(), depth
        if depth >= 2:
            assert ab["nodes"].sum() < mm["nodes"].sum(), depth


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def _gpu_search(onb, roots, depth, ctx_size=None, first=0):
    n = ctx_size or len(roots)
    with onb.Context(n, planes=False) as ctx:
        if ctx_size:
            ctx.reset()
        ctx.set_states(roots, first=first)
        r = ctx.alphabeta(depth)
        acts = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,))
    assert np.array_equal(acts, r["best"])  # the chosen actions stay in ONB_BUF_ACTIONS
    return {k: v[first:first + len(roots)] for k, v in r.items()}


@pytest.mark.gpu
def test_gpu_equals_the_oracle_bit_exact(onb):
    roots = np.concatenate([midgame_roots(4096, seed=2024), golden_no_move_roots()])
    for depth in range(1, 7):
        got, want = _gpu_search(onb, roots, depth), A.alphabeta_batch(roots, depth)
        for k in ("best", "score", "nodes"):
            assert np.array_equal(got[k], want[k]), (depth, k, np.nonzero(got[k] != want[k])[0][:5])
    deep = midgame_roots(256, seed=8)
    got, want = _gpu_search(onb, deep, 8), A.alphabeta_batch(deep, 8)
    for k in ("best", "score", "nodes"):
        assert np.array_equal(got[k], want[k]), (8, k)
    assert (got["best"][deep["result"] == 0] != NONE).all()


@pytest.mark.gpu
def test_results_do_not_depend_on_the_batch(onb):
    roots = midgame_roots(1000, seed=66)
    base = _gpu_search(onb, roots, 4)
    other = _gpu_search(onb, roots, 4, ctx_size=2500, first=777)  # a larger context, other games around, another offset
    for k in ("best", "score", "nodes"):
        assert np.array_equal(base[k], other[k]), k
    for lo, hi in ((0, 1), (13, 40), (500, 1000)):
        part = _gpu_search(onb, roots[lo:hi], 4)
        for k in ("best", "score", "nodes"):
            assert np.array_equal(part[k], base[k][lo:hi]), (lo, k)


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    """onb_fight with the alpha-beta agent (it searches only the games in which it is to move: the subset path) against
    selfplay.fight driven with Context.alphabeta over all games: identical per-game results, final states and W/L/D."""
    n, sims = 48, 24
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=17, mcts_max_sims=120, planes=False) as ctx:
        def py_ab(depth):
            return lambda cx: cx.alphabeta(depth, to_host=False)

        def py_puct(cx):
            cx.search_device(2.0, sims, evaluator=onb.EVAL_UNIFORM)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        def py_uct(cx):
            cx.uct_search(2.0 ** 0.5, 5, 120, to_host=False)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        for name, depth, py_b, nat_b, cap in (
                ("ab-vs-random", 3, None, ctx.agent_random(), 150),
                ("ab-vs-uct", 2, py_uct, ctx.agent_uct(120), 150),
                ("ab-vs-puct", 4, py_puct, ctx.agent_puct(sims, 2.0), 150),
                ("ply-cap", 3, None, ctx.agent_random(), 3)):
            counter = {"i": 0}

            def py_random(cx):
                cx.choose_random(counter["i"], policy=onb.POLICY_AGENT)
                counter["i"] += 1

            ctx.reset()
            want = onb.fight(ctx, py_ab(depth), py_b or py_random, a_is_red, max_plies=cap)
            want_states = ctx.get_states().tobytes()
            want_results = ctx.last_fight_results.copy()
            ctx.reset()
            a, b, d, results = ctx.fight_native(ctx.agent_alphabeta(depth), nat_b, a_is_red, max_plies=cap)
            assert (a, b, d) == want, name
            assert ctx.get_states().tobytes() == want_states, name
            assert np.array_equal(results, want_results), name
            assert a + b + d == n
            if cap == 3:
                assert d > 0
            assert 0 < ctx.last_fight_moves_chosen <= n * ctx.last_fight_plies
            # the agents swap the colours: the same games with alpha-beta as agent B
            ctx.reset()
            b2, a2, d2, _ = ctx.fight_native(nat_b, ctx.agent_alphabeta(depth), ~a_is_red, max_plies=cap)
            assert (a2, b2, d2) == (a, b, d), name
            assert ctx.get_states().tobytes() == want_states, name


@pytest.mark.gpu
def test_moves_chosen_counts_the_searched_games(onb):
    n = 64
    with onb.Context(n, seed=3, planes=False) as ctx:
        ctx.reset()
        ctx.fight_native(ctx.agent_alphabeta(2), ctx.agent_alphabeta(1), np.ones(n, bool), max_plies=150)
        plies, chosen = ctx.last_fight_plies, ctx.last_fight_moves_chosen
        # replay with the public call: count the undecided games at every ply
        ctx.reset()
        states = ctx.get_states()
        live_total = 0
        for ply in range(plies):
            live = states["result"] == 0
            live_total += int(live.sum())
            red = states["side"] == 0
            ctx.alphabeta(2, to_host=False)
            act2 = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)).copy()
            ctx.alphabeta(1, to_host=False)
            act1 = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)).copy()
            ctx.step(np.where(red, act2, act1))
            states = ctx.get_states()
        assert chosen == live_total


@pytest.mark.gpu
def test_depth_three_beats_random(onb):
    n = 256
    with onb.Context(n, seed=99, planes=False) as ctx:
        ctx.reset()
        a, b, d, _ = ctx.fight_native(ctx.agent_alphabeta(3), ctx.agent_random(), (np.arange(n) % 2) == 0)
    rate = a / n
    print("alpha-beta depth 3 vs Random: %d wins, %d losses, %d draws (%.1f %%)" % (a, b, d, 100 * rate))
    assert rate >= 0.8


@pytest.mark.gpu
def test_errors_and_a_context_without_search_pools(onb):
    with onb.Context(16, planes=False) as ctx:  # mcts_max_sims = 0
        ctx.reset()
        for depth in (0, 9):
            with pytest.raises(onb.OnbError) as e:
                ctx.alphabeta(depth)
            assert e.value.code == -1
            with pytest.raises(onb.OnbError) as e:
                ctx.fight_native(ctx.agent_alphabeta(depth), ctx.agent_random(), np.ones(16, bool))
            assert e.value.code == -1
        a, b, d, _ = ctx.fight_native(ctx.agent_alphabeta(2), ctx.agent_random(), (np.arange(16) % 2) == 0)
        assert a + b + d == 16 and a > b
        with pytest.raises(onb.OnbError):  # a searching agent still needs the pools
            ctx.fight_native(ctx.agent_alphabeta(2), ctx.agent_puct(8), np.ones(16, bool))


@pytest.mark.gpu
def test_cpp_mirror_agent_equals_context_alphabeta(onb, tmp_path):
    exe = str(tmp_path / "test_alphabeta_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "test_alphabeta_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(ROOT, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(ROOT, "onitama_alphazero_b200")])
    roots = midgame_roots(200, seed=41)
    roots = roots[(roots["result"] == 0)]
    roots = roots[[len(O.gen_moves(roots[i:i + 1])) > 0 for i in range(len(roots))]][:40]
    depth = 3
    lines = ["%d %d" % (len(roots), depth)]
    for r in roots:
        lines.append(" ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"])))
    p = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = np.array([[int(float(x)) for x in ln.split()] for ln in p.stdout.strip().splitlines()[:len(roots)]])
    want = _gpu_search(onb, roots, depth)
    assert np.array_equal(got[:, 0], want["best"].astype(np.int64))
    assert np.array_equal(got[:, 1], want["score"].astype(np.int64))
