"""The tree-reuse oracle (tests/reuse_oracle.cpp) on the CPU: its reroot is the arena-order filter, a search without a match is the
plain oracle search, and a visit target at or below the kept visits runs no playout."""
import numpy as np

import oracle_lib as O
import reuse_oracle as R


def _roots(n, seed):
    """undecided positions after p random plies (p = game id mod 12)"""
    g = O.new_games(n, seed=seed)
    for step in range(12):
        live = (np.arange(n) % 12) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return g[g["result"] == 0]


def _played(states, actions):
    out = states.copy()
    for i in range(len(out)):
        O.make_move(out[i:i + 1], int(actions[i]))
    return out


def test_reroot_is_the_arena_order_filter():
    roots = _roots(48, 3)
    n = len(roots)
    rs = R.ReuseSet(n)
    first = rs.search(roots, 2.0, 200, evaluator=1)
    before = [rs.dump(i) for i in range(n)]
    after_move = _played(roots, first["best"])
    again = rs.search(after_move, 2.0, 0, evaluator=1)   # target 0: reroot only
    checked = 0
    for i in range(n):
        got = rs.dump(i)
        t = before[i]
        if after_move["result"][i] != 0:
            assert again["kept"][i] == 0 and len(got["visits"]) == 1
            continue
        kids = t["first_child"][0] + np.arange(t["n_child"][0])
        keep = int(kids[t["action"][kids] == first["best"][i]][0])
        want = R.filter_tree(t, keep)
        assert again["kept"][i] == 1 and again["sims_run"][i] == 0
        for k in want:
            assert np.array_equal(got[k], want[k]), (i, k)
        assert got["visits"][0] == t["visits"][keep] and got["parent"][0] == -1
        checked += 1
    assert checked >= n // 2


def test_no_match_is_the_plain_search():
    roots = _roots(32, 5)
    n = len(roots)
    rs = R.ReuseSet(n)
    got = rs.search(roots, 2.0, 120, evaluator=1)
    assert not got["kept"].any()
    for i in range(n):
        want = O.mcts_search(roots[i:i + 1], 2.0, 120, evaluator=1)
        assert got["best"][i] == want["best"] and np.array_equal(got["pi"][i], want["pi"])
        assert got["root_visits"][i] == want["root_visits"] and got["root_q"][i] == want["root_q"]
        assert got["n_nodes"][i] == want["n_nodes"]
    # positions that are not a child of the remembered roots (the same roots again, a different game) start fresh too
    other = _roots(64, 99)[:n]
    again = rs.search(other, 2.0, 120, evaluator=1)
    assert not again["kept"].any()
    for i in range(0, n, 4):
        want = O.mcts_search(other[i:i + 1], 2.0, 120, evaluator=1)
        assert again["best"][i] == want["best"] and again["n_nodes"][i] == want["n_nodes"]


def test_target_at_or_below_the_kept_visits_runs_nothing():
    roots = _roots(24, 7)
    n = len(roots)
    rs = R.ReuseSet(n)
    first = rs.search(roots, 2.0, 400, evaluator=0)
    moved = _played(roots, first["best"])
    probe = rs.search(moved, 2.0, 0)
    kept_n = probe["root_visits"].copy()
    live = probe["kept"] == 1
    assert live.sum() >= n // 2 and (kept_n[live] > 0).all()
    target = int(kept_n[live].min())
    # the remembered roots are the moved positions now: a position is not a child of itself, so every tree starts over
    res = rs.search(moved, 2.0, target)
    assert not res["kept"].any() and (res["sims_run"] == target).all()
    rs2 = R.ReuseSet(n)
    rs2.search(roots, 2.0, 400, evaluator=0)
    res2 = rs2.search(moved, 2.0, target)
    assert (res2["sims_run"][live] == 0).all()
    assert np.array_equal(res2["root_visits"][live], kept_n[live])
    # the whole-game driver: reuse runs fewer simulations for the same games
    starts = O.new_games(6, seed=11)
    a = R.play_games(starts, 2.0, 64, max_plies=20, reuse=True)
    b = R.play_games(starts, 2.0, 64, max_plies=20, reuse=False)
    assert (a["sims"] <= b["sims"]).all() and a["sims"].sum() < b["sims"].sum()
    assert (a["plies"] > 0).all()
