"""Tablebase leaves (DESIGN.md §5i) on the CPU oracle (tests/tb_search_oracle.cpp) with a table the tablebase oracle solves at one
pawn: the per-leaf reward against a pure-Python restatement, roots of another card set against the PUCT oracle bit for bit, and in
every tree every node below the root that the table holds unexpanded with W = N r."""
import numpy as np
import pytest

import oracle_lib as O
import tablebase_oracle as TBO
import tb_search_oracle as TS

CARDS = [0, 1, 2, 3, 11]
NONE = TBO.NONE
RED_TEMPLE_KING, BLUE_TEMPLE_KING = 1 << (31 - 2), 1 << (31 - 22)  # a king on the enemy temple: a decided position


@pytest.fixture(scope="module")
def table():
    return TBO.solve(CARDS, 1)[0]


def py_reward(v, depth, leaf_color):
    """the rule restated: a decided leaf's reward with the table's winner as the winner, from the view of the leaf's parent (the
    root's own colour at depth 0)"""
    if v == 0:
        return 0.0
    winner = leaf_color if v > 0 else 1 - leaf_color
    reward_color = leaf_color if depth == 0 else 1 - leaf_color
    return 1.0 if winner == reward_color else -1.0


def undecided(st):
    return (st["kings"][:, 0] != RED_TEMPLE_KING) & (st["kings"][:, 1] != BLUE_TEMPLE_KING)


def positions(table, rng, n, classes):
    """n undecided states of the set from the given classes (p, q); classes outside the table give roots above it"""
    out = []
    for p, q in classes:
        e = TBO.entries(p, q)
        st = TBO_states(5 * p + q, rng.integers(0, e, 4 * n // len(classes)))
        out.append(st[undecided(st)][:n // len(classes)])
    return np.ascontiguousarray(np.concatenate(out))


def TBO_states(cls, idx):
    import onitama_alphazero_b200 as onb  # onb_tb_state is pure host code
    return onb.tb_states(CARDS, cls, idx)


def node_states(root, tree):
    """the position of every node of a dumped tree, replayed from the root along the actions"""
    st = np.repeat(np.asarray(root).reshape(1), len(tree["parent"]), axis=0)
    for i in range(1, len(st)):
        g = st[tree["parent"][i]:tree["parent"][i] + 1].copy()
        O.make_move(g, int(tree["action"][i]))
        st[i] = g[0]
    return st


def check_tree(root, tree, table):
    """every node below the root that the table holds is unexpanded with W = N r; returns the number of such nodes"""
    st = node_states(root, tree)
    v = TBO.probe(CARDS, 1, table, st).astype(np.int32)
    depth = np.zeros(len(st), int)
    for i in range(1, len(st)):
        depth[i] = depth[tree["parent"][i]] + 1
    hits = 0
    for i in range(1, len(st)):
        if v[i] == NONE or tree["visits"][i] == 0:
            continue
        hits += 1
        r = py_reward(v[i], depth[i], int(st["side"][i]))
        assert tree["n_child"][i] == 0 and not (tree["flags"][i] & 1), i
        assert tree["reward"][i] == tree["visits"][i] * r, (i, tree["reward"][i], tree["visits"][i], r)
    return hits


def test_reward_rule_matches_the_restatement():
    for v in (1, 5, 33, -2, -34, 0):
        for depth in (0, 1, 2):
            for color in (0, 1):
                assert TS.reward(v, depth, color) == py_reward(v, depth, color), (v, depth, color)


@pytest.mark.parametrize("leaves", [1, 4])
def test_hand_built_leaves_at_depth_0_1_2(table, leaves):
    rng = np.random.default_rng(5)
    picks = []  # wins, losses and draws of every class
    for (p, q), t in sorted(table.items()):
        tv = t.astype(np.int32)
        for pool in (np.nonzero((t != NONE) & (tv > 0))[0], np.nonzero((t != NONE) & (tv < 0))[0], np.nonzero(tv == 0)[0]):
            if len(pool):
                picks.append(TBO_states(5 * p + q, rng.choice(pool, 8)))
    roots = np.ascontiguousarray(np.concatenate(picks))
    v = TBO.probe(CARDS, 1, table, roots).astype(np.int32)
    assert (v != NONE).all() and (v > 0).any() and (v < 0).any()
    assert (v == 0).any() == any((t == 0).any() for t in table.values())  # draws, where the set has any at one pawn
    # depth 0: one simulation backs the table's value of the root up into the root, from the root mover's view
    one = TS.search(roots, 2.0, 1, CARDS, 1, table, leaves=leaves)
    assert np.array_equal(one["root_q"], np.sign(v).astype(np.float64))
    assert (one["n_nodes"] > 1).all()  # the root is expanded all the same
    # depth 1: the children of an in-table root are leaves of the table (or decided); depth 2 and below: the two-pawn roots below
    for sims in (2, 3, 20):
        for t in range(0, len(roots), 7):
            tree = TS.search(roots[t:t + 1], 2.0, sims, CARDS, 1, table, leaves=leaves, dump_tree=0)["tree"]
            check_tree(roots[t], tree, table)
            assert (tree["n_child"][1:] == 0).all()  # below an in-table root nothing is expanded


@pytest.mark.parametrize("evaluator", [0, 1])
def test_other_sets_equal_the_puct_oracle(table, evaluator):
    from test_gpu_gumbel import _undecided
    roots = _undecided(256, 21)
    roots = roots[np.array([sorted(r["cards"]) != sorted(CARDS) for r in roots])]
    sims = 60
    want = O.mcts_search_batch(roots, 2.0, sims, evaluator=evaluator, threads=8)
    got = TS.search(roots, 2.0, sims, CARDS, 1, table, evaluator=evaluator)
    for k in ("best", "child_visits", "n_nodes", "root_q", "pi"):
        assert np.array_equal(got[k], want[k]), k
    assert np.array_equal(got["pi"].view(np.uint32), want["pi"].view(np.uint32))


@pytest.mark.parametrize("leaves", [1, 2, 8])
def test_table_nodes_are_unexpanded_with_exact_values(table, leaves):
    rng = np.random.default_rng(9 + leaves)
    # two pawns: one above the one-pawn table, so the first captures lead into it
    roots = positions(table, rng, 48, [(2, 0), (1, 1), (0, 2)])
    hits = 0
    for t in range(len(roots)):
        tree = TS.search(roots[t:t + 1], 2.0, 200, CARDS, 1, table, leaves=leaves, evaluator=1, dump_tree=0)["tree"]
        assert tree["visits"][0] == 200
        hits += check_tree(roots[t], tree, table)
    assert hits > 100
