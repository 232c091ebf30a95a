"""The MCTS solver (onb_mcts_set_solver, DESIGN.md §5k) on the CPU oracle (tests/solver_oracle.cpp): every proof in the trees of roots
inside a table the tablebase oracle solves agrees with the table's sign and no drawn position is proven; with the switch off the
oracle is the PUCT oracle bit for bit; the propagation rule on hand-built trees; and what a proof does to the search's choice."""
import numpy as np
import pytest

import oracle_lib as O
import solver_oracle as SO
import tablebase_oracle as TBO
from test_tb_search_cpu import CARDS, NONE, TBO_states, node_states, undecided

WIN, LOSS = SO.WIN, SO.LOSS


@pytest.fixture(scope="module")
def table():
    return TBO.solve(CARDS, 1)[0]


def table_roots(table, n, seed, sign=None):
    """n undecided roots of the table (every class), of the given sign of value when `sign` is set"""
    rng = np.random.default_rng(seed)
    picks = []
    for (p, q), t in sorted(table.items()):
        tv = t.astype(np.int32)
        ok = t != NONE if sign is None else (t != NONE) & (np.sign(tv) == sign)
        pool = np.nonzero(ok)[0]
        if len(pool):
            st = TBO_states(5 * p + q, rng.choice(pool, 4 * n))
            picks.append(st[undecided(st)])
    st = np.concatenate(picks)
    return np.ascontiguousarray(st[rng.permutation(len(st))[:n]])


def check_proofs(root, tree, table, max_pawns=1):
    """every WIN / LOSS flag agrees with the sign of the table's value of the node's position; returns (proven nodes, drawn nodes)"""
    st = node_states(root, tree)
    v = TBO.probe(CARDS, max_pawns, table, st).astype(np.int32)
    fl = tree["flags"]
    assert not ((fl & WIN) & (fl & LOSS)).any()
    proven = drawn = 0
    for i in range(len(st)):
        if not fl[i] & (WIN | LOSS):
            drawn += int(v[i] == 0)
            continue
        proven += 1
        if v[i] == NONE:  # a decided position: only a terminal child, won by the side that moved into it
            assert fl[i] & 2 and fl[i] & WIN, i
        elif fl[i] & WIN:  # the side that moved into the node wins: the side to move there loses
            assert v[i] < 0, (i, v[i])
        else:
            assert v[i] > 0, (i, v[i])
    return proven, drawn


@pytest.mark.parametrize("sims", [1, 2, 33, 200])
@pytest.mark.parametrize("evaluator", [0, 1])
def test_proofs_agree_with_the_table(table, evaluator, sims):
    roots = table_roots(table, 48, 3 + sims + evaluator)
    proven = 0
    for t in range(len(roots)):
        r = SO.search(roots[t:t + 1], 2.0, sims, evaluator=evaluator, dump_tree=0)
        p, _ = check_proofs(roots[t], r["tree"], table)
        proven += p
        v = int(TBO.probe(CARDS, 1, table, roots[t:t + 1])[0])
        assert r["proof"][0] == 0 or np.sign(v) == r["proof"][0], (t, v, r["proof"][0])
    assert sims == 1 or proven > 0


def test_no_draw_is_proven():
    """the set's one-pawn table has no draw; the two-pawn table has (class (1, 1)): drawn roots, whose trees hold drawn positions"""
    table2 = TBO.solve(CARDS, 2)[0]
    roots = table_roots(table2, 32, 11, sign=0)
    assert len(roots) == 32
    drawn = 0
    for t in range(len(roots)):
        r = SO.search(roots[t:t + 1], 2.0, 300, evaluator=1, dump_tree=0)
        _, d = check_proofs(roots[t], r["tree"], table2, max_pawns=2)
        drawn += d
        assert r["proof"][0] == 0
    assert drawn > 100


@pytest.mark.parametrize("evaluator", [0, 1])
def test_solver_off_equals_the_puct_oracle(evaluator):
    from test_gpu_gumbel import _undecided
    roots = _undecided(256, 31)
    for sims in (1, 33, 120):
        want = O.mcts_search_batch(roots, 2.0, sims, evaluator=evaluator, threads=8)
        got = SO.search(roots, 2.0, sims, solver=False, evaluator=evaluator)
        for k in ("best", "child_visits", "n_nodes", "root_q"):
            assert np.array_equal(got[k], want[k]), k
        assert np.array_equal(got["pi"].view(np.uint32), want["pi"].view(np.uint32))
        assert (got["proof"] == 0).all()
    # the trees too, flags included
    for t in range(0, 256, 37):
        want = O.mcts_search(roots[t:t + 1], 2.0, 60, evaluator=evaluator, dump=True)["tree"]
        got = SO.search(roots[t:t + 1], 2.0, 60, solver=False, evaluator=evaluator, dump_tree=0)["tree"]
        for k in want:
            assert np.array_equal(got[k], want[k]), (t, k)


def _tree(parent):
    """a hand-built tree from its parent list (children contiguous, in index order)"""
    m = len(parent)
    fc = np.zeros(m, np.uint32)
    nc = np.zeros(m, np.uint32)
    for i in range(1, m):
        p = parent[i]
        if nc[p] == 0:
            fc[p] = i
        nc[p] += 1
    return np.array(parent, np.int32), fc, nc


def test_propagation_rules_on_hand_built_trees():
    # root 0 -> {1, 2}; 1 -> {3, 4}; 2 -> {5}; 3 -> {6, 7}
    par, fc, nc = _tree([-1, 0, 0, 1, 1, 2, 3, 3])
    # a WIN makes its parent LOSS; the grandparent becomes WIN only when every child is LOSS
    pr = np.zeros(8, np.uint8)
    pr[6] = WIN
    got = SO.propagate(par, fc, nc, pr, 6)
    assert got[3] == LOSS and got[1] == 0 and got[0] == 0  # 4 is unproven: 1 stays open
    pr = got.copy()
    pr[4] = LOSS
    got = SO.propagate(par, fc, nc, pr, 4)
    assert got[1] == WIN and got[0] == LOSS  # 1's children 3, 4 both LOSS; a WIN child makes the root LOSS
    # LOSS of a single child proves the parent WIN; it goes up as long as the levels change
    pr = np.zeros(8, np.uint8)
    pr[5] = LOSS
    got = SO.propagate(par, fc, nc, pr, 5)
    assert got[2] == WIN and got[0] == LOSS
    # it stops at the first level that does not change
    pr = np.zeros(8, np.uint8)
    pr[7] = LOSS
    got = SO.propagate(par, fc, nc, pr, 7)
    assert (got == pr).all()
    # an already proven parent is left as it is
    pr = np.zeros(8, np.uint8)
    pr[3] = WIN
    pr[6] = WIN
    got = SO.propagate(par, fc, nc, pr, 6)
    assert got[3] == WIN and got[1] == 0


def test_immediate_wins_are_proven_and_played():
    """roots with a move that wins at once: proof +1 after one simulation and a winning best move"""
    from test_gpu_gumbel import _undecided
    roots = _undecided(2048, 17)
    wins = []
    for r in roots:
        g = r.reshape(1).copy()
        moves = O.gen_moves(g)
        w = set()
        for a in moves:
            h = g.copy()
            O.make_move(h, int(a))
            if h["result"][0] != 0:
                w.add(int(a))
        wins.append(w)
    has = np.array([len(w) > 0 for w in wins])
    assert has.sum() > 10
    for sims in (1, 5):
        r = SO.search(roots, 2.0, sims)
        assert (r["proof"][has] == 1).all()
        assert all(int(b) in w for b, w, h in zip(r["best"], wins, has) if h)
