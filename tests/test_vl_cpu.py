"""Leaf parallelism with virtual loss (onb_mcts_set_virtual_loss, DESIGN.md §5h) on the CPU: the oracle's rounds of one descent are
the oracle's PUCT search bit for bit, its per-node choice equals a pure-Python restatement of the definition, and a search of rounds
keeps the visit, node and round counts the definition fixes."""
import math
import struct

import numpy as np
import pytest

import oracle_lib as O
import vl_oracle as VO
from test_gpu_gumbel import _undecided


def _total_key(x):
    b = struct.unpack("<q", struct.pack("<d", x))[0]
    return b ^ ((b >> 63) & 0x7FFFFFFFFFFFFFFF)


def _python_choice(off, P, N, W, V, np_, c, vl):
    """include/onb.h's choice on Python floats (IEEE f64, correctly rounded, no FMA): the LAST child maximising
    q' + (c P) (sqrt(Np') / (N' + 1))"""
    out = []
    for i in range(len(np_)):
        best, bkey = 0, None
        for a in range(off[i], off[i + 1]):
            n = int(N[a]) + int(V[a])
            w = float(W[a]) - vl * float(V[a]) if V[a] else float(W[a])
            q = w / n if n else 0.0
            u = q + c * float(P[a]) * (math.sqrt(float(np_[i])) / float(n + 1))
            k = _total_key(u)
            if bkey is None or k >= bkey:
                best, bkey = a - off[i], k
        out.append(best)
    return np.array(out, np.int64)


def _nodes(n, seed):
    """n random nodes: 1 .. 40 children with 33 .. 36 common, ties in P / W / N, unvisited children, no pending descents or many"""
    rng = np.random.default_rng(seed)
    k = np.where(rng.random(n) < 0.3, rng.integers(33, 37, n), rng.integers(1, 41, n))
    off = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)
    tot = int(off[-1])
    node = np.repeat(np.arange(n), k)
    kind = rng.integers(0, 5, n)[node]
    P = rng.random(tot)
    P = np.where(kind == 1, rng.integers(1, 4, tot) / 8.0, P)  # coarse: ties
    P = np.where(kind == 2, 1.0 / 50.0, P)
    N = (rng.integers(0, 20, tot) * (rng.random(tot) < 0.7)).astype(np.uint32)
    N = np.where(kind == 3, 0, N).astype(np.uint32)  # every child unvisited
    W = np.where(kind == 1, rng.integers(-3, 4, tot).astype(np.float64), rng.random(tot) * 2 - 1) * np.maximum(N, 1)
    W = np.where(N > 0, W.astype(np.float32).astype(np.float64), 0.0)
    V = (rng.integers(0, 32, tot) * (rng.random(tot) < 0.4)).astype(np.uint32)
    V = np.where(kind == 4, 0, V).astype(np.uint32)  # no pending descent: the PUCT choice
    np_ = (np.add.reduceat(N, off[:-1]) + rng.integers(0, 32, n)).astype(np.uint32)
    return off, P, N, W, V, np_


@pytest.mark.parametrize("vl", [0.0, 1.0, 3.0, 0.375])
@pytest.mark.parametrize("c", [2.0, 0.25])
def test_choice_equals_the_python_restatement(vl, c):
    off, P, N, W, V, np_ = _nodes(3000, int(vl * 8 + c * 100))
    got = VO.choice(off, P, N, W, V, np_, c, vl)
    assert np.array_equal(got, _python_choice(off, P, N, W, V, np_, c, vl))


def test_no_pending_descent_is_the_puct_choice():
    # v = 0 everywhere: the choice of the oracle's MctsArena::select (q = winrate, the last maximal child)
    off, P, N, W, _, np_ = _nodes(2000, 5)
    V = np.zeros_like(N)
    got = VO.choice(off, P, N, W, V, np_, 2.0, 1.0)
    assert np.array_equal(got, VO.choice(off, P, N, W, V, np_, 2.0, 0.0))
    assert np.array_equal(got, _python_choice(off, P, N, W, V, np_, 2.0, 1.0))


@pytest.mark.parametrize("evaluator", [0, 1])
@pytest.mark.parametrize("sims", [1, 2, 37, 160])
def test_one_descent_per_round_is_the_puct_search(evaluator, sims):
    roots = _undecided(300, 60 + sims)
    want = O.mcts_search_batch(roots, 2.0, sims, evaluator=evaluator, threads=8)
    for vl in (0.0, 1.0):
        got = VO.search(roots, 2.0, sims, 1, vl, evaluator=evaluator)
        for k in ("best", "child_visits", "n_nodes", "root_q", "pi"):
            assert np.array_equal(got[k], want[k]), (vl, k)
        assert (got["rounds"] == sims).all()


@pytest.mark.parametrize("leaves,vl", [(2, 1.0), (8, 0.0), (8, 1.0), (32, 3.0)])
@pytest.mark.parametrize("sims", [1, 2, 33, 200])
def test_visit_node_and_round_counts(leaves, vl, sims):
    roots = _undecided(200, 7 + sims)
    got = VO.search(roots, 2.0, sims, leaves, vl, evaluator=1)
    assert (got["root_visits"] == sims).all()
    assert (got["n_nodes"] <= 1 + 40 * sims).all()
    assert (got["rounds"] == 1 + -(-(sims - 1) // leaves)).all()
    assert (got["child_visits"].sum(axis=1) == sims - 1).all()  # every descent after round 0 enters a root child


@pytest.mark.parametrize("leaves", [2, 8, 16])
def test_round_one_spreads_over_distinct_root_children(leaves):
    # uniform priors, vl = 1, value 0: a pending descent makes q' = -1, which outweighs the exploration term c P sqrt(Np') / 2 < 1
    # of every child (c_puct sqrt(1 + K) < 2), so round 1's K descents enter K different root children
    roots = _undecided(300, 91)
    got = VO.search(roots, 0.3, 1 + leaves, leaves, 1.0, evaluator=0)
    k = (O.mcts_search_batch(roots, 2.0, 1, evaluator=0)["n_nodes"] - 1)
    wide = k >= leaves
    assert wide.sum() > 50
    cv = got["child_visits"][wide]
    assert ((cv == 1).sum(axis=1) == leaves).all() and (cv.max(axis=1) == 1).all()
