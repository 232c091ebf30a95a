"""The endgame tablebase (onb_tb_*, DESIGN.md §5g) without a GPU: the index of the C ABI's host helpers against a pure-Python
restatement, and the oracle (tests/tablebase_oracle.cpp) on hand-built cases, on its own consistency and against the alpha-beta
oracle."""
from math import comb

import numpy as np
import pytest

import alphabeta_oracle as A
import oracle_lib as O
import tablebase_oracle as T

CARDS = [0, 1, 2, 3, 11]  # Tiger, Dragon, Frog, Rabbit, Horse: the card set of SURVEY App. A
NONE = T.NONE
SIZES = {(0, 0): 36000, (1, 0): 828000, (0, 1): 828000, (2, 0): 9108000, (0, 2): 9108000, (1, 1): 18216000, (3, 0): 63756000,
         (0, 3): 63756000, (2, 1): 191268000, (1, 2): 191268000, (4, 0): 318780000, (0, 4): 318780000, (3, 1): 1275120000,
         (1, 3): 1275120000, (2, 2): 1912680000}


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def squares(board):
    """reference layout: square n is bit 31 - n"""
    return [n for n in range(25) if (int(board) >> (31 - n)) & 1]


def py_index(cards, s):
    """the index as include/onb.h states it, restated in Python"""
    srt = sorted(cards)
    j = srt.index(int(s["cards"][4]))
    rem = [c for c in srt if c != srt[j]]
    a, b = sorted(rem.index(int(s["cards"][k])) for k in (0, 1))
    cfg = 6 * j + comb(a, 1) + comb(b, 2)
    kr, kb = squares(s["kings"][0])[0], squares(s["kings"][1])[0]
    pr, pb = squares(s["pawns"][0]), squares(s["pawns"][1])
    p, q = len(pr), len(pb)

    def rank(sq, occ):
        return sum(comb(x - sum(1 for o in occ if o < x), i + 1) for i, x in enumerate(sorted(sq)))

    idx = ((cfg * 2 + int(s["side"])) * 600 + 24 * kr + kb - (kb > kr)) * comb(23, p) * comb(23 - p, q)
    idx += rank(pr, [kr, kb]) * comb(23 - p, q) + rank(pb, [kr, kb] + pr)
    return 5 * p + q, idx


def random_states(rng, n, cards, max_pawns=4):
    out = np.zeros(n, dtype=O.STATE_DTYPE)
    for i in range(n):
        sq = rng.permutation(25)
        p = int(rng.integers(0, max_pawns + 1))
        q = int(rng.integers(0, max_pawns - p + 1))
        out[i]["kings"] = [1 << (31 - int(sq[0])), 1 << (31 - int(sq[1]))]
        out[i]["pawns"] = [sum(1 << (31 - int(x)) for x in sq[2:2 + p]), sum(1 << (31 - int(x)) for x in sq[2 + p:2 + p + q])]
        out[i]["cards"] = rng.permutation(cards)
        out[i]["side"] = int(rng.integers(0, 2))
    return out


def test_class_sizes(onb):
    for (p, q), e in SIZES.items():
        assert T.entries(p, q) == e == 36000 * comb(23, p) * comb(23 - p, q)
    assert sum(e for (p, q), e in SIZES.items() if p + q <= 1) == 1692000
    assert sum(e for (p, q), e in SIZES.items() if p + q <= 2) == 38124000
    assert sum(e for (p, q), e in SIZES.items() if p + q <= 3) == 548172000
    assert sum(SIZES.values()) == 5648652000


def test_index_and_state_are_inverse_on_every_entry_up_to_two_pawns(onb):
    for (p, q), e in SIZES.items():
        if p + q > 2:
            continue
        for lo in range(0, e, 1 << 22):
            idx = np.arange(lo, min(e, lo + (1 << 22)), dtype=np.int64)
            st = onb.tb_states(CARDS, 5 * p + q, idx)
            cls, back = onb.tb_index(CARDS, st)
            assert (cls == 5 * p + q).all() and np.array_equal(back, idx), (p, q, lo)
            assert (st["result"] == 0).all() and (st["flags"] == 0).all()
            assert (st["cards"][:, 0] < st["cards"][:, 1]).all() and (st["cards"][:, 2] < st["cards"][:, 3]).all()
    with pytest.raises(onb.OnbError):
        onb.tb_states(CARDS, 0, [36000])


def test_index_agrees_with_the_python_restatement(onb):
    rng = np.random.default_rng(5)
    for cards in (CARDS, [15, 4, 9, 7, 12], [5, 6, 13, 14, 10]):
        st = random_states(rng, 3000, cards)
        cls, idx = onb.tb_index(cards, st)
        for i in range(len(st)):
            assert (cls[i], idx[i]) == py_index(cards, st[i]), i
        # the order within a hand is not part of the position
        sw = st.copy()
        sw["cards"][:, [0, 1, 2, 3]] = sw["cards"][:, [1, 0, 3, 2]]
        assert np.array_equal(onb.tb_index(cards, sw)[1], idx)
        assert (idx < np.array([SIZES[(c // 5, c % 5)] for c in cls])).all()
    # not positions of the classes: another card set, a missing king, overlapping pieces, five pawns
    bad = random_states(rng, 4, CARDS)
    bad[0]["cards"][0] = 9
    bad[1]["kings"][0] = 0
    bad[2]["pawns"][0] = bad[2]["kings"][1]
    free = [n for n in range(25) if n not in squares(bad[3]["kings"][0]) + squares(bad[3]["kings"][1])]
    bad[3]["pawns"] = [sum(1 << (31 - n) for n in free[:3]), sum(1 << (31 - n) for n in free[3:5])]
    cls, idx = onb.tb_index(CARDS, bad)
    assert (cls == -1).all() and (idx == -1).all()
    with pytest.raises(onb.OnbError):
        onb.tb_index([0, 1, 2, 3, 3], bad)


# ------------------------------------------------------------------ the oracle
def sq(row, col):
    return 1 << (31 - (row * 5 + col))


def test_oracle_hand_built_cases(onb):
    tables, info = T.solve(CARDS, 1)
    # Red's Tiger steps two rows up from c2 onto the blue king on c4: a king capture
    s = O.make_state([0, 1, 2, 3, 11], kings=[sq(3, 2), sq(1, 2)], pawns=[0, 0], side=0)
    assert T.probe(CARDS, 1, tables, s)[0] == 1
    # every position of class (0, 0) whose every move allows an immediate win (and which has none itself) is -2, and only those
    allst = onb.tb_states(CARDS, 0, np.arange(36000))
    vals = T.probe(CARDS, 1, tables, allst)
    n_minus2 = 0
    for i in range(0, 36000, 7):
        g = allst[i:i + 1]
        if vals[i] == NONE or vals[i] == 1:
            continue
        replies_win = True
        for a in O.gen_moves(g):
            c = g.copy()
            O.make_move(c, int(a))
            assert c["result"][0] == 0
            if not any(_wins(c, int(b)) for b in O.gen_moves(c)):
                replies_win = False
                break
        assert replies_win == (vals[i] == -2), i
        n_minus2 += replies_win
    assert n_minus2 > 10


def _wins(g, a):
    c = g.copy()
    O.make_move(c, a)
    return c["result"][0] != 0


def test_oracle_solves_a_position_without_legal_moves_through_its_pass_children(onb):
    """No position with at most three pawns of the mover lacks a legal move (red king and pawns on column a with Tiger and Horse
    is one of the five-piece ones): the rule is checked on its two pass children with hand-set values in a (4, 0) table."""
    cards = [0, 11, 2, 3, 1]  # Red holds Tiger and Horse
    s = O.make_state(cards, kings=[sq(4, 0), sq(2, 2)], pawns=[sq(0, 0) | sq(1, 0) | sq(2, 0) | sq(3, 0), 0], side=0)
    assert len(O.gen_moves(s)) == 0
    tables = {(4, 0): np.zeros(SIZES[(4, 0)], np.int16)}
    cls, (idx,) = onb.tb_index(cards, s)
    assert cls[0] == 20
    kids = []
    for slot in (0, 1):
        c = s.copy()
        c["cards"][0, [slot, 4]] = c["cards"][0, [4, slot]]
        c["side"] = 1
        kids.append(onb.tb_index(cards, c)[1][0])
    for v0, v1, want in ((3, 5, -6), (-4, 7, 5), (0, 9, 0), (-2, -6, 3)):
        tables[(4, 0)][kids] = [v0, v1]
        for held in (want, want + 2):
            tables[(4, 0)][idx] = held
            bad, _ = T.check_local(cards, 4, tables, 4, 0, idx=[idx])
            assert bad == (held != want), (v0, v1, held)


def test_oracle_table_is_locally_consistent_and_colour_symmetric_up_to_two_pawns():
    tables, info = T.solve(CARDS, 2)
    for (p, q), t in tables.items():
        bad, first = T.check_local(CARDS, 2, tables, p, q)
        assert bad == 0, (p, q, first)
        assert T.check_swap(CARDS, 2, tables, p, q) == 0, (p, q)
        assert ((t == NONE).sum()) == 47 * 60 * comb(23, p) * comb(23 - p, q)
        assert info[(p, q)]["max_win"] == t[t != NONE].max() or t[t != NONE].max() <= 0
    print({k: v for k, v in info.items()})


def test_oracle_agrees_with_alpha_beta_at_depth_six(onb):
    tables, _ = T.solve(CARDS, 2)
    rng = np.random.default_rng(11)
    picks = []
    for (p, q), t in sorted(tables.items()):
        short = np.nonzero((t != NONE) & (np.abs(t.astype(np.int32)) <= 6) & (t != 0))[0]
        other = np.nonzero((t != NONE) & ((np.abs(t.astype(np.int32)) > 6) | (t == 0)))[0]
        for pool in (short, other):
            if len(pool):
                picks += [(5 * p + q, int(i)) for i in rng.choice(pool, 200, replace=len(pool) < 200)]
    assert len(picks) >= 2000
    states = np.concatenate([onb.tb_states(CARDS, c, [i]) for c, i in picks])
    v = np.array([tables[(c // 5, c % 5)][i] for c, i in picks], np.int32)
    score = A.alphabeta_batch(states, 6)["score"]
    short = (v != 0) & (np.abs(v) <= 6)
    assert np.array_equal(score[short], np.sign(v[short]) * (A.WIN - np.abs(v[short])))
    assert (np.abs(score[~short]) < A.WIN - 6).all()
    assert short.sum() >= 1000
