"""Interior selection of Gumbel MuZero (onb_gumbel_config.interior, DESIGN.md §5f) on the CPU: the oracle's per-node rule against a
pure-Python restatement of the definition bit for bit and against a float64 numpy restatement of mctx's
qtransform_completed_by_mix_value + _prepare_argmax_input, the interior-off entry point against the root-only search, and known answers."""
import math

import numpy as np
import pytest

import gumbel_interior_oracle as GIO
import gumbel_oracle as GO
import oracle_lib as O
from test_gumbel_cpu import DRAGON, FROG, HORSE, RABBIT, TIGER, CRAB, sq

DBL_MIN = 2.2250738585072014e-308


def _nodes(n, seed):
    """n random nodes with ties, zero priors, all-zero priors, unvisited children and nodes without a visited child"""
    rng = np.random.default_rng(seed)
    k = np.where(rng.random(n) < 0.5, rng.integers(1, 14, n), rng.integers(1, 41, n))
    off = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)
    tot = int(off[-1])
    node = np.repeat(np.arange(n), k)
    kind = rng.integers(0, 6, n)[node]  # per node: how its priors, visits and values are drawn
    # priors: continuous, coarse (ties), with zeros, all zero
    P = rng.random(tot)
    P = np.where(kind == 1, rng.integers(0, 4, tot) / 8.0, P)
    P = np.where((kind == 2) & (rng.random(tot) < 0.3), 0.0, P)
    P = np.where(kind == 3, 0.0, P)
    P = np.where(kind == 5, 1.0 / 50.0, P)
    # visits: mostly small, many zeros; kind 4 and 5 nodes have no visited child; values W / N from f32 sums
    N = rng.integers(0, 12, tot) * (rng.random(tot) < 0.7)
    N = np.where((kind == 4) | (kind == 5), 0, N).astype(np.uint32)
    W = np.where(kind == 1, rng.integers(-3, 4, tot).astype(np.float64), rng.random(tot) * 2 - 1) * np.maximum(N, 1)
    W = W.astype(np.float32).astype(np.float64)
    Q = np.where(N > 0, W / np.maximum(N, 1), 0.0)
    rx = rng.random(n).astype(np.float32).astype(np.float64) * 2 - 1
    rx[rng.random(n) < 0.1] = 1.0
    rx[rng.random(n) < 0.1] = 0.0
    return off, P, N, Q, rx


def _python_choice(off, P, N, Q, rx, c_visit, c_scale):
    """the definition of include/onb.h restated on Python floats (IEEE f64 with correct rounding), onb_log / onb_exp from the oracle
    build (test_gumbel_cpu checks them bit for bit against a pure-Python restatement)"""
    n = len(rx)
    P, N, Q = P.tolist(), N.tolist(), Q.tolist()
    off = off.tolist()
    pre = []
    log_in = []
    for i in range(n):
        a0, a1 = off[i], off[i + 1]
        k = a1 - a0
        sP = 0.0
        for a in range(a0, a1):
            sP += P[a]
        uni = not (sP > 0.0)
        tot = float(k) if uni else sP
        Pu = [1.0 if uni else P[a] for a in range(a0, a1)]
        p = [max(DBL_MIN, x / tot) for x in Pu]
        log_at = []
        for x in Pu:
            if x > 0.0:
                log_at.append(len(log_in))
                log_in.append(x)
            else:
                log_at.append(-1)
        pre.append((a0, k, p, log_at))
    logs = GO.onb_log(np.array(log_in)).tolist()
    zs, exp_in = [], []
    for i, (a0, k, p, log_at) in enumerate(pre):
        sum_n, max_n, spq, sp = 0, 0, 0.0, 0.0
        for j in range(k):
            nj = N[a0 + j]
            if nj:
                spq += p[j] * Q[a0 + j]
                sp += p[j]
                sum_n += nj
                max_n = max(max_n, nj)
        wq = spq / sp if sp > 0.0 else 0.0
        v_mix = (-rx[i] + float(sum_n) * wq) / float(sum_n + 1)
        qh = [Q[a0 + j] if N[a0 + j] else v_mix for j in range(k)]
        lo, hi = min(qh), max(qh)
        rng_ = max(hi - lo, 1e-8)
        coef = (c_visit + float(max_n)) * c_scale
        z = [(logs[log_at[j]] if log_at[j] >= 0 else -math.inf) + coef * ((qh[j] - lo) / rng_) for j in range(k)]
        zmax = max(z)
        zs.append((len(exp_in), sum_n))
        exp_in.extend(x - zmax for x in z)
    e = GO.onb_exp(np.array(exp_in)).tolist()
    out = np.zeros(n, np.int64)
    for i, (a0, k, _, _) in enumerate(pre):
        base, sum_n = zs[i]
        se = 0.0
        for j in range(k):
            se += e[base + j]
        best, bs = 0, -math.inf
        for j in range(k):
            sc = e[base + j] / se - float(N[a0 + j]) / float(sum_n + 1)
            if sc > bs:
                best, bs = j, sc
        out[i] = best
    return out


def _pad(off, x, fill):
    k = np.diff(off)
    K = int(k.max())
    out = np.full((len(k), K), fill, dtype=np.asarray(x).dtype)
    col = np.arange(len(x)) - np.repeat(off[:-1], k)
    out[np.repeat(np.arange(len(k)), k), col] = x
    return out, np.arange(K)[None, :] < k[:, None]


def _softmax(x, valid):
    x = np.where(valid, x, -np.inf)
    m = x.max(axis=1, keepdims=True)
    e = np.where(valid, np.exp(x - m), 0.0)
    return e / e.sum(axis=1, keepdims=True)


def _mctx_scores(off, P, N, Q, rx, c_visit, c_scale):
    """mctx's gumbel_muzero_interior_action_selection in float64 numpy: qtransform_completed_by_mix_value (raw value = -r_x) and
    _prepare_argmax_input; prior logits = log of the stored priors (the project's all-zero rule: every P counts as 1)"""
    Pp, valid = _pad(off, P, 0.0)
    Np = _pad(off, N.astype(np.float64), 0.0)[0]
    Qp = _pad(off, Q, 0.0)[0]
    allzero = ~((Pp * valid).sum(axis=1) > 0)
    Pu = np.where(allzero[:, None], 1.0, Pp)
    with np.errstate(divide="ignore"):
        logits = np.where(valid & (Pu > 0), np.log(np.where(Pu > 0, Pu, 1.0)), -np.inf)
    prior = np.maximum(np.finfo(np.float64).tiny, _softmax(logits, valid))
    visited = valid & (Np > 0)
    sum_n = Np.sum(axis=1)
    sum_probs = np.where(visited, prior, 0.0).sum(axis=1)
    wq = np.where(visited, prior * Qp / np.where(sum_probs > 0, sum_probs, 1.0)[:, None], 0.0).sum(axis=1)
    value = (-rx + sum_n * wq) / (sum_n + 1)
    completed = np.where(visited, Qp, value[:, None])
    lo = np.where(valid, completed, np.inf).min(axis=1, keepdims=True)
    hi = np.where(valid, completed, -np.inf).max(axis=1, keepdims=True)
    resc = (completed - lo) / np.maximum(hi - lo, 1e-8)
    sigma = (c_visit + Np.max(axis=1, keepdims=True)) * c_scale * resc
    probs = _softmax(logits + sigma, valid)
    return np.where(valid, probs - Np / (1 + sum_n[:, None]), -np.inf)


@pytest.mark.parametrize("c_visit,c_scale", [(50.0, 0.1), (50.0, 1.0), (0.0, 0.05)])
def test_oracle_choice_equals_a_python_restatement_bit_for_bit(c_visit, c_scale):
    off, P, N, Q, rx = _nodes(100_000 if c_scale == 0.1 else 20_000, 3 + int(c_scale * 100))
    got = GIO.choice(off, P, N, Q, rx, c_visit, c_scale)
    want = _python_choice(off, P, N, Q, rx, c_visit, c_scale)
    assert np.array_equal(got, want)
    # the cases the generator is meant to produce are there
    k = np.diff(off)
    node = np.repeat(np.arange(len(rx)), k)
    no_visit = np.bincount(node, weights=N, minlength=len(rx)) == 0
    all_zero = np.bincount(node, weights=P, minlength=len(rx)) == 0
    n = len(rx)
    assert no_visit.sum() > n // 10 and all_zero.sum() > n // 10 and (P == 0).sum() > n // 10


def test_oracle_choice_equals_mctx_in_numpy():
    off, P, N, Q, rx = _nodes(100_000, 11)
    got = GIO.choice(off, P, N, Q, rx)
    sc = _mctx_scores(off, P, N, Q, rx, 50.0, 0.1)
    top2 = -np.sort(-sc, axis=1)[:, :2] if sc.shape[1] > 1 else np.concatenate([sc, np.full_like(sc, -np.inf)], axis=1)
    clear = ~(top2[:, 0] - top2[:, 1] <= 1e-12)
    assert clear.sum() > 50_000
    assert np.array_equal(got[clear], np.argmax(sc, axis=1)[clear])


def test_known_answers():
    # no visited child: pi' = the priors, the first maximal prior wins
    assert GIO.choice([0, 4], [0.1, 0.4, 0.4, 0.1], [0, 0, 0, 0], [0.0] * 4, [0.3])[0] == 1
    # all priors 0 and no visits: every child ties, the first one wins
    assert GIO.choice([0, 3], [0.0] * 3, [0, 0, 0], [0.0] * 3, [-0.5])[0] == 0
    # a zero-prior child is never chosen while another child has a prior and no child is visited
    assert GIO.choice([0, 2], [0.0, 1e-300], [0, 0], [0.0, 0.0], [0.0])[0] == 1
    # equal priors, one child visited with a good value: the visit-count term sends the next descent to the other child
    assert GIO.choice([0, 2], [0.5, 0.5], [1, 0], [1.0, 0.0], [0.0], 50.0, 0.0)[0] == 1


def _roots(n, seed, plies=12):
    g = O.new_games(2 * n, seed=seed)
    for step in range(plies):
        live = (np.arange(2 * n) % plies) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return np.ascontiguousarray(g[g["result"] == 0][:n])


@pytest.mark.parametrize("evaluator", [0, 1])
def test_interior_off_equals_the_root_only_search(evaluator):
    roots = _roots(64, 5 + evaluator)
    for m, sims in ((16, 1), (4, 50), (16, 200)):
        a = GO.search(roots, 2.0, sims, evaluator=evaluator, m=m, seed=3, step=2, dump_tree=7)
        b = GIO.search(roots, 2.0, sims, evaluator=evaluator, m=m, seed=3, step=2, dump_tree=7, interior=0)
        for k in a:
            if k == "tree":
                for f in a[k]:
                    assert np.array_equal(a[k][f], b[k][f]), f
            else:
                assert np.array_equal(a[k], b[k]), k
        c = GIO.search(roots, 2.0, sims, evaluator=evaluator, m=m, seed=3, step=2, interior=1)
        assert np.array_equal(c["root_visits"], a["root_visits"])
        if sims == 200:  # below the root the descent differs, and so do the trees
            assert not np.array_equal(c["n_nodes"], a["n_nodes"])


def test_immediate_wins_are_found():
    s = O.make_state([RABBIT, FROG, TIGER, DRAGON, HORSE], kings=[sq(1, 3), 0x20000000], side=1)
    t = O.make_state([TIGER, FROG, RABBIT, CRAB, HORSE], kings=[sq(2, 2), sq(0, 0)], pawns=[0, 0], side=0)
    for root in (s, t):
        moves = O.gen_moves(root)
        wins = {int(a) for a in moves if O.make_move(root.copy(), a) in (1, 2)}
        assert wins
        for sims in (len(moves) + 1, len(moves) + 9, 3 * len(moves)):
            r = GIO.search(root, 2.0, sims, evaluator=0, m=40, gumbel_scale=0.0, threads=1, interior=1)
            assert int(r["best"][0]) in wins, sims
