"""The Gumbel root search (onb_mcts_set_gumbel, DESIGN.md §5f) on the CPU: the project's onb_log / onb_exp against libm and against a
pure-Python restatement, the sequential-halving table against an independent restatement, the oracle's completed-Q policy and action
against numpy, the sims = 1 action distribution against the prior, and known answers."""
import math
import struct

import numpy as np
import pytest
from scipy import stats

import gumbel_oracle as GO
import oracle_lib as O

TIGER, DRAGON, FROG, RABBIT, CRAB, ELEPHANT, GOOSE, ROOSTER, MONKEY, MANTIS, CRANE, HORSE, OX, BOAR, EEL, COBRA = range(16)


def sq(row, col):
    return 1 << (31 - (row * 5 + col))


def _ulps(a, b):
    """distance in units in the last place between two positive finite doubles (or two values of one sign)"""
    return np.abs(a.view(np.int64) - b.view(np.int64))


# ------------------------------------------------------------------ onb_log / onb_exp
def test_log_and_exp_are_within_two_ulp_of_libm():
    rng = np.random.default_rng(5)
    # log: the arguments the search forms (priors in (0, 1], u in (0, 1), -log u in (0, 23)) and a wide range of magnitudes
    x = np.concatenate([rng.random(400_000), np.exp(rng.uniform(-700, 700, 400_000)), rng.uniform(0.5, 2.0, 200_000),
                        (np.arange(1, 20001) + 0.5) * 2.0 ** -32])
    x = x[x > 0]
    assert len(x) >= 1_000_000
    got, want = GO.onb_log(x), np.log(x)
    pos = want != 0
    assert np.all(np.sign(got[pos]) == np.sign(want[pos]))
    assert _ulps(np.abs(got[pos]), np.abs(want[pos])).max() <= 2
    assert GO.onb_log(np.array([1.0]))[0] == 0.0
    # exp: softmax arguments (<= 0) and both signs elsewhere
    y = np.concatenate([-rng.exponential(5.0, 500_000), rng.uniform(-700, 700, 400_000), rng.uniform(-1, 1, 100_000)])
    got, want = GO.onb_exp(y), np.exp(y)
    assert _ulps(got, want).max() <= 2
    e = GO.onb_exp(np.array([0.0, -np.inf, np.inf, -800.0]))
    assert e[0] == 1.0 and e[1] == 0.0 and np.isposinf(e[2]) and e[3] == 0.0
    assert np.isneginf(GO.onb_log(np.array([0.0]))[0])


def _hi(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0] >> 32


def _lo(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0] & 0xFFFFFFFF


def _with_hi(x, hi):
    return struct.unpack("<d", struct.pack("<Q", ((hi & 0xFFFFFFFF) << 32) | _lo(x)))[0]


def py_log(x):
    """onb_log restated in Python (IEEE double arithmetic, one operation at a time), for positive normal x"""
    ln2_hi, ln2_lo = 6.93147180369123816490e-01, 1.90821492927058770002e-10
    Lg = [6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01, 1.818357216161805012e-01,
          1.531383769920937332e-01, 1.479819860511658591e-01]
    hx = _hi(x)
    k = (hx >> 20) - 1023
    hx &= 0x000FFFFF
    i0 = (hx + 0x95F64) & 0x100000
    x = _with_hi(x, hx | (i0 ^ 0x3FF00000))
    k += i0 >> 20
    f = x - 1.0
    dk = float(k)
    if (0x000FFFFF & (2 + hx)) < 3:
        if f == 0.0:
            return 0.0 if k == 0 else dk * ln2_hi + dk * ln2_lo
        R = (f * f) * (0.5 - 0.33333333333333333 * f)
        return f - R if k == 0 else dk * ln2_hi - ((R - dk * ln2_lo) - f)
    s = f / (2.0 + f)
    z = s * s
    i = hx - 0x6147A
    w = z * z
    j = 0x6B851 - hx
    t1 = w * (Lg[1] + w * (Lg[3] + w * Lg[5]))
    t2 = z * (Lg[0] + w * (Lg[2] + w * (Lg[4] + w * Lg[6])))
    i |= j
    R = t2 + t1
    if i > 0:
        hfsq = (0.5 * f) * f
        if k == 0:
            return f - (hfsq - s * (hfsq + R))
        return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f)
    if k == 0:
        return f - s * (f - R)
    return dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f)


def py_exp(x):
    """onb_exp restated in Python, for finite x in [-745, 709]"""
    ln2_hi, ln2_lo, invln2 = 6.93147180369123816490e-01, 1.90821492927058770002e-10, 1.44269504088896338700e+00
    P = [1.66666666666666019037e-01, -2.77777777770155933842e-03, 6.61375632143793436117e-05, -1.65339022054652515390e-06,
         4.13813679705723846039e-08]
    hx = _hi(x)
    xsb = (hx >> 31) & 1
    hx &= 0x7FFFFFFF
    k, hi, lo = 0, 0.0, 0.0
    if hx > 0x3FD62E42:
        if hx < 0x3FF0A2B2:
            hi = x + ln2_hi if xsb else x - ln2_hi
            lo = -ln2_lo if xsb else ln2_lo
            k = 1 - 2 * xsb
        else:
            k = int(invln2 * x + (-0.5 if xsb else 0.5))  # truncation towards zero
            t = float(k)
            hi = x - t * ln2_hi
            lo = t * ln2_lo
        x = hi - lo
    elif hx < 0x3E300000:
        return 1.0 + x
    t = x * x
    c = x - t * (P[0] + t * (P[1] + t * (P[2] + t * (P[3] + t * P[4]))))
    if k == 0:
        return 1.0 - ((x * c) / (c - 2.0) - x)
    y = 1.0 - ((lo - (x * c) / (2.0 - c)) - hi)
    if k >= -1021:
        return _with_hi(y, _hi(y) + (k << 20))
    return _with_hi(y, _hi(y) + ((k + 1000) << 20)) * 9.33263618503218878990e-302


def test_the_oracle_build_equals_a_python_restatement_bit_for_bit():
    rng = np.random.default_rng(9)
    x = np.concatenate([rng.random(6000), np.exp(rng.uniform(-700, 700, 6000)), 1.0 + rng.uniform(-1e-6, 1e-6, 1000)])
    got = GO.onb_log(x)
    assert all(struct.pack("<d", float(g)) == struct.pack("<d", py_log(float(v))) for g, v in zip(got, x))
    y = np.concatenate([-rng.exponential(5.0, 6000), rng.uniform(-740, 700, 6000), rng.uniform(-1e-8, 1e-8, 500)])
    got = GO.onb_exp(y)
    assert all(struct.pack("<d", float(g)) == struct.pack("<d", py_exp(float(v))) for g, v in zip(got, y))


# ------------------------------------------------------------------ sequential halving
def py_seq(m, n):
    """mctx's get_sequence_of_considered_visits"""
    if m <= 1:
        return list(range(n))
    log2max = int(math.ceil(math.log2(m)))
    seq, visits, c = [], [0] * m, m
    while len(seq) < n:
        extra = max(1, int(n / (log2max * c)))
        for _ in range(extra):
            seq.extend(visits[:c])
            for i in range(c):
                visits[i] += 1
        c = max(2, c // 2)
    return seq[:n]


def test_sequential_halving_table():
    for m in range(1, 41):
        for n in range(0, 1001):
            got = GO.seq(m, n)
            if n % 97 == 0 or n < 60 or m in (1, 2, 16, 40):  # the Python restatement is slow: every m, a spread of n
                assert got.tolist() == py_seq(m, n), (m, n)
            assert np.all(got[:min(m, n)] == 0)
            # replay the schedule on m actions: every descent finds an action with the scheduled visit count
            if m > 1 and n % 13 == 0:
                counts = np.zeros(m, np.int64)
                for v in got:
                    hit = np.nonzero(counts == v)[0]
                    assert len(hit), (m, n)
                    counts[hit[0]] += 1
                assert counts.sum() == n


# ------------------------------------------------------------------ the oracle against numpy
def _roots(n, seed, plies=12):
    g = O.new_games(n, seed=seed)
    for step in range(plies):
        live = (np.arange(n) % plies) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return g[g["result"] == 0]


def _numpy_policy(tree, r0, m, c_visit, c_scale, scale, seed, game, step):
    """pi' and the final action from a dumped root, in numpy (libm log / exp)"""
    k, fc = int(tree["n_child"][0]), int(tree["first_child"][0])
    ch = np.arange(fc, fc + k)
    P, N, W, act = tree["prior"][ch], tree["visits"][ch].astype(np.int64), tree["reward"][ch], tree["action"][ch].astype(np.int64)
    logit = np.where(P > 0, np.log(np.where(P > 0, P, 1.0)), -np.inf)
    u = (np.array([O.lib().orc_rand_u32(seed, game, step, 0x10000 + a) for a in range(k)], np.float64) + 0.5) * 2.0 ** -32
    g = scale * -np.log(-np.log(u))
    p = np.maximum(np.finfo(np.float64).tiny, P / P.sum())
    vis = N > 0
    q = np.where(vis, W / np.maximum(N, 1), 0.0)
    wq = (p[vis] * q[vis]).sum() / p[vis].sum() if vis.any() else 0.0
    v_mix = (-r0 + N.sum() * wq) / (N.sum() + 1)
    qh = np.where(vis, q, v_mix)
    sigma = (c_visit + N.max()) * c_scale * (qh - qh.min()) / max(qh.max() - qh.min(), 1e-8)
    score = np.maximum(-1e9, g + (logit - logit.max()) + sigma)
    score = np.where(N == N.max(), score, -np.inf)
    best = int(act[int(np.argmax(score))])
    z = logit + sigma
    e = np.exp(z - z.max())
    pi = np.zeros(50)
    np.add.at(pi, ((act >> 10) & 1) * 25 + (act & 31), e / e.sum())
    return pi, best


@pytest.mark.parametrize("evaluator,sims,m,scale", [(1, 17, 16, 1.0), (1, 50, 4, 1.0), (0, 40, 16, 0.0), (1, 2, 16, 1.0)])
def test_oracle_policy_and_action_equal_a_numpy_restatement(evaluator, sims, m, scale):
    roots = _roots(60, 7)
    for i in range(0, len(roots), 7):
        r = GO.search(roots[i:i + 1], 2.0, sims, evaluator=evaluator, m=m, gumbel_scale=scale, seed=11, step=3, game0=i, dump_tree=0, threads=1)
        pi, best = _numpy_policy(r["tree"], r["r0"][0], m, 50.0, 0.1, scale, 11, i, 3)
        # the oracle rounds its f64 pi' to f32: within one f32 rounding of the numpy value (which agrees with it to ~1e-15)
        got = r["pi"][0].reshape(50).astype(np.float64)
        assert np.all(np.abs(got - pi) <= np.spacing(np.abs(pi).astype(np.float32)).astype(np.float64) * 0.5 + 1e-12)
        assert r["best"][0] == best


def test_one_simulation_samples_the_prior():
    root = _roots(8, 3)[:1]
    n = 20000
    r = GO.search(np.repeat(root, n), 2.0, 1, evaluator=1, m=16, seed=21, step=0, game0=0)
    tree = GO.search(root, 2.0, 1, evaluator=1, dump_tree=0, threads=1)["tree"]
    k, fc = int(tree["n_child"][0]), int(tree["first_child"][0])
    acts, P = tree["action"][fc:fc + k], tree["prior"][fc:fc + k]
    counts = np.array([(r["best"] == a).sum() for a in acts])
    assert counts.sum() == n
    expect = P / P.sum() * n
    assert stats.chisquare(counts, expect).pvalue > 1e-3


def test_immediate_wins_are_found():
    s = O.make_state([RABBIT, FROG, TIGER, DRAGON, HORSE], kings=[sq(1, 3), 0x20000000], side=1)
    t = O.make_state([TIGER, FROG, RABBIT, CRAB, HORSE], kings=[sq(2, 2), sq(0, 0)], pawns=[0, 0], side=0)
    for root in (s, t):
        moves = O.gen_moves(root)
        wins = {int(a) for a in moves if O.make_move(root.copy(), a) in (1, 2)}
        assert wins
        for sims in (len(moves) + 1, len(moves) + 9, 3 * len(moves)):
            r = GO.search(root, 2.0, sims, evaluator=0, m=40, gumbel_scale=0.0, threads=1)
            assert int(r["best"][0]) in wins, sims
