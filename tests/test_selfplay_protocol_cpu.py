"""The self-play move protocol's host-side pieces (DESIGN.md §5j) without a GPU: the restated move rule samples in proportion to
N^(1/tau), and selfplay.resign_threshold agrees with a brute-force scan."""
import numpy as np
import pytest
from scipy import stats

import oracle_lib as O
import selfplay_protocol_oracle as SP


@pytest.mark.parametrize("tau", [0.5, 1.0, 2.0])
@pytest.mark.parametrize("visits", [[3, 0, 12, 1, 40, 7, 0, 2], [1] * 40, [400, 1, 0, 0, 9, 33] + [2] * 30])
def test_move_frequencies_follow_the_tempered_visits(visits, tau):
    draws = 100000
    w = SP.weights(visits, tau)
    lib = O.lib()
    counts = np.zeros(len(visits), np.int64)
    for i in range(draws):
        c = SP.sample_index(visits, w, lib.orc_rand_u32(7, 1000 + i % 997, i // 997, SP.DRAW_MOVE))
        counts[c] += 1
    n = np.asarray(visits, np.float64)
    assert counts[n == 0].sum() == 0  # an unvisited child is never played
    p = n[n > 0] ** (1.0 / tau)
    p /= p.sum()
    expect = p * draws
    # merge the rare cells so that every expected count is at least 5
    obs, exp, acc_o, acc_e = [], [], 0, 0.0
    for o, e in sorted(zip(counts[n > 0], expect), key=lambda x: x[1]):
        acc_o, acc_e = acc_o + o, acc_e + e
        if acc_e >= 5:
            obs.append(acc_o); exp.append(acc_e); acc_o, acc_e = 0, 0.0
    if acc_e:
        obs[-1] += acc_o; exp[-1] += acc_e
    if len(obs) > 1:
        assert stats.chisquare(obs, exp).pvalue > 1e-3


def test_weights_match_the_exact_powers():
    for tau in (0.5, 1.0, 2.0):
        w = SP.weights([1, 2, 10, 400], tau)
        assert np.allclose(w, np.array([1, 2, 10, 400], np.float64) ** (1 / tau), rtol=1e-14)
    assert SP.weights([0, 5], 1.0)[0] == 0.0


def test_rounding_falls_back_to_the_last_visited_child():
    # u * sum can only reach the total through rounding; the rule then takes the last child with N > 0
    assert SP.sample_index([2, 3, 0], [2.0, 3.0, 0.0], 0xFFFFFFFF) == 1
    assert SP.sample_index([0, 0], [0.0, 0.0], 5) is None


def _brute(result, min_m, fp):
    """the largest candidate v (a minimum, or +inf) below which at most floor(fp G) held-out games have a non-loser with min m < v,
    counted as non-loser minima (conservative: a draw counts both sides)"""
    k = int(np.floor(fp * len(result)))
    vals = [min_m[i, 0] for i in range(len(result)) if result[i] != 2] + [min_m[i, 1] for i in range(len(result)) if result[i] != 1]
    best = -np.inf
    for v in sorted(set(vals)) + [np.inf]:
        if sum(1 for x in vals if x < v) <= k:
            best = max(best, v)
    # ... and at that v at most k games are false positives
    fp_games = sum(1 for i in range(len(result)) if (result[i] != 2 and min_m[i, 0] < best) or (result[i] != 1 and min_m[i, 1] < best))
    assert fp_games <= k
    return best if len(vals) > k else np.inf


@pytest.mark.parametrize("seed", range(40))
def test_resign_threshold_equals_a_brute_force_scan(seed):
    from onitama_alphazero_b200.selfplay import resign_threshold
    rng = np.random.default_rng(seed)
    g = int(rng.integers(0, 60))
    kind = seed % 4
    result = rng.integers(0, 3, g) if kind != 1 else np.zeros(g, np.int64)  # kind 1: all draws
    min_m = np.round(rng.uniform(-1, 1, (g, 2)), 2)                          # rounded: ties happen
    if g and kind == 2:
        min_m[rng.integers(0, g), rng.integers(0, 2)] = np.inf                 # a side that never searched
    for fp in (0.0, 0.05, 0.1, 0.5):
        got = resign_threshold(dict(result=result, min_m=min_m), fp)
        assert got == _brute(result, min_m, fp), (g, fp)


def test_resign_threshold_with_fewer_games_than_one_over_fp():
    from onitama_alphazero_b200.selfplay import resign_threshold
    result = np.array([1, 2, 0])
    min_m = np.array([[-0.2, -0.9], [-0.95, -0.1], [-0.5, -0.6]])
    assert resign_threshold(dict(result=result, min_m=min_m), 0.05) == -0.6   # k = 0: the smallest non-loser minimum
    assert resign_threshold(dict(result=result, min_m=min_m), 0.0) == -0.6
    assert resign_threshold(dict(result=result[:0], min_m=min_m[:0]), 0.05) == np.inf
