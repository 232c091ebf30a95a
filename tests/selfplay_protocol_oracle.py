"""Restatement of the self-play move protocol's choice (include/onb.h onb_self_play_set_protocol, DESIGN.md §5j) in plain Python
floats (IEEE f64, no FMA) on top of the host build of onb_gumbel.cuh's onb_log / onb_exp and the oracle's counter RNG. TEST
INFRASTRUCTURE: the kernels (k_mcts_choose) are compared against this bit for bit."""
import numpy as np

import gumbel_oracle as GO
import oracle_lib as O

DRAW_MOVE, DRAW_HELD = 0x20000, 0x20001


def weights(visits, temperature):
    """w(c) = onb_exp(onb_log(N(c)) / tau) for N(c) > 0, else 0 (child order)"""
    n = np.asarray(visits, dtype=np.float64)
    w = np.zeros(len(n))
    pos = n > 0
    if pos.any():
        w[pos] = GO.onb_exp(GO.onb_log(n[pos]) / temperature)   # numpy's f64 division is IEEE: the kernel's __ddiv_rn
    return [float(x) for x in w]


def sample_index(visits, w, r):
    """the sampled child for draw r (u = (r + 0.5) 2^-32): the first child whose inclusive running sum exceeds u * sum, else the last
    child with N > 0, else None"""
    total = 0.0
    for x in w:
        total += x
    thr = ((float(r) + 0.5) * 2.0 ** -32) * total
    acc, last = 0.0, None
    for c, x in enumerate(w):
        if visits[c] > 0:
            last = c
        acc += x
        if acc > thr:
            return c
    return last


def choose(root_w, root_n, visits, rewards, actions, best, sample, temperature, seed, game, step):
    """(move, m) of one searched root: visits / rewards / actions of the root's children in child order, best = onb_mcts_finish's"""
    m = -(root_w / root_n) if root_n else 0.0
    j = [c for c, a in enumerate(actions) if a == best]
    if j and visits[j[0]] > 0:
        q = rewards[j[0]] / visits[j[0]]
        if q > m:
            m = q
    move = best
    if sample and len(visits):
        c = sample_index(visits, weights(visits, temperature), O.lib().orc_rand_u32(seed, game, step, DRAW_MOVE))
        if c is not None:
            move = int(actions[c])
    return move, m


def held_out(seed, game, generation, holdout):
    """onb_rand_u32(seed, g, gen, 0x20001) < floor(h 2^32), compared as uint64"""
    return int(O.lib().orc_rand_u32(seed, game, generation, DRAW_HELD)) < int(np.floor(holdout * 4294967296.0))
