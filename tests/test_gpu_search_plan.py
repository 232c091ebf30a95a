"""A search runs with the settings it was begun with (onb_mcts_begin): include/onb.h says train-mode noise "applies to the searches
started after the call", so switching it on between the begin and the simulations must not reach the search already running --
neither the fused onb_mcts_run nor the split phase -- while the next search does see it."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


KEYS = ("best", "pi", "root_visits", "root_q", "child_visits")


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_noise_switched_on_after_the_begin_does_not_reach_the_running_search(onb, fused):
    n, sims, c = 512, 32, 2.0
    with onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()
        for step in range(4):
            ctx.step_random(step)
        states = ctx.get_states()
        want = ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused)  # eval mode throughout

        ctx.set_states(states)
        ctx.mcts_begin(c, sims)
        ctx.mcts_set_noise(True, seed=5)
        if fused:
            ctx.mcts_run(onb.EVAL_HASH, sims)
        else:
            for _ in range(sims):
                ctx.mcts_select()
                ctx.mcts_eval(onb.EVAL_HASH)
                ctx.mcts_expand_backup()
        got = ctx.mcts_finish()
        for k in KEYS:
            assert np.array_equal(got[k], want[k]), k

        ctx.set_states(states)
        train = ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused)  # begun with the switch on: the noise is there
        assert not np.array_equal(train["child_visits"], want["child_visits"])
