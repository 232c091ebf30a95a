"""Search-tree reuse between moves (onb_mcts_set_reuse) on the GPU against the CPU restatement (tests/reuse_oracle.cpp): the rerooted
trees bit for bit, continued searches over several plies, the no-match cases, order / subset / shard invariance, native self-play,
the switch, the limits and the refused split phase."""
import numpy as np
import pytest

import oracle_lib as O
import reuse_oracle as R

KEYS = ("visits", "reward", "prior", "action", "parent", "first_child", "n_child", "flags")


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def _roots(n, seed, plies=12):
    g = O.new_games(n, seed=seed)
    for step in range(plies):
        live = (np.arange(n) % plies) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return g


def _undecided(n, seed):
    g = _roots(2 * n, seed)
    return np.ascontiguousarray(g[g["result"] == 0][:n])


def _played(states, actions):
    out = states.copy()
    for i in range(len(out)):
        if out["result"][i] == 0 and actions[i] != 0xFFFF:
            O.make_move(out[i:i + 1], int(actions[i]))
    return out


def _same_results(a, b, mask=None, keys=("best", "pi", "root_visits", "root_q", "child_visits")):
    """mask: compare these games only (the oracle comparisons leave out decided positions, as test_gpu_parity does)"""
    for k in keys:
        x, y = a[k], b[k]
        if mask is not None:
            x, y = x[mask], y[mask]
        assert np.array_equal(x, y), k


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [0, 1])
def test_reroot_equals_the_oracle(onb, evaluator):
    n, sims, c = 4096, 64, 2.0
    roots = _undecided(n, 21 + evaluator)
    assert len(roots) == n
    rs = R.ReuseSet(n)
    want = rs.search(roots, c, sims, evaluator=evaluator)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_reuse(True)
        ctx.set_states(roots)
        ctx.mcts_begin(c, sims)
        ctx.mcts_run(evaluator, sims)
        got = ctx.mcts_finish()
        _same_results(got, want)
        ctx.mcts_play_best()
        moved = _played(roots, want["best"])
        assert np.array_equal(ctx.get_states(), moved)
        ctx.mcts_begin(c, sims)                    # reroot only
        rs.search(moved, c, 0, evaluator=evaluator)
        sizes, _ = ctx.mcts_tree_info()
        kept = 0
        for i in range(n):
            t_gpu, t_orc = ctx.mcts_dump_tree(i), rs.dump(i)
            assert len(t_gpu["visits"]) == len(t_orc["visits"]) == sizes[i], i
            for k in KEYS:
                assert np.array_equal(t_gpu[k], t_orc[k].astype(t_gpu[k].dtype)), (i, k)
            kept += len(t_gpu["visits"]) > 1
        assert kept > n // 2


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [0, 1])
@pytest.mark.parametrize("sims", [400, 800])
def test_continued_search_equals_the_oracle(onb, evaluator, sims):
    n, c, plies = 256, 2.0, 4
    states = _undecided(n, 40 + sims + evaluator)
    rs = R.ReuseSet(n)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_reuse(True)
        ctx.set_states(states)
        ctx.reuse_stats(clear=True)
        total_run = 0
        for ply in range(plies):
            want = rs.search(states, c, sims, evaluator=evaluator)
            ctx.mcts_begin(c, sims)
            ctx.mcts_run(evaluator, sims)
            got = ctx.mcts_finish()
            live = states["result"] == 0
            _same_results(got, want, live)
            sizes, _ = ctx.mcts_tree_info()
            assert np.array_equal(sizes.astype(np.int64)[live], want["n_nodes"][live]), ply
            total_run += int(want["sims_run"].sum())
            if ply:
                assert want["kept"].sum() > 0
            ctx.mcts_play_best()
            states = _played(states, want["best"])
            assert np.array_equal(ctx.get_states(), states)
        st = ctx.reuse_stats()
        assert st["sims"] == total_run and st["trees"] == n * plies and st["sims"] < n * plies * sims


@pytest.mark.gpu
def test_continued_search_with_the_fused_network(onb):
    from test_net_cpu import lively_model
    model = lively_model(3, seed=21)
    n, sims, c = 8, 48, 2.0
    states = _undecided(n, 77)
    rs = R.ReuseSet(n)
    with onb.Context(1, mcts_max_sims=2, planes=False) as one, onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        one.net_load(model)
        ctx.net_load(model)

        def eval_one(planes525):
            one.write(onb.BUF_LEAF_PLANES, np.asarray(planes525, dtype=np.float32).reshape(1, 525))
            one.net_forward(onb.BUF_LEAF_PLANES)
            return one.read(onb.BUF_POLICY, np.float32, (50,)), float(one.read(onb.BUF_VALUE, np.float32, (1,))[0])

        ctx.set_reuse(True)
        ctx.set_states(states)
        kept = 0
        for ply in range(3):
            want = rs.search(states, c, sims, callback=eval_one)
            ctx.mcts_begin(c, sims)
            ctx.mcts_run(onb.EVAL_NET, sims)
            got = ctx.mcts_finish()
            live = states["result"] == 0
            _same_results(got, want, live)
            for i in np.nonzero(live)[0]:
                t_gpu, t_orc = ctx.mcts_dump_tree(i), rs.dump(i)
                for k in ("visits", "reward", "prior"):
                    assert np.array_equal(t_gpu[k], t_orc[k]), (ply, i, k)
            kept += int(want["kept"].sum())
            ctx.mcts_play_best()
            states = _played(states, want["best"])
        assert kept >= n


@pytest.mark.gpu
def test_no_match_equals_a_fresh_search(onb):
    n, sims, c = 512, 200, 2.0
    roots = _undecided(n, 5)
    with onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ctx, onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ref:
        ctx.set_reuse(True)

        def both(states=None, reset=False):
            for x in (ctx, ref):
                if reset:
                    x.reset()
                if states is not None:
                    x.set_states(states)
            a = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
            b = ref.search(c, sims, evaluator=onb.EVAL_HASH)
            _same_results(a, b)
            return a

        both(roots)
        both(reset=True)                                  # after onb_env_reset
        both(roots)
        other = _undecided(n, 6)
        both(other)                                       # after set_states with unrelated positions
        both(roots)
        # a move other than the searched best (the least visited child): its subtree is the one kept, as the oracle keeps it
        alt = np.zeros(n, np.uint16)
        for i in range(n):
            t = ctx.mcts_dump_tree(i)
            kids = t["first_child"][0] + np.arange(t["n_child"][0])
            order = np.argsort(t["visits"][kids], kind="stable")
            alt[i] = t["action"][kids[order[0]]]
        moved = _played(roots, alt)
        for x in (ctx, ref):
            x.step(alt)
        a = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
        rs = R.ReuseSet(n)
        rs.search(roots, c, sims, evaluator=1)
        want = rs.search(moved, c, sims, evaluator=1)
        _same_results(a, want, moved["result"] == 0)
        assert want["kept"][moved["result"] == 0].all()


@pytest.mark.gpu
def test_results_do_not_depend_on_order_subset_or_shards(onb):
    n, sims, c = 1024, 100, 2.0
    states = _undecided(n, 8)
    sub = np.arange(0, n, 3)

    def plies(ctx, st, k=3, train=False):
        ctx.set_reuse(True)
        if train:
            ctx.mcts_set_noise(True, 0.25, 0.03, 7)
        ctx.set_states(st)
        out = []
        for _ in range(k):
            out.append(ctx.search(c, sims, evaluator=onb.EVAL_HASH))
            ctx.mcts_play_best()
        return out

    with onb.Context(n, mcts_max_sims=sims, planes=False) as full:
        a = plies(full, states)
    with onb.Context(len(sub), mcts_max_sims=sims, planes=False) as part:
        b = plies(part, np.ascontiguousarray(states[sub]))
    for x, y in zip(a, b):
        for k in ("best", "pi", "root_visits", "root_q", "child_visits"):
            assert np.array_equal(x[k][sub], y[k]), k
    # one context against two shards (game ids game_id_base + i key the root noise: train mode)
    with onb.Context(n, mcts_max_sims=sims, planes=False) as one:
        a = plies(one, states, train=True)
    h = n // 2
    with onb.Context(h, mcts_max_sims=sims, planes=False) as s0, onb.Context(h, game_id_base=h, mcts_max_sims=sims, planes=False) as s1:
        b0 = plies(s0, np.ascontiguousarray(states[:h]), train=True)
        b1 = plies(s1, np.ascontiguousarray(states[h:]), train=True)
    for x, y0, y1 in zip(a, b0, b1):
        for k in ("best", "pi", "root_visits", "root_q", "child_visits"):
            assert np.array_equal(x[k], np.concatenate([y0[k], y1[k]])), k


@pytest.mark.gpu
def test_native_self_play_with_reuse(onb):
    import torch
    n, sims, c, games = 40, 48, 2.0, 100
    with onb.Context(n, seed=17, mcts_max_sims=sims) as ctx:
        for train in (False, True):
            py = onb.self_play_continuous(ctx, c, sims, n_games=games, max_plies=30, evaluator=onb.EVAL_HASH, train=train, noise_seed=5, reuse=True)
            ctx.reuse_stats(clear=True)
            nat = ctx.self_play_native(c, sims, games, max_plies=30, evaluator=onb.EVAL_HASH, train=train, noise_seed=5, reuse=True)
            st = ctx.reuse_stats()
            assert nat["games"] == py["games"] == games and not nat["truncated"]
            for k in ("planes", "pi", "z", "serial", "color"):
                assert torch.equal(nat[k], py[k]), (k, train)
            assert st["kept"] > 0 and st["sims"] < st["trees"] * sims   # fewer leaf evaluations than n_live x sims summed over plies
            off = ctx.self_play_native(c, sims, games, max_plies=30, evaluator=onb.EVAL_HASH, train=train, noise_seed=5, reuse=False)
            assert off["games"] == games
            # every game complete, z = the final result from the sample's colour (0: cut at the cap)
            ser, z = nat["serial"].cpu().numpy(), nat["z"].cpu().numpy()
            for s in np.unique(ser):
                zs = z[ser == s]
                assert len(np.unique(np.abs(zs))) == 1
    # eval mode, one game per slot: the oracle's whole-game driver with reuse
    n, sims = 6, 64
    with onb.Context(n, seed=31, mcts_max_sims=sims) as ctx:
        nat = ctx.self_play_native(c, sims, n, max_plies=40, evaluator=onb.EVAL_HASH, reuse=True)
        want = R.play_games(O.new_games(n, seed=31), c, sims, evaluator=1, max_plies=40, reuse=True)
        ser, pi = nat["serial"].cpu().numpy(), nat["pi"].cpu().numpy()
        for s in range(n):
            rows = pi[ser == s]
            assert len(rows) == want["plies"][s]
            assert np.array_equal(rows, want["pi"][s, :want["plies"][s]]), s


@pytest.mark.gpu
def test_switch_off_and_fight(onb):
    n, sims, c = 256, 64, 2.0
    roots = _undecided(n, 12)
    with onb.Context(n, seed=4, mcts_max_sims=sims) as a, onb.Context(n, seed=4, mcts_max_sims=sims) as b:
        a.set_reuse(True)
        a.set_reuse(False)
        for x in (a, b):
            x.set_states(roots)
        for _ in range(2):
            _same_results(a.search(c, sims, evaluator=onb.EVAL_HASH), b.search(c, sims, evaluator=onb.EVAL_HASH))
            a.mcts_play_best()
            b.mcts_play_best()
        ra = a.self_play_native(c, 16, n, max_plies=10)
        rb = b.self_play_native(c, 16, n, max_plies=10)
        for k in ("pi", "z", "serial"):
            assert bool((ra[k] == rb[k]).all()), k
        # onb_fight ignores the switch
        red = (np.arange(n) % 2).astype(np.uint8)
        agent_a, agent_b = onb.Context.agent_puct(32, evaluator=onb.EVAL_HASH), onb.Context.agent_puct(16)
        a.set_reuse(True)
        for x in (a, b):
            x.reset()
        fa = a.fight_native(agent_a, agent_b, red, max_plies=20)
        fb = b.fight_native(agent_a, agent_b, red, max_plies=20)
        assert fa[:3] == fb[:3] and np.array_equal(fa[3], fb[3])
        assert a.last_fight_moves_chosen == b.last_fight_moves_chosen


@pytest.mark.gpu
def test_limits_and_refused_split_phase(onb):
    n, sims, c = 128, 200, 2.0
    roots = _undecided(n, 14)
    with onb.Context(n, mcts_max_sims=sims, mcts_node_cap=300, planes=False) as small:
        small.set_reuse(True)
        small.set_states(roots)
        for _ in range(3):
            small.search(c, sims, evaluator=onb.EVAL_HASH)
            _, flags = small.mcts_tree_info()
            assert (flags & 2).any()                          # kTreeOverflow, no fault
            small.mcts_play_best()
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_reuse(True)
        ctx.set_states(roots)
        for _ in range(4):
            r = ctx.search(c, sims, evaluator=onb.EVAL_HASH)
            _, flags = ctx.mcts_tree_info()
            assert not (flags & 2).any() and (r["root_visits"] <= sims).all()
            ctx.mcts_play_best()
        ctx.mcts_begin(c, sims)
        for call in (ctx.mcts_select, lambda: ctx.mcts_eval(onb.EVAL_UNIFORM), ctx.mcts_expand_backup,
                     lambda: ctx.mcts_run(onb.EVAL_HASH, sims - 1)):
            with pytest.raises(onb.OnbError):
                call()
        with pytest.raises(ValueError):
            ctx.search_device(c, sims, net=lambda p: None)
        ctx.set_reuse(False)
        ctx.mcts_begin(c, sims)
        ctx.mcts_select()                                     # reuse off: the split phase works again


@pytest.mark.gpu
def test_cpp_mirror_reuse_equals_the_context(onb, tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "test_reuse_mirror")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "test_reuse_mirror.cpp"),
                           "-o", exe, "-L" + os.path.join(root, "onitama_alphazero_b200"), "-lonb",
                           "-Wl,-rpath," + os.path.join(root, "onitama_alphazero_b200")])
    start = _undecided(1, 51)
    plies, sims = 8, 200
    r = start[0]
    line = " ".join(str(int(x)) for x in (*r["pawns"], *r["kings"], *r["cards"], r["side"]))
    p = subprocess.run([exe], input="%d %d\n%s\n" % (plies, sims, line), capture_output=True, text=True, timeout=600)
    assert p.returncode == 0 and p.stdout.strip().endswith("ALL OK"), p.stdout + p.stderr
    got = [int(x) for x in p.stdout.split("stats")[0].split()]
    want = []
    with onb.Context(1, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_reuse(True)
        ctx.set_states(start)
        for _ in range(len(got)):
            want.append(int(ctx.search(2.0, sims, evaluator=onb.EVAL_HASH)["best"][0]))
            ctx.mcts_play_best()
    assert got == want
