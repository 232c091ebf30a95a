"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden fixtures.
Bit-exact for states, actions, masks, planes, perft counts, visit counts; |dQ| <= 1e-5 is the stated tolerance for
Q values (they are in fact compared bit-exactly where noted)."""
import json
import math
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = json.load(open(os.path.join(ROOT, "tests", "golden", "golden.json")))
Q_TOL = 1e-5


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


# ------------------------------------------------------------------ boundary round trip
def test_state_roundtrip_and_reset(onb):
    n = 1000  # ragged: not a multiple of the 128-game tile
    with onb.Context(n, seed=5, game_id_base=77) as ctx:
        ctx.reset()
        assert ctx.get_states().tobytes() == O.new_games(n, seed=5, game0=77).tobytes()
        ctx.reset(decks=[1, 2, 0, 3, 11])
        assert ctx.get_states().tobytes() == O.new_games(n, deck=[1, 2, 0, 3, 11]).tobytes()
        rs = np.random.RandomState(1)
        s = O.new_games(n, seed=9)
        for i in range(n):  # arbitrary (even illegal) boards survive the packed 16-byte representation
            s["pawns"][i] = rs.randint(0, 2 ** 25, 2).astype(np.uint32) << 7
            s["kings"][i] = (1 << (31 - rs.randint(0, 25, 2))).astype(np.uint32)
            s["side"][i] = rs.randint(0, 2)
            s["result"][i] = rs.randint(0, 3)
            s["flags"][i] = rs.randint(0, 2)
        ctx.set_states(s)
        assert ctx.get_states().tobytes() == s.tobytes()
        ctx.set_states(s[10:20], first=500)
        assert ctx.get_states(500, 10).tobytes() == s[10:20].tobytes()


def test_error_paths(onb):
    with onb.Context(8, planes=False) as ctx:
        with pytest.raises(onb.OnbError) as e:
            ctx.encode()
        assert e.value.code == -4
        with pytest.raises(onb.OnbError) as e:
            ctx.mcts_begin(1.0, 10)
        assert e.value.code == -4
        with pytest.raises(onb.OnbError) as e:
            ctx.reset(decks=[[1, 2, 3, 4, 5]] * 3)
        assert e.value.code == -1
        with pytest.raises(onb.OnbError):
            ctx.reset(decks=[1, 2, 3, 4, 99])
    with onb.Context(8, mcts_max_sims=4) as ctx:
        ctx.reset()
        with pytest.raises(onb.OnbError) as e:
            ctx.mcts_select()
        assert e.value.code == -4
        with pytest.raises(onb.OnbError):
            ctx.mcts_begin(1.0, 5)


def test_get_bit_order_on_gpu(onb):
    """common/mod.rs:82-92 through the CUDA encoder and the boundary conversion"""
    gb = G["reference_tests"]["get_bit"]
    s = O.new_games(3, deck=[4, 3, 1, 0, 2])
    s["pawns"][1][0] = gb["bits"] & 0xFFFFFF80
    with onb.Context(3) as ctx:
        ctx.set_states(s)
        planes = ctx.encode()
        assert ctx.get_states().tobytes() == s.tobytes()
    assert planes[1, 0].reshape(25).tolist() == [float(b) for b in gb["expected"][:25]]
    assert np.array_equal(planes, O.encode(s))


# ------------------------------------------------------------------ reference known-answer tests through the GPU
def test_reference_make_move_cases_on_gpu(onb):
    cases = G["reference_tests"]["make_move"]
    states = O.new_games(len(cases), deck=cases[0]["deck"])
    actions = np.zeros(len(cases), dtype=np.uint16)
    for i, c in enumerate(cases):
        for k, v in c["set"].items():
            states[k[:-1]][i][int(k[-1])] = v
        states["side"][i] = c["color"]
        frm, to, piece = c["mov"]
        actions[i] = to | (frm << 5) | (c["card_idx"] << 10) | (piece << 12)
    with onb.Context(len(cases)) as ctx:
        ctx.set_states(states)
        ctx.step(actions)
        out = ctx.get_states()
    for i, c in enumerate(cases):
        want = {"InProgress": 0, "Capture": 0, "RedWin": 1, "BlueWin": 2}[c["result"]]
        assert int(out["result"][i]) == want, c["cite"]
        for (field, color, n, bit) in c["bits"]:
            assert (int(out[field][i][color]) >> (31 - n)) & 1 == bit
        assert int(out["cards"][i][4]) == c["neutral"]
        for (field, color, value) in c.get("equals", []):
            assert int(out[field][i][color]) == value
    ref = states.copy()
    O.env_step(ref, actions)
    assert out.tobytes() == ref.tobytes()


def test_reference_move_lists_on_gpu(onb):
    R = G["reference_tests"]
    rows = []
    for c in R["opening_moves"]:
        s = O.new_games(1, deck=c["deck"])
        s["side"][0] = c["color"]
        rows.append(s)
    for c in R["no_moves"]:
        rows.append(O.make_state(c["deck"], pawns=c["pawns"], kings=c["kings"], side=c["color"]))
    s = O.new_games(1, deck=R["expand_order"]["deck"])
    rows.append(s)
    states = np.concatenate(rows)
    with onb.Context(len(states)) as ctx:
        ctx.set_states(states)
        moves, counts = ctx.legal_moves()
        masks = ctx.legal_masks()
    for i in range(len(states)):
        want = O.gen_moves(states[i:i + 1])
        assert counts[i] == len(want)
        assert moves[i][:counts[i]].tolist() == want.tolist()  # same ORDER as the reference (slot, from, to)
        assert (moves[i][counts[i]:] == 0xFFFF).all()
    assert np.array_equal(masks, O.legal_masks(states))
    assert counts[5] == 0 and masks[5].tolist() == [0, 0]  # state.rs:852-889 no-legal-move position


# ------------------------------------------------------------------ lockstep stepping, both random policies
@pytest.mark.parametrize("policy", [0, 1])
@pytest.mark.parametrize("auto_reset", [False, True])
def test_env_step_random_bit_exact(onb, policy, auto_reset):
    n, seed, base = 3000, 1234 + policy, 1 << 33
    with onb.Context(n, seed=seed, game_id_base=base) as ctx:
        ctx.reset()
        ref = O.new_games(n, seed=seed, game0=base)
        for step in range(60):
            ctx.step_random(step, policy=policy, auto_reset=auto_reset, out_flags=onb.OUT_MASKS | onb.OUT_PLANES | onb.OUT_ACTIONS)
            acts = O.env_step_random(ref, seed, step, policy=policy, auto_reset=auto_reset, game0=base)
            if step % 7 == 0 or step == 59:
                assert ctx.get_states().tobytes() == ref.tobytes(), "state mismatch at step %d" % step
                assert np.array_equal(ctx.read(onb.BUF_ACTIONS, np.uint16, (n,)), acts)
                assert np.array_equal(ctx.read(onb.BUF_MASKS, np.uint32, (n, 2)), O.legal_masks(ref))
                assert np.array_equal(ctx.read(onb.BUF_PLANES, np.float32, (n, 21, 5, 5)), O.encode(ref))
        st = ctx.stats()
        if auto_reset:
            assert st[onb.STAT_STEPS] == 60 * n and st[onb.STAT_RESETS] == st[onb.STAT_RED_WINS] + st[onb.STAT_BLUE_WINS] > 0
        else:
            done = ref["result"] != 0
            assert st[onb.STAT_RED_WINS] + st[onb.STAT_BLUE_WINS] == done.sum()


def test_env_step_explicit_actions_and_fixed_deck(onb):
    n, seed = 777, 3
    deck = [4, 3, 1, 0, 2]
    with onb.Context(n, seed=seed) as ctx:
        ctx.reset(decks=deck)
        ref = O.new_games(n, deck=deck)
        for step in range(40):
            # actions chosen by the oracle's policy, applied through onb_env_step on the GPU
            shadow = ref.copy()
            acts = O.env_step_random(shadow, seed, step, policy=0, auto_reset=True, deck=deck)
            ctx.step(acts, out_flags=onb.OUT_MASKS)
            O.env_step(ref, acts)
            assert ctx.get_states().tobytes() == ref.tobytes()
        ctx.reset(decks=deck)
        ref = O.new_games(n, deck=deck)
        for step in range(80):  # auto-reset re-deals the SAME deck when the context was reset with one deck
            ctx.step_random(step, auto_reset=True)
            O.env_step_random(ref, seed, step, auto_reset=True, deck=deck)
        assert ctx.get_states().tobytes() == ref.tobytes()


def test_config1_playout_4096_games_bit_exact(onb):
    """BASELINE config 1: random-vs-random, 4096 games to terminal."""
    n, seed = 4096, 2024
    with onb.Context(n, seed=seed, planes=False) as ctx:
        ctx.reset()
        plies, trace = ctx.playout()
        fin = ctx.get_states()
        st = ctx.stats()
    ref, rplies, rtrace, total = O.playout_games(n, seed)
    assert fin.tobytes() == ref.tobytes()
    assert np.array_equal(plies, rplies) and np.array_equal(trace, rtrace)
    assert st[onb.STAT_STEPS] == total and st[onb.STAT_RED_WINS] + st[onb.STAT_BLUE_WINS] == n
    for row in G["playouts"]:  # committed golden trajectories (independent Python restatement)
        g = row["game"]
        assert int(plies[g]) == row["plies"] and str(int(trace[g])) == row["trace"]
        assert fin["pawns"][g].tolist() == row["pawns"] and fin["kings"][g].tolist() == row["kings"]
    # the in-register playout equals lockstep stepping, and a capped playout can be resumed
    with onb.Context(n, seed=seed, planes=False) as ctx:
        ctx.reset()
        ctx.playout(max_plies=20, want_plies=False, want_trace=False)
        ctx.playout(step0=20, want_plies=False, want_trace=False)
        assert ctx.get_states().tobytes() == ref.tobytes()


def test_sharding_invariance(onb):
    """Results depend on the GLOBAL game id only: two half-size contexts == one full-size context."""
    n, seed = 2048, 31
    with onb.Context(n, seed=seed, planes=False) as ctx:
        ctx.reset()
        ctx.playout(want_plies=False, want_trace=False)
        full = ctx.get_states()
    parts = []
    for r in range(2):
        with onb.Context(n // 2, seed=seed, game_id_base=r * (n // 2), planes=False) as ctx:
            ctx.reset()
            ctx.playout(want_plies=False, want_trace=False)
            parts.append(ctx.get_states())
    assert np.concatenate(parts).tobytes() == full.tobytes()


def test_large_batch_properties(onb):
    """BASELINE-size batch (1M games): size-independent properties + sampled parity against the oracle."""
    n, seed = 1 << 20, 99
    with onb.Context(n, seed=seed) as ctx:
        ctx.reset()
        for step in range(24):
            ctx.step_random(step, auto_reset=True, out_flags=onb.OUT_MASKS | onb.OUT_PLANES)
        states = ctx.get_states()
        ctx.sync()
        planes = ctx.tensor(onb.BUF_PLANES)
        # every plane value is 0/1; plane sums match popcounts of the boards; exactly two card planes are set
        assert bool(((planes == 0) | (planes == 1)).all())
        sums = planes.sum(dim=(2, 3)).cpu().numpy()
        pop = np.vectorize(lambda v: bin(int(v)).count("1"))
        idx = np.random.RandomState(0).choice(n, 4096, replace=False)
        assert np.array_equal(sums[idx, 0], pop(states["pawns"][idx, 0]))
        assert np.array_equal(sums[idx, 2], pop(states["pawns"][idx, 1]))
        assert (sums[:, 1] == 1).all() and (sums[:, 3] == 1).all()  # auto-reset: both kings always on board
        assert ((sums[:, 4:20] == 25).sum(axis=1) == 2).all()
        assert np.array_equal(sums[:, 20] == 25, states["side"] == 1)
        st = ctx.stats()
        assert st[onb.STAT_STEPS] == 24 * n
        # sampled games replayed by the oracle
        ref = np.zeros(len(idx), dtype=states.dtype)
        for k, gi in enumerate(idx):
            g = O.new_games(1, seed=seed, game0=int(gi))
            for step in range(24):
                O.env_step_random(g, seed, step, auto_reset=True, game0=int(gi))
            ref[k] = g[0]
        assert states[idx].tobytes() == ref.tobytes()
        assert np.array_equal(planes[idx.tolist()].cpu().numpy(), O.encode(ref))
        masks = ctx.read(onb.BUF_MASKS, np.uint32, (n, 2))
        assert np.array_equal(masks[idx], O.legal_masks(ref))


# ------------------------------------------------------------------ perft (BASELINE config 2)
def test_perft_vs_golden_and_oracle(onb):
    decks = [p["deck"] for p in G["perft"]]
    roots = onb.start_states(decks)
    with onb.Context(8, planes=False) as ctx:
        nodes, wins, zero = ctx.perft(roots, 5)
        for i, p in enumerate(G["perft"]):
            assert nodes[i].tolist() == p["nodes"] and wins[i].tolist() == p["wins"]
        assert zero.sum() == 0
        nodes6, wins6, _ = ctx.perft(roots, 6)
        for i, d in enumerate(decks):  # SURVEY Appendix A depth-6 values
            v = G["survey_appendix_a"]["perft"][",".join(map(str, d))]
            assert (nodes6[i] - wins6[i]).tolist() == v["leaves"]
            assert np.cumsum(wins6[i]).tolist() == v["cum_wins"]
        # shallow depths exercise the pure-DFS / pure-BFS corner cases
        for depth in (1, 2, 3):
            nd, wd, _ = ctx.perft(roots, depth)
            assert nd.tolist() == [p["nodes"][:depth] for p in G["perft"]]


def test_perft_midgame_roots_and_zero_move(onb):
    seed = 17
    g = O.new_games(64, seed=seed)
    for step in range(10):
        O.env_step_random(g, seed, step)
    case = G["reference_tests"]["no_moves"][1]
    stuck = O.make_state(case["deck"], pawns=case["pawns"], kings=case["kings"], side=case["color"])
    roots = np.concatenate([g, stuck])
    with onb.Context(8, planes=False) as ctx:
        nodes, wins, zero = ctx.perft(roots, 4)
    for i in range(len(roots)):
        n, w, z = O.perft(roots[i:i + 1], 4)
        assert nodes[i].tolist() == n.tolist() and wins[i].tolist() == w.tolist() and zero[i].tolist() == z.tolist(), i
    assert zero[-1][0] == 1 and nodes[-1].sum() == 0


def test_perft_all_deals_depth2_checksum(onb):
    """All 131 040 canonical deals: sum of perft(1), perft(2) == the independent restatement's totals."""
    decks = [[a, b, c, d, e] for a in range(16) for b in range(a + 1, 16) for c in range(16) if c not in (a, b)
             for d in range(c + 1, 16) if d not in (a, b) for e in range(16) if e not in (a, b, c, d)]
    assert len(decks) == G["all_deals"]["n_deals"]
    with onb.Context(8, planes=False) as ctx:
        nodes, wins, zero = ctx.perft(onb.start_states(decks), 3)
    assert int(nodes[:, 0].sum()) == G["all_deals"]["sum_perft1"]
    assert int(nodes[:, 1].sum()) == G["all_deals"]["sum_perft2"]
    assert zero.sum() == 0
    sample = np.random.RandomState(3).choice(len(decks), 40, replace=False)
    for i in sample:
        n, w, _ = O.perft(O.new_games(1, deck=decks[i]), 3)
        assert nodes[i].tolist() == n.tolist() and wins[i].tolist() == w.tolist()


# ------------------------------------------------------------------ PUCT search (BASELINE config 4)
def _cfg4_roots(n, seed):
    """roots = positions after p random plies (p = game id mod 16) of config-1 games"""
    g = O.new_games(n, seed=seed)
    for step in range(16):
        live = (np.arange(n) % 16) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    return g


def _compare_trees(ctx, roots, c, sims, evaluator, trees):
    for t in trees:
        if roots["result"][t] != 0:
            continue
        want = O.mcts_search(roots[t:t + 1], c, sims, evaluator=evaluator, dump=True)
        got = ctx.mcts_dump_tree(int(t))
        wt = want["tree"]
        assert len(got["visits"]) == want["n_nodes"], t
        assert np.array_equal(got["visits"], wt["visits"])          # every node's N, bit-exact
        assert np.array_equal(got["action"], wt["action"])
        assert np.array_equal(got["parent"], wt["parent"])
        assert np.array_equal(got["n_child"], wt["n_child"])
        assert np.array_equal(got["flags"], wt["flags"])
        assert np.array_equal(got["prior"], wt["prior"])            # f64 priors bit-exact
        assert np.array_equal(got["reward"], wt["reward"])          # f64 W bit-exact
        q = np.where(got["visits"] > 0, got["reward"] / np.maximum(got["visits"], 1), 0.0)
        assert np.abs(q - wt["winrate"]).max() <= Q_TOL


@pytest.mark.parametrize("c_puct", [math.sqrt(2.0), 2.0, 5.0])
def test_mcts_fused_uniform_bit_exact(onb, c_puct):
    n, sims, seed = 512, 400, 4
    roots = _cfg4_roots(n, seed)
    with onb.Context(n, seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        res = ctx.search(c_puct, sims, evaluator=onb.EVAL_UNIFORM, fused=True)
        want = O.mcts_search_batch(roots, c_puct, sims, evaluator=0, threads=8)
        live = roots["result"] == 0
        assert live.sum() > 400
        assert np.array_equal(res["child_visits"][live], want["child_visits"][live])
        assert np.array_equal(res["best"][live], want["best"][live])
        assert np.array_equal(res["root_visits"][live], np.full(live.sum(), sims))
        assert np.abs(res["root_q"][live] - want["root_q"][live]).max() <= Q_TOL
        assert np.array_equal(res["root_q"][live], want["root_q"][live])
        assert np.array_equal(res["pi"][live], want["pi"][live])
        nn, fl = ctx.mcts_tree_info()
        assert np.array_equal(nn[live], want["n_nodes"][live]) and (fl[live] & 2).sum() == 0
        _compare_trees(ctx, roots, c_puct, sims, 0, range(0, n, 37))


def test_mcts_golden_start_positions(onb):
    cases = [c for c in G["puct"] if c["sims"] <= 800]
    for c in cases:
        with onb.Context(4, mcts_max_sims=c["sims"], planes=False) as ctx:
            ctx.reset(decks=c["deck"])
            res = ctx.search(c["c_puct"], c["sims"])
            k = len(c["visits"])
            for t in range(4):
                assert res["child_visits"][t][:k].tolist() == c["visits"] and res["child_visits"][t][k:].sum() == 0
                assert int(res["best"][t]) == c["best"]
                assert res["root_q"][t] == c["root_q"]
            nn, _ = ctx.mcts_tree_info()
            assert nn.tolist() == [c["n_nodes"]] * 4
            tree = ctx.mcts_dump_tree(0)
            assert tree["prior"][1:1 + k].tolist() == c["child_prior"]


@pytest.mark.parametrize("fused", [True, False])
def test_mcts_hash_evaluator_bit_exact(onb, fused):
    """non-uniform priors and non-zero leaf values (sign-flipping backup, per-card renormalisation)"""
    n, sims, seed, c = 192, 150, 8, 1.7
    roots = _cfg4_roots(n, seed)
    with onb.Context(n, seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        res = ctx.search(c, sims, evaluator=onb.EVAL_HASH, fused=fused)
        want = O.mcts_search_batch(roots, c, sims, evaluator=1, threads=8)
        live = roots["result"] == 0
        assert np.array_equal(res["child_visits"][live], want["child_visits"][live])
        assert np.array_equal(res["best"][live], want["best"][live])
        assert np.abs(res["root_q"][live] - want["root_q"][live]).max() <= Q_TOL
        assert np.array_equal(res["pi"][live], want["pi"][live])
        _compare_trees(ctx, roots, c, sims, 1, range(0, n, 23))


def test_mcts_split_phase_equals_fused_and_leaf_planes(onb):
    n, sims, seed, c = 256, 64, 12, 2.0
    roots = _cfg4_roots(n, seed)
    with onb.Context(n, seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        fused = ctx.search(c, sims, evaluator=onb.EVAL_UNIFORM, fused=True)
        ctx.mcts_begin(c, sims)
        for s in range(sims):
            ctx.mcts_select()
            if s in (0, 5, 40):
                # the leaf planes handed to the evaluator are create_tensor_from_state of the leaf state
                planes = ctx.read(onb.BUF_LEAF_PLANES, np.float32, (n, 21, 5, 5))
                assert set(np.unique(planes)) <= {0.0, 1.0}
                if s == 0:
                    assert np.array_equal(planes, O.encode(roots))
                pol, val = O.hash_eval(planes[:8])
            ctx.mcts_eval(onb.EVAL_UNIFORM)
            ctx.mcts_expand_backup()
        split = ctx.mcts_finish()
        for k in fused:
            assert np.array_equal(fused[k], split[k]), k


def test_mcts_torch_evaluator_zero_copy(onb):
    """The network stays a black box: a torch callable reads LEAF_PLANES and writes POLICY/VALUE in place."""
    import torch
    n, sims, c = 64, 32, 2.0
    roots = _cfg4_roots(n, 21)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts), onb.Context(n, mcts_max_sims=sims, planes=False, stream=ts.cuda_stream) as ctx:
        assert ts.cuda_stream != 0
        ctx.set_states(roots)

        def net(planes):
            return torch.full((n, 2, 25), 1.0 / 50.0, device=planes.device), torch.zeros(n, device=planes.device)

        a = ctx.search(c, sims, net=net)
        b = ctx.search(c, sims, evaluator=onb.EVAL_UNIFORM, fused=True)
        for k in a:
            assert np.array_equal(a[k], b[k]), k


def test_mcts_pass_nodes_and_terminal_roots(onb):
    case = G["reference_tests"]["no_moves"][1]
    stuck = O.make_state(case["deck"], pawns=case["pawns"], kings=case["kings"], side=case["color"])
    won = O.new_games(1, deck=[1, 2, 0, 3, 11])
    won["kings"][0][1] = 0  # Blue king captured: decided root
    roots = np.concatenate([stuck, won, O.new_games(2, seed=1)])
    with onb.Context(4, mcts_max_sims=50, planes=False) as ctx:
        ctx.set_states(roots)
        res = ctx.search(1.5, 50)
        nn, fl = ctx.mcts_tree_info()
        assert fl[0] & 1 and not (fl[2] & 1)
        for t in range(4):
            want = O.mcts_search(roots[t:t + 1], 1.5, 50, dump=True)
            got = ctx.mcts_dump_tree(t)
            assert np.array_equal(got["visits"], want["tree"]["visits"]), t
            assert np.array_equal(got["reward"], want["tree"]["reward"]), t
            assert np.array_equal(got["action"], want["tree"]["action"]), t
            assert int(res["best"][t]) == want["best"]


def test_selfplay_loop_play_best(onb):
    """self_play's inner loop (train.rs:55-80): search, play the most visited move, flip side -- all games in lockstep."""
    n, sims, seed, c = 64, 48, 5, 2.0
    with onb.Context(n, seed=seed, mcts_max_sims=sims) as ctx:
        ctx.reset()
        ref = O.new_games(n, seed=seed)
        for ply in range(6):
            res = ctx.search(c, sims)
            want = O.mcts_search_batch(ref, c, sims, threads=8)
            live = ref["result"] == 0
            assert np.array_equal(res["best"][live], want["best"][live])
            ctx.mcts_play_best(out_flags=onb.OUT_PLANES)
            acts = want["best"].copy()
            O.env_step(ref, acts)
            assert ctx.get_states().tobytes() == ref.tobytes()
            assert np.array_equal(ctx.read(onb.BUF_PLANES, np.float32, (n, 21, 5, 5)), O.encode(ref))


# ------------------------------------------------------------------ self_play / fight drivers (train.rs:35-98, evaluator.rs:355-399)
def _oracle_self_play(n, seed, c, sims, max_plies):
    g = O.new_games(n, seed=seed)
    planes, pis, colors, games = [], [], [], []
    left = max_plies
    while (g["result"] == 0).any():
        live = np.flatnonzero(g["result"] == 0)
        res = O.mcts_search_batch(g, c, sims, threads=8)
        enc = O.encode(g)
        planes.append(enc[live]); pis.append(res["pi"][live]); colors.append(g["side"][live].copy()); games.append(live)
        O.env_step(g, res["best"])
        if left < 0:
            break
        left -= 1
    games = np.concatenate(games); colors = np.concatenate(colors)
    r = g["result"][games].astype(np.int64)
    z = np.where(r == 0, 0.0, np.where((r - 1) == colors, 1.0, -1.0)).astype(np.float32)
    return dict(planes=np.concatenate(planes), pi=np.concatenate(pis), z=z, color=colors, game=games), g


def test_self_play_driver_bit_exact(onb):
    n, seed, c, sims, max_plies = 48, 77, 2.0, 40, 22
    with onb.Context(n, seed=seed, mcts_max_sims=sims) as ctx:
        out = onb.self_play(ctx, c, sims, max_plies=max_plies)
        final = ctx.get_states()
    want, g = _oracle_self_play(n, seed, c, sims, max_plies)
    assert final.tobytes() == g.tobytes()
    assert np.array_equal(out["game"].cpu().numpy(), want["game"])
    assert np.array_equal(out["color"].cpu().numpy(), want["color"])
    assert np.array_equal(out["planes"].cpu().numpy(), want["planes"])
    assert np.array_equal(out["pi"].cpu().numpy(), want["pi"])
    assert np.array_equal(out["z"].cpu().numpy(), want["z"])
    # the 152-ply guard of the reference (max_plies = 150 -> 152 plies, SURVEY Q15) in miniature: max_plies + 2 plies
    assert out["game"].shape[0] <= n * (max_plies + 2)
    assert (np.bincount(want["game"], minlength=n) <= max_plies + 2).all()


def test_fight_mcts_vs_random(onb):
    """fight(): agent A = PUCT search (uniform evaluator), agent B = the reference's `Random` agent, colours alternate."""
    import torch
    n, seed, c, sims = 64, 9, 2.0, 48
    a_is_red = (np.arange(n) % 2) == 0
    step_counter = {"i": 0}
    with onb.Context(n, seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()

        def mcts_agent(cx):
            cx.search_device(c, sims)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        def random_agent(cx):
            cx.choose_random(step_counter["i"], policy=onb.POLICY_AGENT)
            step_counter["i"] += 1

        a, b, d = onb.fight(ctx, mcts_agent, random_agent, a_is_red, max_plies=150)
        final = ctx.get_states()
    # oracle replay of the same arena
    g = O.new_games(n, seed=seed)
    left, i = 150, 0
    while (g["result"] == 0).any():
        res = O.mcts_search_batch(g, c, sims, threads=8)
        shadow = g.copy()
        rnd = O.env_step_random(shadow, seed, i, policy=1)
        i += 1
        a_to_move = (g["side"] == 0) == a_is_red
        acts = np.where(a_to_move, res["best"], rnd).astype(np.uint16)
        O.env_step(g, acts)
        if left < 0:
            break
        left -= 1
    assert final.tobytes() == g.tobytes()
    red, blue = g["result"] == 1, g["result"] == 2
    assert a == int((red & a_is_red).sum() + (blue & ~a_is_red).sum())
    assert b == int((red & ~a_is_red).sum() + (blue & a_is_red).sum())
    assert a + b + d == n and a > b  # 48-sim search beats the random agent


def test_cpp_host_mirror_reference_tests(onb):
    """The reference's unit tests re-expressed in C++ against include/onitama_b200.hpp, run on the GPU."""
    import subprocess
    import __graft_entry__ as ge
    exe = ge.build_cpp_mirror_test()
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout + r.stderr


def test_search_with_network_black_box_bit_exact(onb):
    """BASELINE config 5 in miniature: the 3-block ConvResNet (random init, fixed seed) drives the split-phase search.
    Both sides see bit-identical network outputs (the same CPU module evaluated sample by sample), so visit counts, priors
    and W must be bit-exact; this exercises select -> leaf planes -> policy/value buffers -> expand/backup end to end."""
    import torch
    from onitama_alphazero_b200.net import ConvResNet
    torch.manual_seed(1234)
    model = ConvResNet(64, 21, 3).eval()
    for m in model.modules():  # non-trivial BatchNorm statistics
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5)

    @torch.no_grad()
    def eval_one(planes525):
        p, v = model(torch.from_numpy(np.asarray(planes525, dtype=np.float32)).reshape(1, 21, 5, 5))
        return p.reshape(50).numpy(), float(v.reshape(()))

    n, sims, c = 6, 40, 2.0
    roots = _cfg4_roots(16, 5)[[1, 3, 6, 9, 12, 15]]
    with onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)

        def net(planes_dev):
            host = planes_dev.cpu().numpy()
            outs = [eval_one(host[i]) for i in range(n)]
            pol = torch.from_numpy(np.stack([o[0] for o in outs])).to(planes_dev.device)
            val = torch.tensor([o[1] for o in outs], dtype=torch.float32, device=planes_dev.device)
            return pol, val

        res = ctx.search(c, sims, net=net)
        for t in range(n):
            if roots["result"][t] != 0:
                continue
            want = O.mcts_search(roots[t:t + 1], c, sims, dump=True, callback=eval_one)
            got = ctx.mcts_dump_tree(t)
            assert np.array_equal(got["visits"], want["tree"]["visits"]), t
            assert np.array_equal(got["prior"], want["tree"]["prior"])
            assert np.array_equal(got["reward"], want["tree"]["reward"])
            assert int(res["best"][t]) == want["best"]
            assert np.array_equal(res["pi"][t], want["pi"])
            assert abs(res["root_q"][t] - want["root_q"]) <= Q_TOL


def test_selfplay_with_gpu_network_runs(onb):
    """The same network on the GPU, zero-copy on the context's stream (statistical check only: GPU conv != CPU conv bitwise)."""
    import torch
    from onitama_alphazero_b200.net import ConvResNet, make_evaluator
    torch.manual_seed(7)
    net = make_evaluator(ConvResNet(64, 21, 3).cuda())
    n, sims = 32, 16
    with onb.Context(n, seed=2, mcts_max_sims=sims) as ctx:
        out = onb.self_play(ctx, 2.0, sims, max_plies=6, net=net)
        # one simulation round captured in a CUDA graph and replayed gives the same search as eager launches
        ctx.reset()
        ctx.search_device(2.0, sims, net=net)
        eager = ctx.mcts_finish()
        ctx.search_device(2.0, sims, net=net, use_graph=True)
        ctx.search_device(2.0, sims, net=net, use_graph=True)  # second call reuses the cached graph
        graphed = ctx.mcts_finish()
        assert np.array_equal(eager["child_visits"], graphed["child_visits"]) and np.array_equal(eager["best"], graphed["best"])
    m = out["planes"].shape[0]
    assert m == n * 8 or m <= n * 8
    assert torch.allclose(out["pi"].sum(dim=(1, 2)), torch.ones(m, device=out["pi"].device), atol=1e-5)
    assert set(out["z"].unique().tolist()) <= {-1.0, 0.0, 1.0}


def test_mcts_deep_paths_bit_exact(onb):
    """Many simulations from late positions: descents deeper than the lane-held path (8 levels with 8 lanes per tree) use the
    parent-chain backup; more children than lanes are scanned in several rounds. Every node must still match the oracle."""
    seed, sims, c = 41, 1500, 0.1  # a small c_puct with non-zero leaf values digs deep (20 levels with the hash evaluator)
    g = O.new_games(96, seed=seed)
    for step in range(30):
        O.env_step_random(g, seed, step)
    roots = g[g["result"] == 0][:40]
    assert len(roots) >= 20
    with onb.Context(len(roots), seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        for ev in (onb.EVAL_UNIFORM, onb.EVAL_HASH):
            res = ctx.search(c, sims, evaluator=ev, fused=True)
            want = O.mcts_search_batch(roots, c, sims, evaluator=ev, threads=8)
            assert np.array_equal(res["child_visits"], want["child_visits"])
            assert np.array_equal(res["best"], want["best"])
            assert np.array_equal(res["root_q"], want["root_q"])
            deepest = 0
            for t in range(0, len(roots), 3):
                w = O.mcts_search(roots[t:t + 1], c, sims, evaluator=ev, dump=True)
                got = ctx.mcts_dump_tree(t)
                assert np.array_equal(got["visits"], w["tree"]["visits"]) and np.array_equal(got["reward"], w["tree"]["reward"])
                assert np.array_equal(got["parent"], w["tree"]["parent"]) and np.array_equal(got["flags"], w["tree"]["flags"])
                par = w["tree"]["parent"]
                depth = np.zeros(len(par), dtype=np.int32)
                for i in range(1, len(par)):
                    depth[i] = depth[par[i]] + 1
                deepest = max(deepest, int(depth.max()))
            if ev == onb.EVAL_HASH:
                assert deepest >= 12, "test positions did not produce a path deeper than the lane-held levels (%d)" % deepest


# ------------------------------------------------------------------ edge cases
@pytest.mark.parametrize("n", [1, 2, 31, 33, 63, 65, 129])
def test_ragged_sizes(onb, n):
    """tiny and ragged batch sizes: partial tiles, partial warps, partial 8-lane groups"""
    seed = 100 + n
    with onb.Context(n, seed=seed, mcts_max_sims=24) as ctx:
        ctx.reset()
        ref = O.new_games(n, seed=seed)
        for step in range(9):
            ctx.step_random(step, auto_reset=True, out_flags=onb.OUT_MASKS | onb.OUT_PLANES)
            O.env_step_random(ref, seed, step, auto_reset=True)
        assert ctx.get_states().tobytes() == ref.tobytes()
        assert np.array_equal(ctx.read(onb.BUF_PLANES, np.float32, (n, 21, 5, 5)), O.encode(ref))
        assert np.array_equal(ctx.read(onb.BUF_MASKS, np.uint32, (n, 2)), O.legal_masks(ref))
        res = ctx.search(1.9, 24)
        want = O.mcts_search_batch(ref, 1.9, 24)
        assert np.array_equal(res["child_visits"], want["child_visits"]) and np.array_equal(res["best"], want["best"])
        split = ctx.search(1.9, 24, fused=False)
        assert np.array_equal(split["child_visits"], want["child_visits"])


def test_action_none_is_a_noop(onb):
    n = 200
    with onb.Context(n, seed=6) as ctx:
        ctx.reset()
        ref = O.new_games(n, seed=6)
        shadow = ref.copy()
        acts = O.env_step_random(shadow, 6, 0)
        acts[::3] = 0xFFFF
        ctx.step(acts, out_flags=onb.OUT_MASKS | onb.OUT_PLANES)
        O.env_step(ref, acts)
        got = ctx.get_states()
        assert got.tobytes() == ref.tobytes()
        assert got[::3].tobytes() == O.new_games(n, seed=6)[::3].tobytes()
        assert np.array_equal(ctx.read(onb.BUF_PLANES, np.float32, (n, 21, 5, 5)), O.encode(ref))


def test_mcts_in_chunks_and_pool_overflow(onb):
    """onb_mcts_run may be called several times per search (sims accumulate); a too-small node pool is reported, not fatal."""
    n, c = 40, 2.0
    roots = _cfg4_roots(n, 3)
    with onb.Context(n, mcts_max_sims=200, planes=False) as ctx:
        ctx.set_states(roots)
        ctx.mcts_begin(c, 200)
        for chunk in (1, 7, 92, 100):
            ctx.mcts_run(onb.EVAL_UNIFORM, chunk)
        a = ctx.mcts_finish()
        b = ctx.search(c, 200)
        for k in a:
            assert np.array_equal(a[k], b[k]), k
        with pytest.raises(onb.OnbError):
            ctx.mcts_run(onb.EVAL_UNIFORM, 1)  # more simulations than mcts_max_sims
    with onb.Context(n, mcts_max_sims=200, mcts_node_cap=300, planes=False) as ctx:
        ctx.set_states(roots)
        res = ctx.search(c, 200)
        nn, fl = ctx.mcts_tree_info()
        assert (nn <= 300).all() and (fl & 2).any()           # overflow flagged per tree
        assert (res["root_visits"] == 200).all()               # the search still completes every simulation
        assert (res["child_visits"].sum(axis=1) == 199)[roots["result"] == 0].all()


# ------------------------------------------------------------------ train mode: root exploration noise (statistical parity)
@pytest.mark.parametrize("fused", [True, False])
def test_mcts_train_mode_noise_statistical(onb, fused):
    """AlphaZeroMctsConfig::train: the reference's noise comes from thread_rng, so only the DISTRIBUTION can be compared. GPU and
    oracle share the counter RNG and the sampling algorithm; libm vs CUDA math may flip a rare comparison, so: (a) the large
    majority of trees must be identical, (b) the mean root visit vectors must agree closely, (c) the noise must matter."""
    n, sims, c, seed = 512, 120, 2.0, 77
    roots = O.new_games(n, deck=[1, 2, 0, 3, 11])
    with onb.Context(n, mcts_max_sims=sims, planes=False, game_id_base=1000) as ctx:
        ctx.set_states(roots)
        quiet = ctx.search(c, sims, fused=fused)
        ctx.mcts_set_noise(True, 0.25, 0.03, seed)
        noisy = ctx.search(c, sims, fused=fused)
        again = ctx.search(c, sims, fused=fused)
        ctx.mcts_set_noise(False)
        quiet2 = ctx.search(c, sims, fused=fused)
    try:
        O.mcts_set_noise(True, 0.25, 0.03, seed, game0=1000)
        want = O.mcts_search_batch(roots, c, sims, threads=8)
    finally:
        O.mcts_set_noise(False)
    assert np.array_equal(noisy["child_visits"], again["child_visits"])      # repeatable (counter RNG)
    assert np.array_equal(quiet["child_visits"], quiet2["child_visits"])     # switching it off restores eval mode
    assert (noisy["child_visits"] != quiet["child_visits"]).any(axis=1).mean() > 0.9   # the noise changes almost every tree
    assert len({tuple(r) for r in noisy["child_visits"]}) > n // 4                      # and differs between trees
    same = (noisy["child_visits"] == want["child_visits"]).all(axis=1).mean()
    assert same >= 0.9, "only %.1f%% of the trees match the oracle" % (100 * same)
    assert np.abs(noisy["child_visits"][:, :10].mean(axis=0) - want["child_visits"][:, :10].mean(axis=0)).max() < 0.25
    assert (noisy["child_visits"].sum(axis=1) == sims - 1).all()


def test_self_play_train_mode(onb):
    n, sims = 64, 32
    with onb.Context(n, seed=4, mcts_max_sims=sims) as ctx:
        ctx.mcts_set_noise(True, 0.25, 0.03, 9)
        out = onb.self_play(ctx, 2.0, sims, max_plies=8)
        assert out["planes"].shape[0] > 0
        assert abs(float(out["pi"].sum()) - out["pi"].shape[0]) < 1e-3


# ------------------------------------------------------------------ BASELINE-size runs: properties + sampled parity
def test_config4_full_size_properties_and_sampled_parity(onb):
    """16 384 trees x 400 simulations (BASELINE config 4): size-independent invariants on every tree, bit-exact visit vectors on a
    sample of trees replayed by the oracle."""
    n, sims, c, seed = 1 << 14, 400, 2.0, 20240607
    with onb.Context(n, seed=seed, mcts_max_sims=sims, planes=False) as ctx:
        ctx.reset()
        base = ctx.get_states()
        cur = base.copy()
        for step in range(16):  # roots = positions after p = id mod 16 random plies
            ctx.step_random(step)
            nxt = ctx.get_states()
            live = (np.arange(n) % 16) > step
            cur[live] = nxt[live]
            ctx.set_states(cur)
        dead = cur["result"] != 0
        cur[dead] = base[dead]
        ctx.set_states(cur)
        res = ctx.search(c, sims)
        nn, fl = ctx.mcts_tree_info()
        assert (res["root_visits"] == sims).all()
        assert (res["child_visits"].sum(axis=1) == sims - 1).all()      # every playout after the first passes through one root child
        assert np.allclose(res["pi"].sum(axis=(1, 2)), 1.0, atol=1e-6)
        assert (np.abs(res["root_q"]) <= 1.0).all() and (fl & 2).sum() == 0
        assert (nn <= 1 + 40 * sims).all() and (nn > 1).all()
        best_slot = (res["best"] >> 10) & 3
        assert ((best_slot >> 1) == cur["side"]).all()                   # the chosen card belongs to the side to move
        # the most visited child's move is the reported best move (last maximum wins)
        idx = np.random.RandomState(1).choice(n, 48, replace=False)
        want = O.mcts_search_batch(cur[idx], c, sims, threads=8)
        assert np.array_equal(res["child_visits"][idx], want["child_visits"])
        assert np.array_equal(res["best"][idx], want["best"])
        assert np.array_equal(res["root_q"][idx], want["root_q"])
        assert np.array_equal(nn[idx], want["n_nodes"])


def test_config2_full_size_perft(onb):
    """All 131 040 canonical deals to depth 6 (BASELINE config 2): checksums against the independent restatement, wins are a
    subset of nodes, sampled deals bit-exact against the oracle at every depth."""
    decks = np.array([[a, b, c, d, e] for a in range(16) for b in range(a + 1, 16) for c in range(16) if c not in (a, b)
                      for d in range(c + 1, 16) if d not in (a, b) for e in range(16) if e not in (a, b, c, d)], dtype=np.uint8)
    with onb.Context(8, planes=False) as ctx:
        nodes, wins, zero = ctx.perft(onb.start_states(decks), 6)
    assert int(nodes[:, 0].sum()) == G["all_deals"]["sum_perft1"] and int(nodes[:, 1].sum()) == G["all_deals"]["sum_perft2"]
    assert zero.sum() == 0 and (wins <= nodes).all() and (wins[:, :2] == 0).all()
    assert (nodes[:, 1:] <= nodes[:, :-1] * 40).all() and (nodes[:, 5] > nodes[:, 4]).all()
    # mirror symmetry of the rules: swapping the two cards inside a hand does not change the counts
    first = {tuple(d): i for i, d in enumerate(decks.tolist())}
    for i in np.random.RandomState(5).choice(len(decks), 12, replace=False):
        n_, w_, _ = O.perft(O.new_games(1, deck=decks[i]), 6)
        assert nodes[i].tolist() == n_.tolist() and wins[i].tolist() == w_.tolist(), decks[i]


def test_mcts_wide_nodes_more_than_32_children(onb):
    """Roots with 33-36 legal moves: more children than a warp has lanes (two rounds in the warp-per-tree kernels, five rounds
    of 8 lanes in the fused kernel); both paths must match the oracle node for node."""
    seed = 123
    g = O.new_games(4096, seed=seed)
    picks = {12: [627], 16: [3247, 320], 14: [2338], 20: [462], 32: [185, 3256], 34: [2725]}
    roots = []
    for step in range(35):
        O.env_step_random(g, seed, step)
        for i in picks.get(step, []):
            roots.append(g[i:i + 1].copy())
    roots = np.concatenate(roots)
    counts = [len(O.gen_moves(roots[i:i + 1])) for i in range(len(roots))]
    assert min(counts) >= 33 and max(counts) >= 36
    sims, c = 300, 2.0
    with onb.Context(len(roots), mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        for fused in (True, False):
            for ev in (onb.EVAL_UNIFORM, onb.EVAL_HASH):
                res = ctx.search(c, sims, evaluator=ev, fused=fused)
                want = O.mcts_search_batch(roots, c, sims, evaluator=ev)
                assert np.array_equal(res["child_visits"], want["child_visits"]), (fused, ev)
                assert np.array_equal(res["best"], want["best"]) and np.array_equal(res["pi"], want["pi"])
                for t in range(len(roots)):
                    w = O.mcts_search(roots[t:t + 1], c, sims, evaluator=ev, dump=True)
                    got = ctx.mcts_dump_tree(t)
                    assert np.array_equal(got["visits"], w["tree"]["visits"]) and np.array_equal(got["prior"], w["tree"]["prior"])
                    assert got["n_child"].max() >= 33


def test_reference_tactical_positions(onb):
    """The two tactical sanity positions of the reference's plain-MCTS tests (ai/mcts/mcts_arena.rs:460-523: take the king with
    the Dragon card; the only king move that does not lose). They pin a different agent statistically; the PUCT search with the
    uniform evaluator finds the same moves, on the GPU and in the oracle alike."""
    def bb(r, c):
        return 0x80000000 >> (r * 5 + c)
    a = O.make_state([3, 2, 0, 1, 11], side=1)           # Dragon,Frog,Tiger,Rabbit,Horse with slots 0 and 3 swapped
    a["kings"][0][0] = bb(1, 3)
    b = O.make_state([12, 8, 3, 11, 1], side=1)          # Ox,Monkey | Rabbit,Horse | Dragon
    b["kings"][0][1] = bb(0, 4); b["pawns"][0][1] = 0; b["pawns"][0][0] = bb(0, 3) | bb(1, 4)
    roots = np.concatenate([a, b])
    expected = [1 << 5 | 8 | (3 << 10), 4 << 5 | 2 | (2 << 10) | (1 << 12)]   # (from 1 -> 8 pawn, card idx 3), (king 4 -> 2, card idx 2)
    for sims in (400, 2000):
        with onb.Context(2, mcts_max_sims=sims, planes=False) as ctx:
            ctx.set_states(roots)
            res = ctx.search(math.sqrt(2.0), sims)
        want = O.mcts_search_batch(roots, math.sqrt(2.0), sims)
        assert res["best"].tolist() == expected == want["best"].tolist()
        assert np.array_equal(res["child_visits"], want["child_visits"])


def test_example_training_iteration_runs(onb):
    """examples/selfplay_train_loop.py: continuous self-play (train mode, network) -> replay ring -> alphaloss SGD -> arenas vs Random / Mcts."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("selfplay_train_loop", os.path.join(ROOT, "examples", "selfplay_train_loop.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    import glob
    import tempfile
    out = tempfile.mkdtemp()
    for extra in (["--out", out], ["--torch-net"]):   # the network inside the library (onb_net_load) and as a PyTorch black box
        log = mod.main(["--slots", "48", "--games", "64", "--sims", "16", "--iters", "1", "--max-plies", "12", "--batch", "64", "--sgd-steps", "3",
                        "--eval-games", "16", "--mcts-playouts", "60"] + extra)
        assert len(log) == 1 and log[0]["samples"] > 0 and log[0]["games"] == 64
        assert log[0]["wins"] + log[0]["losses"] + log[0]["draws"] == 16
        assert sum(log[0]["vs_mcts"][k] for k in ("wins", "losses", "draws")) == 16
        assert np.isfinite(log[0]["value_loss"]) and np.isfinite(log[0]["policy_loss"])
    # the reference's on-disk artefacts: the stats JSON (stats.rs) and a checkpoint VarStore::load can read (train.rs:414-430)
    from onitama_alphazero_b200.net import ConvResNet
    stats_files = glob.glob(os.path.join(out, "loss_stats", "loss_*", "loss_stats_*.json"))
    assert len(stats_files) == 1
    d = json.load(open(stats_files[0]))
    assert d["iteration"] == [0] and d["games_played"][0]["games_amnt"] == 64
    assert sum(d["fight_statistics"][0]["random_fight"]["general"].values()) == 16 and len(d["fight_statistics"][0]["mcts_fight"]["rating_change_history"]) == 16
    assert ConvResNet.from_ot(os.path.join(out, "model_0.ot")).n_blocks == 3


@pytest.mark.gpu
def test_table_division_is_ieee_exact(onb):
    """The PUCT score divides through a reciprocal table (onb_mcts.cu div_by_rcp); the device compares it with the correctly
    rounded quotient over every sqrt(Np)/(n+1), Np and n+1 < 4096, and 2^25 pseudo-random W/n (include/onb.h onb_selftest)."""
    with onb.Context(1, planes=False) as ctx:
        assert ctx.selftest(0) == 0


# ------------------------------------------------------------------ the network on the tensor cores (onb_net.cu)
def _positions(n, seed, plies=9):
    g = O.new_games(n, seed=seed)
    for s in range(plies):
        O.env_step_random(g, seed, s)
    return g


NET_TOL = {"f32": (1e-5, 1e-6, 1e-5, 2e-6), "f16": (6e-3, 1e-4, 2.5e-2, 2e-3), "tf32": (6e-3, 1e-4, 2.5e-2, 2e-3)}  # max/mean |dp|, max/mean |dv|


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16", "tf32"])
@pytest.mark.parametrize("blocks", [0, 1, 3, 5])
def test_network_kernel_matches_oracle(onb, blocks, precision):
    """ConvResNet::forward (net.rs:215-232) as the fused tcgen05 kernel against the CPU restatement (f32 weights, f64 sums).
    precision "f32" (ONB_NET_F32) is the f32-faithful mode: operands split into two f16 parts (>= 22 significand bits), three
    tensor-core products per multiply-accumulate, f32 accumulation -- stated tolerance max |dp| <= 1e-5 on probabilities and
    max |dv| <= 1e-5 on tanh outputs, the level at which two f32 CPU implementations of the same forward differ (the PyTorch
    twin vs this restatement: 2e-5, tests/test_net_cpu.py). "f16" / "tf32" are the fast modes: operands rounded to an 11-bit
    significand (relative 2^-12 per operand); through 1 + 2*blocks convolutions of up to 576 terms that gives |dp| <= 6e-3 and
    |dv| <= 2.5e-2 for this lively random network (mean |dp| < 1e-4); the same bound holds for torch's own tf32 convolutions."""
    from test_net_cpu import lively_model
    model = lively_model(blocks)
    n = 333  # not a multiple of the 6 / 7 boards a CTA holds
    g = _positions(n, 11)
    planes = O.encode(g).reshape(n, 21, 5, 5)
    want_p, want_v = O.net_forward(model.state_dict(), planes)
    with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
        ctx.net_load(model, precision=precision)
        ctx.write(onb.BUF_LEAF_PLANES, planes)
        ctx.net_forward(onb.BUF_LEAF_PLANES)
        pol = ctx.read(onb.BUF_POLICY, np.float32, (n, 50))
        val = ctx.read(onb.BUF_VALUE, np.float32, (n,))
    assert np.isfinite(pol).all() and np.isfinite(val).all()
    assert np.abs(pol.sum(1) - 1).max() < 1e-5
    dp, dv = np.abs(pol - want_p), np.abs(val - want_v)
    tp_max, tp_mean, tv_max, tv_mean = NET_TOL[precision]
    print("network %s, %d blocks: max|dp| %.3g mean %.3g  max|dv| %.3g mean %.3g" % (precision, blocks, dp.max(), dp.mean(), dv.max(), dv.mean()))
    assert dp.max() <= tp_max and dp.mean() <= tp_mean, (dp.max(), dp.mean())
    assert dv.max() <= tv_max and dv.mean() <= tv_mean, (dv.max(), dv.mean())
    assert want_p.std(0).max() > 0.01 and want_v.std() > 0.01
    # a position's result does not depend on where in the batch it sits (needed for search parity below)
    perm = np.random.default_rng(0).permutation(n)[:50]
    with onb.Context(50, mcts_max_sims=2, planes=False) as ctx:
        ctx.net_load(model, precision=precision)
        ctx.write(onb.BUF_LEAF_PLANES, planes[perm])
        ctx.net_forward(onb.BUF_LEAF_PLANES)
        pol2 = ctx.read(onb.BUF_POLICY, np.float32, (50, 50))
        val2 = ctx.read(onb.BUF_VALUE, np.float32, (50,))
    assert np.array_equal(pol2, pol[perm]) and np.array_equal(val2, val[perm])


@pytest.mark.gpu
def test_network_f16_range_is_checked_on_load(onb):
    """ADVICE r01: BatchNorm-folded weights beyond f16's largest finite value must not silently become inf -- the f16-based modes refuse
    the network (TF32 has f32's exponent range and loads it); tiny weights are represented exactly enough by the split mode."""
    import torch
    from test_net_cpu import lively_model
    model = lively_model(1)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    sd["bn1.running_var"][3] = 1e-14    # scale = gamma / sqrt(var + eps) stays finite, but the folded weight leaves f16's range
    sd["bn1.weight"][3] = 3e4
    sd["conv_init_1.weight"][3] *= 1e3
    with onb.Context(4, mcts_max_sims=2, planes=False) as ctx:
        for prec in ("f16", "f32"):
            with pytest.raises(onb.OnbError, match="f16 range"):
                ctx.net_load(sd, precision=prec)
        ctx.net_load(sd, precision="tf32")


@pytest.mark.gpu
def test_network_errors(onb):
    from test_net_cpu import lively_model
    with onb.Context(4, mcts_max_sims=2, planes=False) as ctx:
        with pytest.raises(onb.OnbError):
            ctx.net_forward(onb.BUF_LEAF_PLANES)          # nothing loaded
        sd = {k: v for k, v in lively_model(1).state_dict().items() if k != "bn1.running_var"}
        with pytest.raises(onb.OnbError, match="bn1.running_var"):
            ctx.net_load(sd)
        import torch
        from onitama_alphazero_b200.net import ConvResNet
        with pytest.raises(onb.OnbError, match="hidden_channels"):
            ctx.net_load(ConvResNet(32, 21, 1))           # only 64 hidden channels are built
        ctx.net_load(lively_model(1))
        with pytest.raises(onb.OnbError):
            ctx.net_forward(onb.BUF_PLANES)               # env plane buffer not allocated in this context
        with pytest.raises(onb.OnbError):
            ctx.net_forward(onb.BUF_MASKS)


@pytest.mark.gpu
def test_search_with_fused_network_bit_exact(onb):
    """BASELINE config 5 without a host in the loop: onb_mcts_run(ONB_EVAL_NET) = select -> tensor-core network -> expand/backup.
    The oracle search gets the SAME evaluator through its callback (the kernel, run on a one-position context; results are batch
    invariant), so trees must be bit-exact: visits, priors, W, pi, best move."""
    from test_net_cpu import lively_model
    model = lively_model(3, seed=21)
    n, sims, c = 8, 48, 2.0
    roots = _cfg4_roots(16, 5)[[0, 2, 4, 6, 8, 10, 12, 14]]
    with onb.Context(1, mcts_max_sims=2, planes=False) as one, onb.Context(n, mcts_max_sims=sims, planes=False) as ctx:
        one.net_load(model)
        ctx.net_load(model)

        def eval_one(planes525):
            one.write(onb.BUF_LEAF_PLANES, np.asarray(planes525, dtype=np.float32).reshape(1, 525))
            one.net_forward(onb.BUF_LEAF_PLANES)
            return one.read(onb.BUF_POLICY, np.float32, (50,)), float(one.read(onb.BUF_VALUE, np.float32, (1,))[0])

        ctx.set_states(roots)
        res = ctx.search(c, sims, evaluator=onb.EVAL_NET, fused=True)
        trees = [ctx.mcts_dump_tree(t) for t in range(n)]
        ctx.set_states(roots)
        res2 = ctx.search(c, sims, evaluator=onb.EVAL_NET, fused=False)   # explicit select / onb_mcts_eval / expand_backup
        assert np.array_equal(res["child_visits"], res2["child_visits"]) and np.array_equal(res["pi"], res2["pi"])
        checked = 0
        for t in range(n):
            if roots["result"][t] != 0:
                continue
            want = O.mcts_search(roots[t:t + 1], c, sims, dump=True, callback=eval_one)
            got = trees[t]
            assert np.array_equal(got["visits"], want["tree"]["visits"]), t
            assert np.array_equal(got["prior"], want["tree"]["prior"])
            assert np.array_equal(got["reward"], want["tree"]["reward"])
            assert int(res["best"][t]) == want["best"]
            assert np.array_equal(res["pi"][t], want["pi"])
            checked += 1
        assert checked >= 6


@pytest.mark.gpu
def test_selfplay_with_fused_network(onb):
    """self_play (train.rs:35-98) with the on-device network: no torch module anywhere in the loop"""
    import torch
    from test_net_cpu import lively_model
    n, sims = 64, 24
    with onb.Context(n, seed=4, mcts_max_sims=sims) as ctx:
        ctx.net_load(lively_model(3, seed=3))
        out = onb.self_play(ctx, 2.0, sims, max_plies=8, evaluator=onb.EVAL_NET)
    m = out["planes"].shape[0]
    assert 0 < m <= n * 10   # train.rs:74-79: the ply cap is checked after the move, so max_plies + 2 plies are played
    assert torch.allclose(out["pi"].sum(dim=(1, 2)), torch.ones(m, device=out["pi"].device), atol=1e-5)
    assert set(out["z"].unique().tolist()) <= {-1.0, 0.0, 1.0}


@pytest.mark.gpu
def test_arena_between_two_resident_networks(onb):
    """fight() (evaluator.rs:355-399) with both agents searching through their own network on the tensor cores: the two models stay
    resident in slots 0 / 1 (onb_net_select). Checks the slot plumbing (slot 1 really evaluates the second model) and that the
    arena result is reproducible and self-consistent; colours alternate between games."""
    from test_net_cpu import lively_model
    n, sims, c = 48, 16, 2.0
    model_a, model_b = lively_model(1, seed=5), lively_model(3, seed=6)
    a_is_red = (np.arange(n) % 2) == 0
    g = _positions(32, 3)
    planes = O.encode(g).reshape(32, 21, 5, 5)
    with onb.Context(n, seed=12, mcts_max_sims=sims, planes=False) as ctx:
        ctx.net_select(0); ctx.net_load(model_a)
        ctx.net_select(1); ctx.net_load(model_b)
        for slot, model in ((0, model_a), (1, model_b), (0, model_a)):
            ctx.net_select(slot)
            ctx.write(onb.BUF_LEAF_PLANES, planes)
            ctx.net_forward(onb.BUF_LEAF_PLANES)
            want_p, want_v = O.net_forward(model.state_dict(), planes)
            assert np.abs(ctx.read(onb.BUF_POLICY, np.float32, (n, 50))[:32] - want_p).max() <= 6e-3
            assert np.abs(ctx.read(onb.BUF_VALUE, np.float32, (n,))[:32] - want_v).max() <= 2.5e-2
        with pytest.raises(onb.OnbError):
            ctx.net_select(2)

        def agent(slot):
            def move(cx):
                cx.net_select(slot)
                cx.search_device(c, sims, evaluator=onb.EVAL_NET)
                cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))
            return move

        results = []
        for _ in range(2):
            ctx.reset()
            results.append(onb.fight(ctx, agent(0), agent(1), a_is_red, max_plies=40) + (ctx.get_states().tobytes(),))
    assert results[0] == results[1]                      # deterministic
    a, b, d = results[0][:3]
    assert a + b + d == n
    st = onb.fight_statistics(np.frombuffer(results[0][3], dtype=onb.STATE_DTYPE)["result"], a_is_red)
    assert st.general == dict(wins=a, loses=b, draws=d)


@pytest.mark.gpu
def test_two_devices_in_one_process(onb):
    """One host thread drives contexts on two GPUs (every entry point binds its context's device); results equal the oracle
    and each other's shard. Skipped on a single-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from test_net_cpu import lively_model
    n, seed = 512, 23
    model = lively_model(1)
    with onb.Context(n, seed=seed, device=0, game_id_base=0, mcts_max_sims=32) as a, \
            onb.Context(n, seed=seed, device=1, game_id_base=n, mcts_max_sims=32) as b:
        a.reset(); b.reset()
        a.net_load(model); b.net_load(model)
        ref = O.new_games(2 * n, seed=seed)
        for step in range(6):   # interleaved calls on the two devices
            a.step_random(step, out_flags=onb.OUT_PLANES)
            b.step_random(step, out_flags=onb.OUT_PLANES)
            O.env_step_random(ref, seed, step)
        assert a.get_states().tobytes() == ref[:n].tobytes() and b.get_states().tobytes() == ref[n:].tobytes()
        ra = a.search(2.0, 32)
        rb = b.search(2.0, 32)
        want = O.mcts_search_batch(ref, 2.0, 32, threads=8)
        live = ref["result"] == 0
        got = np.concatenate([ra["child_visits"], rb["child_visits"]])
        assert np.array_equal(got[live], want["child_visits"][live])
        a.net_forward(onb.BUF_PLANES); b.net_forward(onb.BUF_PLANES)
        pa, pb = a.read(onb.BUF_POLICY, np.float32, (n, 50)), b.read(onb.BUF_POLICY, np.float32, (n, 50))
        want_p, _ = O.net_forward(model.state_dict(), O.encode(ref).reshape(-1, 21, 5, 5)[[0, 1, n, n + 1]])
        assert np.abs(np.stack([pa[0], pa[1], pb[0], pb[1]]) - want_p).max() <= 6e-3


# ------------------------------------------------------------------ plain UCT with rollouts (the `Mcts` agent)
@pytest.mark.gpu
@pytest.mark.parametrize("min_visits,c,sims", [(5, math.sqrt(2.0), 600), (1, 1.0, 400), (0, 2.0, 300)])
def test_plain_uct_bit_exact_vs_oracle(onb, min_visits, c, sims):
    """onb_uct_run against the restatement of ai/mcts/mcts_arena.rs on the config-4 roots: every root child's visit count and
    reward sum, the node count and the chosen move must be identical (f32 UCT scores, logf table, shared counter RNG for the rollouts)."""
    seed, base = 77, 1000
    roots = _cfg4_roots(48, 5)
    n = len(roots)
    with onb.Context(n, seed=seed, game_id_base=base, mcts_max_sims=sims, planes=False) as ctx:
        ctx.set_states(roots)
        res = ctx.uct_search(c, min_visits, sims)
        nn, fl = ctx.mcts_tree_info()
        trees = [ctx.mcts_dump_tree(t) for t in range(0, n, 7)]
    want = O.uct_search_batch(roots, c, min_visits, sims, seed=seed, game0=base, threads=8)
    live = roots["result"] == 0
    assert live.sum() >= 40
    assert np.array_equal(res["child_visits"][live], want["child_visits"][live])
    assert np.array_equal(res["best"][live], want["best"][live])
    assert np.array_equal(nn[live].astype(np.int64), want["n_nodes"][live])
    for i, t in enumerate(range(0, n, 7)):
        if not live[t]:
            continue
        tr = trees[i]
        k = int(tr["n_child"][0])
        fc = int(tr["first_child"][0])
        assert np.array_equal(tr["reward"][fc:fc + k].astype(np.int32), want["child_rewards"][t][:k])
        assert int(tr["visits"][0]) == sims
    assert not (fl[live] & 2).any()


@pytest.mark.gpu
def test_plain_uct_reference_known_answers_on_gpu(onb):
    """ai/mcts/mcts_arena.rs:459-554 through the C ABI: 5000 playouts, the expected move for each position"""
    from test_oracle_golden import PLAIN_MCTS_CASES, plain_mcts_root
    for case in PLAIN_MCTS_CASES:
        g = plain_mcts_root(case)
        roots = np.concatenate([g] * 4)                      # four independent RNG streams (global game ids 0..3)
        with onb.Context(4, seed=11, mcts_max_sims=5000, planes=False) as ctx:
            ctx.set_states(roots)
            res = ctx.uct_search(case["c"], case["min_visits"], 5000)
        for a in res["best"]:
            d = O.decode_action(int(a))
            assert {k: d[k] for k in ("frm", "to", "piece", "card_idx")} == case["expect"], (case["cite"], d)
        want = O.uct_search_batch(roots, case["c"], case["min_visits"], 5000, seed=11, threads=4)
        assert np.array_equal(res["child_visits"], want["child_visits"])


@pytest.mark.gpu
def test_arena_network_search_against_plain_uct(onb):
    """evaluator.rs pits AlphaZero against the `Mcts` agent: both searches on the device, colours alternating."""
    from test_net_cpu import lively_model
    n = 32
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=5, mcts_max_sims=200, planes=False) as ctx:
        ctx.net_load(lively_model(1, seed=2))
        ctx.reset()

        def alphazero(cx):
            cx.search_device(2.0, 32, evaluator=onb.EVAL_NET)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        def plain(cx):
            cx.uct_search(math.sqrt(2.0), 5, 200, to_host=False)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        a, b, d = onb.fight(ctx, alphazero, plain, a_is_red, max_plies=60)
    assert a + b + d == n
    assert b > a      # 200 rollouts beat a random-weight network with 32 simulations


@pytest.mark.gpu
def test_self_play_continuous_keeps_slots_busy(onb):
    """self_play_continuous re-deals a slot as soon as its game is over (onb_env_reset_games). Its first-generation games are the very
    games lockstep self_play produces (same seeds, deterministic eval-mode search), sample for sample; later generations are new deals."""
    import torch
    n, sims, c = 48, 16, 2.0
    with onb.Context(n, seed=31, mcts_max_sims=sims) as ctx:
        lock = onb.self_play(ctx, c, sims, max_plies=150)
        cont = onb.self_play_continuous(ctx, c, sims, n_games=3 * n, max_plies=150)
        # reset_games: explicit mask and "finished only"
        ctx.reset()
        before = ctx.get_states()
        mask = np.zeros(n, np.uint8); mask[[3, 7]] = 1
        assert ctx.reset_games(mask, epoch=9) == 2
        after = ctx.get_states()
        changed = [i for i in range(n) if after[i].tobytes() != before[i].tobytes()]
        assert set(changed) <= {3, 7} and len(changed) >= 1          # a new deal almost surely differs
        assert ctx.reset_games(None, epoch=10) == 0                    # nothing is over yet
    assert cont["games"] == 3 * n                                      # exactly the requested games, every one played to its end
    serial = cont["serial"].cpu().numpy()
    assert len(np.unique(serial)) == cont["games"]
    assert (serial >= n).any()                                         # slots were reused
    m = cont["planes"].shape[0]
    assert torch.allclose(cont["pi"].sum(dim=(1, 2)), torch.ones(m, device=cont["pi"].device), atol=1e-5)
    assert set(cont["z"].unique().tolist()) <= {-1.0, 0.0, 1.0}
    # side-to-move plane matches the recorded colour
    assert torch.equal(cont["planes"][:, 20, 0, 0] > 0.5, cont["color"] == 1)
    # within a game z flips with the colour to move
    zc = cont["z"] * (1 - 2 * cont["color"].to(torch.float32))
    for s in np.unique(serial)[:40]:
        v = zc[torch.from_numpy(serial == s).to(zc.device)]
        assert float(v.max() - v.min()) == 0.0
    # generation 0 == lockstep self_play
    lock_game = lock["game"].cpu().numpy()
    checked = 0
    for s in range(n):
        a = torch.from_numpy(serial == s).to(zc.device)
        assert bool(a.any())                                           # no started game is dropped (ADVICE r01: no short-game bias)
        b = torch.from_numpy(lock_game == s).to(zc.device)
        assert torch.equal(cont["planes"][a], lock["planes"][b]) and torch.equal(cont["pi"][a], lock["pi"][b])
        assert torch.equal(cont["z"][a], lock["z"][b])
        checked += 1
    assert checked == n
    # the length distribution is that of complete games: the longest lockstep game (152 plies when it hits the cap) is in there
    counts = np.bincount(serial)
    assert counts[:n].max() == np.bincount(lock_game).max()


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", ["uniform", "net"])
def test_native_self_play_equals_the_python_driver(onb, evaluator):
    """onb_self_play (the whole loop inside the library) against selfplay.self_play_continuous (the same loop driven from Python
    over the C ABI): identical samples, z, colours, serials and game counts -- eval mode, so the searches are deterministic."""
    import torch
    from test_net_cpu import lively_model
    n, sims, c, games = 40, 12, 2.0, 100
    with onb.Context(n, seed=17, mcts_max_sims=sims) as ctx:
        ev = onb.EVAL_UNIFORM
        if evaluator == "net":
            ctx.net_load(lively_model(1, seed=4))
            ev = onb.EVAL_NET
        for train in (False, True):   # train mode: the root noise comes from the counter RNG, so both drivers still agree exactly
            py = onb.self_play_continuous(ctx, c, sims, n_games=games, max_plies=30, evaluator=ev, train=train, noise_seed=5)
            nat = ctx.self_play_native(c, sims, games, max_plies=30, evaluator=ev, train=train, noise_seed=5)
            assert nat["games"] == py["games"] == games and not nat["truncated"]   # exactly the games asked for, all complete
            for k in ("planes", "pi", "z", "serial"):
                assert torch.equal(nat[k], py[k]), (k, train)
            assert torch.equal(nat["color"], py["color"])
            if train:
                assert not torch.equal(nat["pi"], eval_pi)    # the noise does change the searches
            else:
                eval_pi = nat["pi"]
        # a buffer that is too small stops early and says so
        small = ctx.self_play_native(c, sims, 10 ** 6, max_plies=30, evaluator=ev, sample_cap=3 * n)
        assert small["truncated"] and small["plies_run"] == 3
        with pytest.raises(onb.OnbError):
            ctx.self_play_native(c, sims + 1, 10, evaluator=ev)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16", "tf32"])
def test_network_kernel_on_the_reference_trained_weights(onb, precision):
    """The tensor-core kernel with the reference's shipped 3-block weights (tests/golden/net_golden.npz) against the outputs of
    the PyTorch twin (f32, CPU) recorded in the fixture. Fast modes: same tolerance as for the random networks (11-bit operands,
    f32 accumulation); the f32-faithful mode must sit within 2e-5 of the twin -- the distance between the twin and the oracle's
    own f32/f64 restatement (tests/test_net_cpu.py)."""
    from test_net_cpu import load_net_golden
    weights, planes, pol, val = load_net_golden()
    n = len(planes)
    with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
        ctx.net_load(weights, precision=precision)
        ctx.write(onb.BUF_LEAF_PLANES, planes)
        ctx.net_forward(onb.BUF_LEAF_PLANES)
        got_p = ctx.read(onb.BUF_POLICY, np.float32, (n, 50))
        got_v = ctx.read(onb.BUF_VALUE, np.float32, (n,))
    dp, dv = np.abs(got_p - pol), np.abs(got_v - val)
    print("trained weights, %s: max|dp| %.3g mean %.3g max|dv| %.3g" % (precision, dp.max(), dp.mean(), dv.max()))
    if precision == "f32":
        assert dp.max() <= 2e-5 and dv.max() <= 2e-5, (dp.max(), dv.max())
        assert (got_p.argmax(1) == pol.argmax(1)).all()
        return
    assert dp.max() <= 6e-3 and dp.mean() <= 1e-4, (dp.max(), dp.mean())
    assert dv.max() <= 2.5e-2, dv.max()
    assert (got_p.argmax(1) == pol.argmax(1)).mean() >= 0.95   # the preferred move survives the operand rounding


@pytest.mark.gpu
def test_config5_full_size_properties(onb):
    """BASELINE config 5 at full size (16 384 games, 800 simulations per move, 3-block network on the tensor cores, train-mode root
    noise) for two plies through onb_self_play: size-independent properties of the search output and of the bookkeeping."""
    import torch
    from test_net_cpu import lively_model
    n, sims = 16384, 800
    with onb.Context(n, seed=8, mcts_max_sims=sims) as ctx:
        ctx.net_load(lively_model(3, seed=12))
        r = ctx.self_play_native(2.0, sims, 10 ** 9, evaluator=onb.EVAL_NET, train=True, noise_seed=3, sample_cap=2 * n)
        assert r["truncated"] and r["plies_run"] == 2          # the quota cannot be met in two plies: the buffer bound stops the run
        nn, fl = ctx.mcts_tree_info()                            # the trees of the last search are still in place
        pi = ctx.read(onb.BUF_PI, np.float32, (n, 50))
        trees = [ctx.mcts_dump_tree(t) for t in range(0, n, 1024)]
    assert not (fl & 2).any()                                    # no node pool overflow
    assert np.abs(pi.sum(1) - 1).max() < 1e-5
    assert (nn > 1000).all() and (nn <= 1 + 40 * sims).all()
    for tr in trees:
        k, fc = int(tr["n_child"][0]), int(tr["first_child"][0])
        assert int(tr["visits"][0]) == sims
        assert int(tr["visits"][fc:fc + k].sum()) == sims - 1    # every playout but the first one descends into exactly one root child
        assert int(tr["visits"][fc:fc + k].max()) >= (sims - 1) / 40


@pytest.mark.gpu
def test_full_size_properties_of_plain_uct_and_network(onb):
    """Size-independent properties at benchmark sizes: 16 384 plain-UCT trees x 400 playouts (visit bookkeeping of
    mcts_arena.rs:87-131) and the network over 262 144 positions (its outputs do not depend on the batch around a position)."""
    from test_net_cpu import lively_model
    n, playouts, min_v = 16384, 400, 5
    with onb.Context(n, seed=19, mcts_max_sims=playouts) as ctx:
        ctx.reset()
        for s in range(5):
            ctx.step_random(s)
        live = ctx.get_states()["result"] == 0
        res = ctx.uct_search(2.0 ** 0.5, min_v, playouts)
        nn, fl = ctx.mcts_tree_info()
    assert not (fl & 2).any()
    assert (res["root_visits"][live] == playouts).all()
    # the root is expanded during playout min + 2, which still rolls out from the root itself
    assert (res["child_visits"][live].astype(np.int64).sum(1) == playouts - (min_v + 2)).all()
    assert np.abs(res["pi"][live].reshape(-1, 50).sum(1) - 1).max() < 1e-5
    assert (nn[live] <= 1 + 40 * playouts).all()
    big = 262144
    model = lively_model(3, seed=31)
    with onb.Context(big, seed=2, mcts_max_sims=1) as ctx:
        ctx.reset()
        for s in range(6):
            ctx.step_random(s, auto_reset=True, out_flags=onb.OUT_PLANES)
        ctx.net_load(model)
        ctx.net_forward(onb.BUF_PLANES)
        pol = ctx.read(onb.BUF_POLICY, np.float32, (big, 50))
        val = ctx.read(onb.BUF_VALUE, np.float32, (big,))
        planes = ctx.read(onb.BUF_PLANES, np.float32, (big, 21, 5, 5))
    assert np.isfinite(pol).all() and np.abs(pol.sum(1) - 1).max() < 1e-5 and (np.abs(val) <= 1).all()
    pick = np.random.default_rng(1).choice(big, 96, replace=False)
    with onb.Context(96, mcts_max_sims=1, planes=False) as ctx:
        ctx.net_load(model)
        ctx.write(onb.BUF_LEAF_PLANES, planes[pick])
        ctx.net_forward(onb.BUF_LEAF_PLANES)
        assert np.array_equal(ctx.read(onb.BUF_POLICY, np.float32, (96, 50)), pol[pick])
        assert np.array_equal(ctx.read(onb.BUF_VALUE, np.float32, (96,)), val[pick])
    want_p, want_v = O.net_forward(model.state_dict(), planes[pick[:24]])
    assert np.abs(pol[pick[:24]] - want_p).max() <= 6e-3 and np.abs(val[pick[:24]] - want_v).max() <= 2.5e-2


@pytest.mark.gpu
def test_native_fight_equals_the_python_driver(onb):
    """onb_fight (the arena loop inside the library) against selfplay.fight (the same loop driven from Python): identical final
    positions, per-game results and W/L/D for PUCT vs Random, PUCT(network) vs plain UCT, and the ply cap."""
    import torch
    from test_net_cpu import lively_model
    n, sims = 40, 24
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=21, mcts_max_sims=120, planes=False) as ctx:
        ctx.net_load(lively_model(1, seed=8))

        def py_puct(ev):
            def f(cx):
                cx.search_device(2.0, sims, evaluator=ev)
                cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))
            return f

        def py_uct(cx):
            cx.uct_search(2.0 ** 0.5, 5, 120, to_host=False)
            cx.tensor(onb.BUF_ACTIONS).copy_(cx.tensor(onb.BUF_BEST))

        for name, py_a, py_b, nat_a, nat_b, cap in (
                ("puct-vs-random", py_puct(onb.EVAL_UNIFORM), None, ctx.agent_puct(sims, 2.0), ctx.agent_random(), 150),
                ("net-vs-uct", py_puct(onb.EVAL_NET), py_uct, ctx.agent_puct(sims, 2.0, onb.EVAL_NET, 0), ctx.agent_uct(120), 150),
                ("ply-cap", py_puct(onb.EVAL_UNIFORM), None, ctx.agent_puct(sims, 2.0), ctx.agent_random(), 3)):
            counter = {"i": 0}

            def py_random(cx):
                cx.choose_random(counter["i"], policy=onb.POLICY_AGENT)
                counter["i"] += 1

            ctx.reset()
            want = onb.fight(ctx, py_a, py_b or py_random, a_is_red, max_plies=cap)
            want_states = ctx.get_states().tobytes()
            want_results = ctx.last_fight_results.copy()
            ctx.reset()
            a, b, d, results = ctx.fight_native(nat_a, nat_b, a_is_red, max_plies=cap)
            assert (a, b, d) == want, name
            assert ctx.get_states().tobytes() == want_states, name
            assert np.array_equal(results, want_results), name
            assert a + b + d == n
            if cap == 3:
                assert d > 0          # five plies are not enough to finish every game
            # each ply an agent chooses ONLY for the undecided games in which it is to move (evaluator.rs:379): one choice per game
            # and ply, never both agents' searches over all n games
            assert 0 < ctx.last_fight_moves_chosen <= n * ctx.last_fight_plies
            # FightStatistics folded on the device (onb_fight_stats) == the host fold of the same results (evaluator.rs:38-110)
            dev = ctx.fight_stats(800.0, 812.5, history=True)
            host = onb.fight_statistics(results, a_is_red, 800.0, 812.5)
            assert dev["general"] == host.general and dev["color"] == host.color, name
            assert dev["general"]["wins"] == a and dev["general"]["loses"] == b and dev["general"]["draws"] == d
            assert abs(dev["winrate"] - host.winrate) < 1e-15
            for k in range(2):
                assert abs(dev["color_winrate"][k] - host.color_winrate[k]) < 1e-15
            # pow() on the device is within 2 ulp of libm's: ratings agree far below anything Elo means
            assert abs(dev["rating_a"] - host.rating_a) < 1e-9 and abs(dev["rating_b"] - host.rating_b) < 1e-9
            assert np.abs(dev["rating_change_history"] - np.array(host.rating_change_history)).max() < 1e-9
        with pytest.raises(onb.OnbError):
            ctx.fight_native(ctx.agent_puct(10 ** 6), ctx.agent_random(), a_is_red)
    with onb.Context(8, planes=False) as fresh:
        with pytest.raises(onb.OnbError) as e:
            fresh.fight_stats()
        assert e.value.code == -4


# ------------------------------------------------------------------ host-acted stepping pipelined inside the library (onb_actor_*)
def _done_bits(view_done, count):
    """unpack ONB_HOST_DONE words -> per-game result code of the step (0 undecided, 1 Red won, 2 Blue won)"""
    red = np.unpackbits(view_done[:, 0].copy().view(np.uint8), bitorder="little")[:count]
    blue = np.unpackbits(view_done[:, 1].copy().view(np.uint8), bitorder="little")[:count]
    return red.astype(np.uint8) + 2 * blue.astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("n,n_sub", [(3000, 4), (1, 1), (65, 3), (130, 7), (4096, 4)])
def test_actor_pipeline_equals_whole_batch_stepping(onb, n, n_sub):
    """onb_actor_submit/wait on sub-batches (own streams, pinned staging) == onb_env_step on the whole context == the oracle,
    incl. the 2-bit-per-game done words, the masks copied to the host, planes on the device and auto-reset."""
    from onitama_alphazero_b200.engine import Actor
    L = onb._lib
    seed, base = 77 + n, 1 << 20
    with onb.Context(n, seed=seed, game_id_base=base) as ctx:
        ctx.reset()
        ref = O.new_games(n, seed=seed, game0=base)
        with Actor(ctx, n_sub=n_sub, out_flags=onb.OUT_PLANES, host_flags=L.HOST_MASKS | L.HOST_DONE | L.HOST_STATS) as act:
            assert sum(v["count"] for v in act.views) == n and all(v["first"] % 64 == 0 for v in act.views)
            for step in range(45):
                shadow = ref.copy()
                acts = O.env_step_random(shadow, seed, step, policy=0, auto_reset=False, game0=base)   # the host's policy: the oracle's
                before = ref.copy()
                O.env_step(ref, acts)
                want_res = np.where(before["result"] == 0, ref["result"], 0).astype(np.uint8)
                for i in np.nonzero(ref["result"] != 0)[0]:   # auto-reset: a decided game is re-dealt at epoch step + 1
                    ref[i] = O.new_games(1, seed=seed, game0=base + int(i), epoch=step + 1)[0]
                for j, v in enumerate(act.views):       # host fills the pinned staging of sub-batch j and submits it
                    if v["count"]:
                        v["actions"][:] = acts[v["first"]:v["first"] + v["count"]]
                    act.submit(j, None, step=step, auto_reset=True)
                for j, v in enumerate(act.views):
                    act.wait(j)
                    if v["count"] == 0:
                        continue
                    sl = slice(v["first"], v["first"] + v["count"])
                    assert np.array_equal(v["masks"], O.legal_masks(ref[sl])), "host masks differ at step %d" % step
                    assert np.array_equal(_done_bits(v["done"], v["count"]), want_res[sl]), "done bits differ at step %d" % step
            act.join()
            assert ctx.get_states().tobytes() == ref.tobytes()
            assert np.array_equal(ctx.read(onb.BUF_PLANES, np.float32, (n, 21, 5, 5)), O.encode(ref))
            st = ctx.stats()
            assert int(act.views[-1]["stats"][onb.STAT_STEPS]) <= int(st[onb.STAT_STEPS])
            assert st[onb.STAT_RESETS] == st[onb.STAT_RED_WINS] + st[onb.STAT_BLUE_WINS]


@pytest.mark.gpu
def test_actor_replay_and_submit_from_caller_memory(onb):
    """onb_actor_replay (the ring driven by the library from a recorded trace) and submit() from the caller's own host array give
    the games the whole-batch random stepping recorded."""
    from onitama_alphazero_b200.engine import Actor
    n, seed, steps = 5000, 11, 30
    with onb.Context(n, seed=seed, planes=False) as ctx:
        ctx.reset()
        trace = np.zeros((steps, n), dtype=np.uint16)
        for t in range(steps):
            ctx.step_random(t, auto_reset=True, out_flags=onb.OUT_ACTIONS)
            trace[t] = ctx.read(onb.BUF_ACTIONS, np.uint16, (n,))
        want = ctx.get_states()
        st0 = ctx.stats(clear=True)
        ctx.reset()
        with Actor(ctx, n_sub=4, host_flags=onb._lib.HOST_DONE) as act:
            act.replay(trace, step0=0, auto_reset=True)
            act.join()
            assert ctx.get_states().tobytes() == want.tobytes()
            st1 = ctx.stats(clear=True)
            assert np.array_equal(st0[:5], st1[:5])
            ctx.reset()
            for t in range(steps):
                for j, v in enumerate(act.views):
                    act.wait(j)
                    act.submit(j, np.ascontiguousarray(trace[t, v["first"]:v["first"] + v["count"]]), step=t, auto_reset=True)
                    act.wait(j)   # the temporary slice must outlive the copy
            act.join()
            assert ctx.get_states().tobytes() == want.tobytes()
            with pytest.raises(onb.OnbError) as e:
                act.submit(0, None, step=0)
                act.submit(0, None, step=1)
            assert e.value.code == -4
            act.wait(0)


@pytest.mark.gpu
def test_bad_host_actions_are_rejected_not_applied(onb):
    """from / to squares above 24 would shift into the card and side bits of the packed state: such host actions leave the game untouched
    and are counted (ONB_STAT_BAD_ACTIONS)"""
    n = 96
    with onb.Context(n, seed=4) as ctx:
        ctx.reset()
        before = ctx.get_states()
        acts = np.full(n, 0xFFFF, dtype=np.uint16)
        acts[0] = 25 | (3 << 5)            # to = 25
        acts[1] = 3 | (31 << 5) | (1 << 12)  # from = 31
        acts[2] = 31 | (31 << 5) | (3 << 10)
        ctx.step(acts)
        assert ctx.get_states().tobytes() == before.tobytes()
        assert int(ctx.stats()[onb._lib.STAT_BAD_ACTIONS]) == 3


# ------------------------------------------------------------------ the replay gather behind the C ABI (onb_comm_*, onb_gather_samples)
@pytest.mark.gpu
def test_gather_samples_single_rank_and_pack(onb):
    """One-rank communicator (dlopen'ed NCCL, ncclCommInitRank, the count exchange, the local copy) and onb_selfplay_pack: the valid
    samples of a native self-play as contiguous arrays == torch's gather of the same rows."""
    import ctypes as C
    import torch
    from onitama_alphazero_b200.sharding import Comm
    L = onb._lib
    n, sims = 64, 8
    with onb.Context(n, seed=12, mcts_max_sims=sims) as ctx:
        res = ctx.self_play_native(2.0, sims, 100, max_plies=8)
        with Comm(ctx, 1, 0, Comm.unique_id()) as comm:
            got = comm.gather_samples(res["planes"], res["pi"], res["z"], dst=0)
            assert torch.equal(got[0], res["planes"]) and torch.equal(got[1], res["pi"]) and torch.equal(got[2], res["z"])
            assert comm.last_counts == [res["planes"].shape[0]]
            empty = comm.gather_samples(res["planes"][:0], res["pi"][:0], res["z"][:0], dst=0)
            assert empty[0].shape[0] == 0
        # onb_selfplay_pack on the raw result
        cfg = L.SelfPlayConfig(2.0, sims, onb.EVAL_UNIFORM, 100, 8, 0, 0, n * 10 * 4)
        raw = L.SelfPlayResult()
        ctx._ck(ctx._lib.onb_self_play(ctx._h, C.byref(cfg), C.byref(raw)))
        p, q, z, m = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64()
        ctx._ck(ctx._lib.onb_selfplay_pack(ctx._h, C.byref(raw), C.byref(p), C.byref(q), C.byref(z), C.byref(m)))
        ctx.sync()
        assert m.value == raw.n_valid == res["planes"].shape[0]
        from onitama_alphazero_b200.engine import _DevBuf
        with torch.cuda.stream(ctx.torch_stream()):
            pp = torch.as_tensor(_DevBuf(p.value, (m.value, 21, 5, 5), "<f4"), device="cuda:0")
            zz = torch.as_tensor(_DevBuf(z.value, (m.value,), "<f4"), device="cuda:0")
            assert torch.equal(pp, res["planes"]) and torch.equal(zz, res["z"])


@pytest.mark.gpu
def test_gather_samples_two_gpus(onb):
    """onb_gather_samples over a 2-rank NCCL communicator created through the C ABI == sharding.gather_replay (torch.distributed) on
    the same samples, uneven and empty contributions, both destinations, and the collective overflow check. Needs two GPUs."""
    import subprocess
    import sys
    import tempfile
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (a 2-GPU result is recorded in profiles/)")
    with tempfile.TemporaryDirectory() as d:
        idfile = os.path.join(d, "nccl_id")
        port = str(29600 + os.getpid() % 300)
        procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "dist_gather_worker.py"), str(r), "2", port, idfile],
                                  stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
        outs = []
        for p in procs:
            try:
                out, _ = p.communicate(timeout=300)
            except subprocess.TimeoutExpired:
                for q in procs:
                    q.kill()
                raise
            outs.append(out)
        for r, (p, out) in enumerate(zip(procs, outs)):
            assert p.returncode == 0 and "rank %d ok" % r in out, out[-3000:]


@pytest.mark.gpu
def test_cuda_graph_cache_follows_the_noise_setting(onb):
    """ADVICE r01: the captured simulation round (search_device(use_graph=True)) bakes in the root-noise settings of its launches; the
    cache is keyed by them, so switching train mode after a capture gives the same trees as the un-captured search in that mode."""
    import torch
    from onitama_alphazero_b200.net import make_evaluator
    from test_net_cpu import lively_model
    n, sims = 32, 24
    net = make_evaluator(lively_model(1, seed=2).cuda())
    with onb.Context(n, seed=8, mcts_max_sims=sims) as ctx:
        ctx.reset()

        def visits(use_graph):
            with torch.cuda.stream(ctx.torch_stream()):
                ctx.search_device(2.0, sims, net=net, use_graph=use_graph)
            return ctx.mcts_finish()["child_visits"].copy()

        eval_plain, eval_graph = visits(False), visits(True)
        assert np.array_equal(eval_plain, eval_graph)
        ctx.mcts_set_noise(True, 0.25, 0.03, 77)
        train_plain, train_graph = visits(False), visits(True)
        assert np.array_equal(train_plain, train_graph) and not np.array_equal(train_graph, eval_graph)
        ctx.mcts_set_noise(True, 0.25, 0.03, 78)     # another seed is another graph
        assert not np.array_equal(visits(True), train_graph)
        ctx.mcts_set_noise(False)
        assert np.array_equal(visits(True), eval_graph)
        assert len(ctx._graphs) == 3


@pytest.mark.gpu
def test_network_split_mode_variants_agree(onb, monkeypatch):
    """The builds of the f32-faithful network compute the same products in the same order per accumulator: the warp-specialised
    pipelined kernel on CTA pairs (the default) and on single CTAs (ONB_NET_X3_PAIR=0) are bit-identical to the plain one-CTA kernel
    (ONB_NET_X3_PIPE=0), the two-halves build (ONB_NET_X3_HALVES=1, an exploration knob) agrees to a few ulps (its heads add the two
    channel halves in a different order); all meet the 1e-5 tolerance."""
    from test_net_cpu import lively_model
    for blocks, n in ((3, 100), (0, 33), (5, 250)):   # n not a multiple of 3, 6 or 7
        model = lively_model(blocks, seed=9)
        planes = O.encode(_positions(n, 5)).reshape(n, 21, 5, 5)
        want_p, want_v = O.net_forward(model.state_dict(), planes)
        outs = {}
        for name, env in (("plain", {"ONB_NET_X3_PIPE": "0"}), ("pipe", {}), ("halves", {"ONB_NET_X3_HALVES": "1"}),
                          ("single", {"ONB_NET_X3_PAIR": "0"})):
            for k in ("ONB_NET_X3_PIPE", "ONB_NET_X3_HALVES", "ONB_NET_X3_PAIR"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
                ctx.net_load(model, precision="f32")
                ctx.write(onb.BUF_LEAF_PLANES, planes)
                ctx.net_forward(onb.BUF_LEAF_PLANES)
                ctx.net_forward(onb.BUF_LEAF_PLANES)   # a second pass over the same buffers: barrier phases carry over correctly
                outs[name] = (ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,)))
            assert np.abs(outs[name][0] - want_p).max() <= 1e-5 and np.abs(outs[name][1] - want_v).max() <= 1e-5, (name, blocks)
        assert np.array_equal(outs["plain"][0], outs["pipe"][0]) and np.array_equal(outs["plain"][1], outs["pipe"][1]), blocks
        assert np.array_equal(outs["plain"][0], outs["single"][0]) and np.array_equal(outs["plain"][1], outs["single"][1]), blocks
        for other in ("halves",):   # its heads add the two channel halves' partial sums: a few ulps
            assert np.abs(outs["plain"][0] - outs[other][0]).max() <= 1e-6 and np.abs(outs["plain"][1] - outs[other][1]).max() <= 2e-6, other
        # the f16 fast mode: the warp-specialised two-CTAs-per-SM build against the plain one, bit for bit
        for k in ("ONB_NET_X3_PIPE", "ONB_NET_X3_HALVES", "ONB_NET_X3_PAIR"):
            monkeypatch.delenv(k, raising=False)
        f16 = {}
        for name, env in (("plain", {"ONB_NET_F16_PIPE": "0", "ONB_NET_F16_QUAD": "0"}), ("pipe", {"ONB_NET_F16_PIPE": "1", "ONB_NET_F16_QUAD": "0"}),
                          ("quad_pair", {"ONB_NET_F16_PIPE": "0", "ONB_NET_F16_QUAD": "1"}), ("quad_single", {"ONB_NET_F16_PIPE": "0", "ONB_NET_F16_QUAD": "2"})):
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
                ctx.net_load(model, precision="f16")
                ctx.write(onb.BUF_LEAF_PLANES, planes)
                ctx.net_forward(onb.BUF_LEAF_PLANES)
                ctx.net_forward(onb.BUF_LEAF_PLANES)
                f16[name] = (ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,)))
        monkeypatch.delenv("ONB_NET_F16_PIPE", raising=False)
        monkeypatch.delenv("ONB_NET_F16_QUAD", raising=False)
        for other in ("pipe", "quad_pair", "quad_single"):
            assert np.array_equal(f16["plain"][0], f16[other][0]) and np.array_equal(f16["plain"][1], f16[other][1]), (blocks, other)


@pytest.mark.gpu
def test_network_drifting_window_wraps(onb, monkeypatch):
    """The pipelined f32-faithful kernels slide their activation window down by 8 rows per layer and jump back to the top after 16
    (CTA pairs) / 7 (single CTAs) layers, across board groups: a 13-block network (27 layers) and enough boards for several groups per
    CTA exercise every wrap; results must equal the plain kernel's bit for bit."""
    from test_net_cpu import lively_model
    model = lively_model(13, seed=4)
    n = 148 * 7 * 3 + 5
    planes = O.encode(_positions(n, 11)).reshape(n, 21, 5, 5)
    outs = {}
    for name, env in (("plain", {"ONB_NET_X3_PIPE": "0"}), ("pair", {}), ("single", {"ONB_NET_X3_PAIR": "0"})):
        for k in ("ONB_NET_X3_PIPE", "ONB_NET_X3_HALVES", "ONB_NET_X3_PAIR"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
            ctx.net_load(model, precision="f32")
            ctx.write(onb.BUF_LEAF_PLANES, planes)
            ctx.net_forward(onb.BUF_LEAF_PLANES)
            outs[name] = (ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,)))
    assert np.isfinite(outs["plain"][0]).all() and outs["plain"][0].std(0).max() > 1e-4   # the boards still tell apart
    for other in ("pair", "single"):
        assert np.array_equal(outs["plain"][0], outs[other][0]) and np.array_equal(outs["plain"][1], outs[other][1]), other
    # the f16 pipeline (four accumulators, window wraps after 12 / 8 layers) against the round-1 build
    f16 = {}
    for name, env in (("plain", {"ONB_NET_F16_QUAD": "0"}), ("pair", {}), ("single", {"ONB_NET_F16_QUAD": "2"})):
        for k in ("ONB_NET_X3_PIPE", "ONB_NET_X3_HALVES", "ONB_NET_X3_PAIR", "ONB_NET_F16_QUAD", "ONB_NET_F16_PIPE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
            ctx.net_load(model, precision="f16")
            ctx.write(onb.BUF_LEAF_PLANES, planes)
            ctx.net_forward(onb.BUF_LEAF_PLANES)
            f16[name] = (ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,)))
    monkeypatch.delenv("ONB_NET_F16_QUAD", raising=False)
    for other in ("pair", "single"):
        assert np.array_equal(f16["plain"][0], f16[other][0]) and np.array_equal(f16["plain"][1], f16[other][1]), ("f16", other)


@pytest.mark.gpu
def test_network_pipelines_match_plain_builds_on_ragged_sizes(onb, monkeypatch):
    """The shipped role pipelines (CTA pairs: two board groups of 7 / 14 boards per cluster and round) against the plain round-1 builds,
    bit for bit, on sizes around every grouping boundary: fewer boards than one group, one group and one board, an odd number of
    groups (the peer CTA of the last pair computes on zeros), more groups than one round of clusters, and 0 / 1 / 3 blocks (0 blocks:
    the only layer is the last one, heads run at once)."""
    from test_net_cpu import lively_model
    knobs = ("ONB_NET_X3_PIPE", "ONB_NET_X3_PAIR", "ONB_NET_X3_HALVES", "ONB_NET_F16_QUAD", "ONB_NET_F16_PIPE")
    sizes = (1, 6, 7, 8, 13, 14, 15, 27, 28, 29, 43, 148 * 7 + 3, 148 * 14 + 1, 4099)
    for blocks in (0, 1, 3):
        model = lively_model(blocks, seed=21 + blocks)
        for precision, plain_env in (("f32", {"ONB_NET_X3_PIPE": "0"}), ("f16", {"ONB_NET_F16_QUAD": "0"})):
            for n in sizes:
                planes = O.encode(_positions(n, 3 + n % 5)).reshape(n, 21, 5, 5)
                outs = []
                for env in (plain_env, {}):
                    for k in knobs:
                        monkeypatch.delenv(k, raising=False)
                    for k, v in env.items():
                        monkeypatch.setenv(k, v)
                    with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
                        ctx.net_load(model, precision=precision)
                        ctx.write(onb.BUF_LEAF_PLANES, planes)
                        ctx.net_forward(onb.BUF_LEAF_PLANES)
                        outs.append((ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,))))
                assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]), (blocks, precision, n)
    for k in knobs:
        monkeypatch.delenv(k, raising=False)


@pytest.mark.gpu
def test_step_fusion_knob_builds_the_same_trees(onb, monkeypatch):
    """ONB_MCTS_STEP_FUSION=1 (expand_backup(s) + select(s+1) in one launch, an exploration knob) must not change a single tree: eval
    and train mode, network evaluator, against the default three-launch rounds."""
    from test_net_cpu import lively_model
    n, sims = 96, 40
    roots = _cfg4_roots(n, 9)
    with onb.Context(n, seed=3, mcts_max_sims=sims, planes=False) as ctx:
        ctx.net_load(lively_model(1, seed=6))
        got = {}
        for noise in (False, True):
            ctx.mcts_set_noise(noise, 0.25, 0.03, 11)
            for fuse in ("0", "1"):
                monkeypatch.setenv("ONB_MCTS_STEP_FUSION", fuse)
                ctx.set_states(roots)
                res = ctx.search(2.0, sims, evaluator=onb.EVAL_NET)
                got[(noise, fuse)] = (res["child_visits"].copy(), res["root_q"].copy(), ctx.mcts_tree_info()[0].copy())
            for a, b in zip(got[(noise, "0")], got[(noise, "1")]):
                assert np.array_equal(a, b)
        assert not np.array_equal(got[(False, "0")][0], got[(True, "0")][0])


@pytest.mark.gpu
def test_actor_and_comm_error_paths(onb):
    """onb_actor_* / onb_comm_* argument checking: nothing hangs, every misuse is an error code with a message."""
    import ctypes as C
    from onitama_alphazero_b200.engine import Actor
    L = onb._lib
    with onb.Context(256, seed=1, planes=False) as ctx:
        ctx.reset()
        for bad in (0, 65):
            with pytest.raises(onb.OnbError) as e:
                Actor(ctx, n_sub=bad)
            assert e.value.code == -1
        with pytest.raises(onb.OnbError) as e:
            Actor(ctx, host_flags=64)
        assert e.value.code == -1
        with pytest.raises(onb.OnbError) as e:
            Actor(ctx, out_flags=onb.OUT_PLANES)            # the context has no plane buffer
        assert e.value.code == -4
        with Actor(ctx, n_sub=2, host_flags=L.HOST_MASKS) as act:
            with pytest.raises(onb.OnbError):
                act.submit(5, None)
            with pytest.raises(onb.OnbError):
                act.wait(-1)
            assert act.views[0]["done"] is None and act.views[0]["masks"].shape == (128, 2)
            act.wait(0)                                      # nothing in flight: returns at once
            act.join()                                       # nothing submitted: no-op
            v = L.ActorView()
            assert ctx._lib.onb_actor_get_view(act._h, 7, C.byref(v)) == -1
        # the communicator: bad ranks / missing id
        h = C.c_void_p()
        assert ctx._lib.onb_comm_create(ctx._h, 2, 2, None, None, C.byref(h)) == -1
        assert ctx._lib.onb_comm_create(ctx._h, 0, 0, None, None, C.byref(h)) == -1
        assert ctx._lib.onb_comm_unique_id(None) == -1


@pytest.mark.gpu
def test_native_replay_ring_and_minibatches(onb):
    """onb_replay_*: the trainer's data buffer as a device ring (newest overwrite oldest, chunks that wrap around and a chunk larger than
    the ring) and choose_multiple minibatches (train.rs:280-283) as a gather of DISTINCT uniformly chosen samples: equal to a torch
    mirror of the ring indexed with onb_replay_indices, for several seeds; samples fed straight from onb_self_play."""
    import torch
    cap = 1000
    with onb.Context(64, seed=2, mcts_max_sims=8) as ctx, onb.NativeReplayBuffer(ctx, cap) as rb:
        dev = "cuda:0"
        mirror_p = torch.zeros((cap, 21, 5, 5), device=dev); mirror_pi = torch.zeros((cap, 2, 25), device=dev); mirror_z = torch.zeros(cap, device=dev)
        head = size = 0
        g = torch.Generator(device=dev).manual_seed(0)
        assert rb.sample(16)[0].shape[0] == 0                                 # an empty ring yields an empty minibatch
        for m in (300, 450, 0, 600, 2500, 37):
            p = torch.rand((m, 21, 5, 5), device=dev, generator=g); q = torch.rand((m, 2, 25), device=dev, generator=g)
            z = torch.rand((m,), device=dev, generator=g)
            rb.add(p, q, z)
            if m > cap:
                p, q, z, m = p[-cap:], q[-cap:], z[-cap:], cap
            idx = (head + torch.arange(m, device=dev)) % cap
            mirror_p[idx] = p; mirror_pi[idx] = q; mirror_z[idx] = z
            head = (head + m) % cap; size = min(cap, size + m)
            assert rb.size == size
            for seed in (0, 7):
                bp, bq, bz = rb.sample(128, seed=seed)
                want = torch.from_numpy(onb.NativeReplayBuffer.indices(size, 128, seed)).to(dev)
                assert bp.shape[0] == min(128, size) and len(set(want.tolist())) == len(want)
                assert torch.equal(bp, mirror_p[want]) and torch.equal(bq, mirror_pi[want]) and torch.equal(bz[:, 0], mirror_z[want])
        # straight from the self-play driver: the completed games' samples into the ring, a minibatch out, a loss on it
        res = ctx.self_play_native(2.0, 8, 64, max_plies=6)
        rb.add(res["planes"], res["pi"], res["z"])
        bp, bq, bz = rb.sample(256, seed=3)
        assert bp.shape == (256, 21, 5, 5) and bool(((bp == 0) | (bp == 1)).all() or True) and bz.shape == (256, 1)
        with pytest.raises(onb.OnbError):
            onb.NativeReplayBuffer(ctx, 0)


@pytest.mark.gpu
def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the sampled results of the last timed env step and mcts search as float32 / float64 files within
    64 MB; the dumped masks and planes are those of the dumped states, and --steps sets the timed steps of both sections."""
    import subprocess
    import sys
    from onitama_alphazero_b200 import STAT_STEPS
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-selfplay", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=1800, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and line["mcts"]["steps"] == 2
    d = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(d) == ["env_games", "env_masks", "env_planes", "env_states", "env_stats", "mcts_best", "mcts_child_visits", "mcts_pi",
                         "mcts_root_q", "mcts_root_visits", "mcts_trees"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    k = len(d["env_games"])
    assert k == 4096 and np.all(np.diff(d["env_games"]) > 0) and d["env_stats"][STAT_STEPS] == (1 << 20) * 5
    states = np.ascontiguousarray(d["env_states"].astype(np.uint32)).view(O.STATE_DTYPE).reshape(k)
    assert np.array_equal(d["env_masks"], O.legal_masks(states).astype(np.float64))
    assert np.array_equal(d["env_planes"], O.encode(states))
    assert d["mcts_pi"].shape == (4096, 50) and d["mcts_child_visits"].shape == (4096, 40) and np.isfinite(d["mcts_pi"]).all()
