"""Networks of 128 hidden channels (ConvResNetConfig{hidden_channels: 128}): the PyTorch twin, the CPU oracle and the .ot round trip
at that width, and on the GPU the k_net_wide tensor-core kernel behind onb_net_load / onb_net_forward / ONB_EVAL_NET in all three
precision modes, next to a 64-wide network in the other slot."""
import functools

import numpy as np
import pytest
import torch

import oracle_lib as O

NET_TOL = {"f32": (1e-5, 1e-6, 1e-5, 2e-6), "f16": (6e-3, 1e-4, 2.5e-2, 2e-3), "tf32": (6e-3, 1e-4, 2.5e-2, 2e-3)}  # max/mean |dp|, max/mean |dv|


@pytest.fixture(scope="module")
def onb():
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as m
    return m


def lively_model_wide(blocks=3, seed=7, res_gain=None):
    """lively_model (tests/test_net_cpu.py) at 128 hidden channels: activations of order one in every layer, non-trivial BatchNorm
    statistics, deterministic for a given torch version."""
    from onitama_alphazero_b200.net import ConvResNet
    torch.manual_seed(seed)
    model = ConvResNet(128, 21, blocks)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.Conv2d):
                torch.nn.init.kaiming_normal_(m.weight, nonlinearity="relu")
                m.bias.normal_(0, 0.1)
            if isinstance(m, torch.nn.Linear):
                m.weight.normal_(0, 2.0 / m.in_features ** 0.5)
                m.bias.normal_(0, 0.3)
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
                m.weight.uniform_(0.7, 1.3)
                m.bias.normal_(0.1, 0.2)
        gain = res_gain if res_gain is not None else (1.0 if blocks <= 3 else 0.5)
        if gain != 1.0:
            for name, p in model.named_parameters():
                if "small_block2.small_block_conv.weight" in name:
                    p.mul_(gain)
        if blocks > 3:  # keep tanh and softmax out of saturation (0.05 rather than 0.02: the value output still varies at 5 blocks)
            model.vh_conv.weight.mul_(0.05)
            model.policy_conv.weight.mul_(0.2)
    return model.eval()


def _planes(n, seed, plies=9):
    g = O.new_games(n, seed=seed)
    for s in range(plies):
        O.env_step_random(g, seed, s)
    return O.encode(g).reshape(n, 21, 5, 5)


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("blocks", [0, 1, 3, 5])
def test_oracle_network_matches_the_pytorch_twin_at_width_128(blocks):
    """orc_net_forward reads the width from bn1.weight: at 128 channels it must agree with net.py as closely as at 64"""
    model = lively_model_wide(blocks)
    planes = _planes(24, 5)
    with torch.no_grad():
        p_ref, v_ref = model(torch.from_numpy(planes))
    pol, val = O.net_forward(model.state_dict(), planes)
    assert np.abs(pol - p_ref.reshape(-1, 50).numpy()).max() < 2e-5
    assert np.abs(val - v_ref.reshape(-1).numpy()).max() < 2e-5
    assert p_ref.reshape(-1, 50).std(0).max() > 0.01 and v_ref.std() > 0.01


def test_wide_ot_round_trip_keeps_width_blocks_and_bits(tmp_path):
    from onitama_alphazero_b200.net import ConvResNet
    m = lively_model_wide(2, seed=5)
    back = ConvResNet.from_ot(m.save_ot(str(tmp_path / "wide.ot")))
    assert back.bn1.weight.numel() == 128 and back.n_blocks == 2 and back.vh_linear1.out_features == 128
    sd, sd2 = m.state_dict(), back.state_dict()
    assert sorted(sd) == sorted(sd2)
    for k in sd:
        if not k.endswith("num_batches_tracked"):
            assert torch.equal(sd[k], sd2[k]), k


# ------------------------------------------------------------------ GPU: the kernel against the oracle
@functools.lru_cache(maxsize=None)
def _reference(blocks, n, n_oracle):
    """planes, oracle outputs on an evenly spread subset of n_oracle positions (indices), and the f64 PyTorch twin on all n"""
    model = lively_model_wide(blocks)
    planes = _planes(n, 11)
    idx = np.unique(np.linspace(0, n - 1, n_oracle).round().astype(np.int64))
    want_p, want_v = O.net_forward(model.state_dict(), planes[idx])
    with torch.no_grad():
        m64 = lively_model_wide(blocks).double().cuda()
        p64, v64 = m64(torch.from_numpy(planes).double().cuda())
    return planes, idx, want_p, want_v, p64.reshape(n, 50).cpu().numpy(), v64.reshape(n).cpu().numpy()


def _forward(onb, model, planes, precision):
    n = planes.shape[0]
    with onb.Context(n, mcts_max_sims=2, planes=False) as ctx:
        ctx.net_load(model, precision=precision)
        ctx.write(onb.BUF_LEAF_PLANES, planes)
        ctx.net_forward(onb.BUF_LEAF_PLANES)
        return ctx.read(onb.BUF_POLICY, np.float32, (n, 50)), ctx.read(onb.BUF_VALUE, np.float32, (n,))


def _check(pol, val, want_p, want_v, precision, what):
    dp, dv = np.abs(pol - want_p), np.abs(val - want_v)
    tp_max, tp_mean, tv_max, tv_mean = NET_TOL[precision]
    print("wide network %s %s: max|dp| %.3g mean %.3g  max|dv| %.3g mean %.3g" % (precision, what, dp.max(), dp.mean(), dv.max(), dv.mean()))
    assert dp.max() <= tp_max and dp.mean() <= tp_mean, (what, dp.max(), dp.mean())
    assert dv.max() <= tv_max and dv.mean() <= tv_mean, (what, dv.max(), dv.mean())


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16", "tf32"])
@pytest.mark.parametrize("blocks", [0, 1, 3, 5])
@pytest.mark.parametrize("n", [333, 5003])
def test_wide_network_kernel_matches_oracle(onb, n, blocks, precision):
    """k_net_wide against the CPU restatement (f32 weights, f64 sums) with the tolerances of the 64-wide kernel: ONB_NET_F32 within
    1e-5 on probabilities and tanh outputs, the 11-bit-operand fast modes within 6e-3 / 2.5e-2. n = 333 is ragged for both the 3 and
    the 7 boards of a pass; at n = 5003 every CTA runs several board groups, so the weight ring's barrier parity wraps across groups.
    The oracle checks all 333 positions, and 280 positions spread over the 5003 (it takes ~30 ms per position at 5 blocks); there
    every position is also checked against the PyTorch twin in f64 with the same bounds. Then batch invariance: a permuted subset
    gives identical bits."""
    model = lively_model_wide(blocks)
    planes, idx, want_p, want_v, p64, v64 = _reference(blocks, n, 333 if n == 333 else 280)
    pol, val = _forward(onb, model, planes, precision)
    assert np.isfinite(pol).all() and np.isfinite(val).all()
    assert np.abs(pol.sum(1) - 1).max() < 1e-5
    _check(pol[idx], val[idx], want_p, want_v, precision, "%d blocks, n %d vs oracle" % (blocks, n))
    _check(pol, val, p64, v64, precision, "%d blocks, n %d vs f64 twin" % (blocks, n))
    assert want_p.std(0).max() > 0.01 and want_v.std() > 0.01
    perm = np.random.default_rng(0).permutation(n)[:50]
    pol2, val2 = _forward(onb, model, planes[perm], precision)
    assert np.array_equal(pol2, pol[perm]) and np.array_equal(val2, val[perm])


# ------------------------------------------------------------------ GPU: search, slots, arena, self-play
@pytest.mark.gpu
def test_search_with_wide_network_bit_exact(onb):
    """onb_mcts_run(ONB_EVAL_NET) with a 3-block 128-wide network, fused and split phase, against the oracle search driven by the same
    kernel on a one-position context (results are batch invariant): visits, priors, W, pi and best move bit-exact."""
    from test_gpu_parity import _cfg4_roots
    model = lively_model_wide(3, seed=21)
    n, sims, c = 8, 48, 2.0
    roots = _cfg4_roots(16, 5)[::2]
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
        res2 = ctx.search(c, sims, evaluator=onb.EVAL_NET, fused=False)
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
def test_mixed_width_slots_fight_and_self_play(onb):
    """A 64-wide network in slot 0 and a 128-wide one in slot 1: each slot's forward matches its own oracle after the other slot was
    loaded, onb_fight between them is reproducible, and onb_self_play with the wide network yields valid pi rows and outcomes."""
    from test_net_cpu import lively_model
    n, sims = 48, 16
    narrow, wide = lively_model(3, seed=6), lively_model_wide(3, seed=8)
    planes = _planes(32, 3)
    a_is_red = (np.arange(n) % 2) == 0
    with onb.Context(n, seed=12, mcts_max_sims=sims) as ctx:
        ctx.net_select(0); ctx.net_load(narrow)
        ctx.net_select(1); ctx.net_load(wide)
        for slot, model in ((0, narrow), (1, wide), (0, narrow)):
            ctx.net_select(slot)
            ctx.write(onb.BUF_LEAF_PLANES, planes)
            ctx.net_forward(onb.BUF_LEAF_PLANES)
            want_p, want_v = O.net_forward(model.state_dict(), planes)
            assert np.abs(ctx.read(onb.BUF_POLICY, np.float32, (n, 50))[:32] - want_p).max() <= 6e-3
            assert np.abs(ctx.read(onb.BUF_VALUE, np.float32, (n,))[:32] - want_v).max() <= 2.5e-2
        results = []
        for _ in range(2):
            ctx.reset()
            a, b, d, per_game = ctx.fight_native(ctx.agent_puct(sims, 2.0, onb.EVAL_NET, 0), ctx.agent_puct(sims, 2.0, onb.EVAL_NET, 1),
                                                 a_is_red, max_plies=40)
            results.append((a, b, d, per_game.tobytes(), ctx.get_states().tobytes()))
        assert results[0] == results[1]
        assert sum(results[0][:3]) == n
        ctx.net_select(1)
        out = ctx.self_play_native(2.0, sims, 64, max_plies=12, evaluator=onb.EVAL_NET)
    m = out["planes"].shape[0]
    assert m > 0 and out["games"] >= 64
    assert torch.allclose(out["pi"].sum(dim=(1, 2)), torch.ones(m, device=out["pi"].device), atol=1e-5)
    assert set(out["z"].unique().tolist()) <= {-1.0, 0.0, 1.0}


# ------------------------------------------------------------------ GPU: the loader
@pytest.mark.gpu
def test_wide_loader_checks(onb):
    """f16 range check at width 128; a tensor of the wrong width is named; widths other than 64 and 128 are refused"""
    from onitama_alphazero_b200.net import ConvResNet
    sd = {k: v.clone() for k, v in lively_model_wide(1).state_dict().items()}
    sd["bn1.running_var"][3] = 1e-14
    sd["bn1.weight"][3] = 3e4
    sd["conv_init_1.weight"][3] *= 1e3
    with onb.Context(4, mcts_max_sims=2, planes=False) as ctx:
        for prec in ("f16", "f32"):
            with pytest.raises(onb.OnbError, match="f16 range"):
                ctx.net_load(sd, precision=prec)
        ctx.net_load(sd, precision="tf32")
        mixed = dict(lively_model_wide(1).state_dict())
        narrow = ConvResNet(64, 21, 1).state_dict()
        for k in ("vh_linear1.weight", "vh_linear1.bias"):
            mixed[k] = narrow[k]
        with pytest.raises(onb.OnbError, match="vh_linear1.weight"):
            ctx.net_load(mixed)
        for width in (32, 96, 256):
            with pytest.raises(onb.OnbError, match="hidden_channels"):
                ctx.net_load(ConvResNet(width, 21, 1))
