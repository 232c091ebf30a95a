"""The network stand-in: architecture restated from net.rs; the reference's shipped 3-block weights come from
tests/golden/net_golden.npz, written into .ot archives where a test needs one."""
import os

import pytest
import torch


def test_shapes_and_param_count():
    from onitama_alphazero_b200.net import ConvResNet
    m = ConvResNet(64, 21, 3).eval()
    n_elems = sum(v.numel() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked"))
    assert n_elems == 240006  # SURVEY.md: model_5e-3_3_resnet.ot = 60 tensors / 240 006 elements
    p, v = m(torch.zeros(7, 21, 5, 5))
    assert p.shape == (7, 2, 25) and v.shape == (7, 1)
    assert torch.allclose(p.reshape(7, -1).sum(-1), torch.ones(7), atol=1e-6) and (v.abs() <= 1).all()
    assert sum(v.numel() for k, v in ConvResNet(64, 21, 5).state_dict().items() if not k.endswith("num_batches_tracked")) == 388742


def test_loads_reference_ot_archive(tmp_path):
    """The reference's 3-block weights in the archive layout VarStore::save writes load tensor for tensor and evaluate; a 5-block
    archive loads into a 5-block module."""
    from onitama_alphazero_b200.net import ConvResNet, make_evaluator
    weights = golden_tensors()
    m = ConvResNet(64, 21, 3).load_ot(golden_ot(tmp_path))
    sd = m.state_dict()
    assert all(torch.equal(sd[k], w) for k, w in weights.items())
    net = make_evaluator(m)
    x = torch.zeros(2, 21, 5, 5)
    x[:, 0, 4, :] = 1
    p, v = net(x)
    assert p.shape == (2, 2, 25) and v.shape == (2,) and torch.isfinite(p).all() and torch.equal(p[0], p[1])
    m5 = ConvResNet(64, 21, 5).load_ot(lively_model(5).save_ot(str(tmp_path / "five.ot")))
    assert m5.n_blocks == 5


def test_alphaloss_matches_reference_formula():
    """net.rs:234-243"""
    from onitama_alphazero_b200.net import alphaloss, sample_minibatch
    g = torch.Generator().manual_seed(0)
    v = torch.tanh(torch.randn(6, 1, generator=g))
    z = torch.tensor([[1.0], [-1.0], [0.0], [1.0], [1.0], [-1.0]])
    p = torch.softmax(torch.randn(6, 50, generator=g), dim=-1).reshape(6, 2, 25)
    pi = torch.softmax(torch.randn(6, 50, generator=g), dim=-1).reshape(6, 2, 25)
    vl, pl = alphaloss(v, p, pi, z)
    assert torch.isclose(vl, ((z - v) ** 2).sum() / 6)
    assert torch.isclose(pl, -(p.log() * pi).sum() / (6 * 25))   # sum over the card dim, mean over batch x 25 squares
    idx = sample_minibatch(100, 32, generator=g)
    assert idx.shape == (32,) and len(set(idx.tolist())) == 32 and int(idx.max()) < 100


def lively_model(blocks=3, seed=7, res_gain=None):
    """ConvResNet with activations of order one in every layer and non-trivial BatchNorm statistics (so that BN folding, the
    residual path and both heads all matter to the output); deterministic for a given torch version. res_gain scales the second
    convolution of every residual block (default: 1 up to 3 blocks, 0.5 beyond -- deeper towers would otherwise saturate tanh)."""
    from onitama_alphazero_b200.net import ConvResNet
    torch.manual_seed(seed)
    model = ConvResNet(64, 21, blocks)
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
        if blocks > 3:  # the trunk's activations grow with depth: keep tanh and softmax out of saturation
            model.vh_conv.weight.mul_(0.02)
            model.policy_conv.weight.mul_(0.2)
    return model.eval()


@pytest.mark.parametrize("blocks", [0, 1, 3])
def test_oracle_network_matches_the_pytorch_twin(blocks):
    """oracle/onb_oracle.cpp orc_net_forward (the checker of the tensor-core kernel) against net.py on real positions"""
    import numpy as np
    import oracle_lib as O
    model = lively_model(blocks)
    g = O.new_games(24, seed=5)
    for s in range(9):
        O.env_step_random(g, 5, s)
    planes = O.encode(g).reshape(-1, 21, 5, 5)
    with torch.no_grad():
        p_ref, v_ref = model(torch.from_numpy(planes))
    pol, val = O.net_forward(model.state_dict(), planes)
    assert np.abs(pol - p_ref.reshape(-1, 50).numpy()).max() < 2e-5
    assert np.abs(val - v_ref.reshape(-1).numpy()).max() < 2e-5
    assert p_ref.reshape(-1, 50).std(0).max() > 0.01 and v_ref.std() > 0.01   # the outputs do depend on the position


def test_oracle_network_with_reference_weights():
    import numpy as np
    import oracle_lib as O
    from onitama_alphazero_b200.net import ConvResNet
    m = ConvResNet(64, 21, 3)
    m.load_state_dict(golden_tensors(), strict=False)
    m.eval()
    g = O.new_games(8, seed=1)
    planes = O.encode(g).reshape(-1, 21, 5, 5)
    with torch.no_grad():
        p_ref, v_ref = m(torch.from_numpy(planes))
    pol, val = O.net_forward(m.state_dict(), planes)
    assert np.abs(pol - p_ref.reshape(-1, 50).numpy()).max() < 2e-5 and np.abs(val - v_ref.reshape(-1).numpy()).max() < 2e-5


def load_net_golden():
    """tests/golden/net_golden.npz (made by tests/golden/gen_net_golden.py from the reference's shipped 3-block weights)"""
    import numpy as np
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "net_golden.npz"))
    weights = {k[2:]: z[k] for k in z.files if k.startswith("w:")}
    return weights, z["planes"], z["policy"], z["value"]


def golden_tensors():
    """the reference's 3-block weights from the fixture as torch tensors (state_dict names, no num_batches_tracked)"""
    return {k: torch.from_numpy(w) for k, w in load_net_golden()[0].items()}


def golden_ot(tmp_path):
    """the fixture's weights written as the reference's 3-block .ot archive; returns its path"""
    from onitama_alphazero_b200.net import write_ot
    path = str(tmp_path / "model_5e-3_3_resnet.ot")
    write_ot(golden_tensors(), path)
    return path


def test_oracle_network_on_the_reference_trained_weights_fixture():
    """The committed fixture (reference weights + outputs of the PyTorch twin) is available on the GPU box too; the oracle must
    reproduce it, and the fixture must be what the twin computes today."""
    import numpy as np
    import oracle_lib as O
    from onitama_alphazero_b200.net import ConvResNet
    weights, planes, pol, val = load_net_golden()
    assert len(weights) == 60 and planes.shape[1:] == (21, 5, 5)
    p, v = O.net_forward(weights, planes)
    assert np.abs(p - pol).max() < 2e-5 and np.abs(v - val).max() < 2e-5
    m = ConvResNet(64, 21, 3)
    m.load_state_dict({k: torch.from_numpy(w) for k, w in weights.items()}, strict=False)
    with torch.no_grad():
        p2, v2 = m.eval()(torch.from_numpy(planes))
    assert np.abs(p2.reshape(-1, 50).numpy() - pol).max() < 1e-6 and np.abs(v2.reshape(-1).numpy() - val).max() < 1e-6
    assert pol.std(0).max() > 0.01          # the trained policy head does depend on the position


def test_ot_archives_block_count_is_inferred_and_mismatches_are_errors(tmp_path):
    """ADVICE r01: four of the reference's five checkpoints have 5 residual blocks (ConvResNetConfig::default, net.rs:82-90); loading one
    into a 3-block module must not silently drop resnet_3 / resnet_4."""
    from onitama_alphazero_b200.net import ConvResNet
    five = lively_model(5).save_ot(str(tmp_path / "model_5e-3.ot"))
    three = golden_ot(tmp_path)
    assert ConvResNet().n_blocks == 5
    assert ConvResNet.from_ot(five).n_blocks == 5
    assert ConvResNet.from_ot(three).n_blocks == 3
    with pytest.raises(KeyError, match="unexpected"):
        ConvResNet(64, 21, 3).load_ot(five)
    with pytest.raises(KeyError, match="missing"):
        ConvResNet(64, 21, 5).load_ot(three)


def test_ot_writer_round_trip(tmp_path):
    """save_ot writes what VarStore::load reads (alphazero_mcts/mod.rs:89-105): a TorchScript archive whose parameters carry the VarStore
    paths with '|' separators, running statistics as parameters without gradient; it reads back bit for bit."""
    from onitama_alphazero_b200.net import ConvResNet, read_ot
    m = lively_model(2, seed=5)
    path = m.save_ot(str(tmp_path / "model_1_20240101_000000.ot"))
    back = ConvResNet.from_ot(path)
    sd, sd2 = m.state_dict(), back.state_dict()
    for k in sd:
        if not k.endswith("num_batches_tracked"):
            assert torch.equal(sd[k], sd2[k]), k
    arch = torch.jit.load(path)
    names = {n: p.requires_grad for n, p in arch.named_parameters()}
    assert "resnet_1|resnet_small_block2|small_block_bn|running_var" in names and "conv_init_1|weight" in names
    assert not any("." in n or "num_batches_tracked" in n for n in names)
    assert names["bn1|running_mean"] is False and names["bn1|weight"] is True
    # same names and shapes as the reference's 3-block archive (the fixture holds its tensors), all f32
    ref = load_net_golden()[0]
    got = read_ot(ConvResNet(64, 21, 3).save_ot(str(tmp_path / "three.ot")))
    assert sorted(got) == sorted(ref) and all(got[k].shape == ref[k].shape and got[k].dtype == torch.float32 for k in ref)


def test_stats_json_layout(tmp_path):
    """stats.rs:14-80: the serde layout of the training log, written and read back"""
    import datetime
    import json
    from onitama_alphazero_b200.selfplay import fight_statistics
    from onitama_alphazero_b200.stats import Stats
    now = datetime.datetime(2024, 6, 7, 12, 34, 56)
    st = Stats(root=str(tmp_path), now=now)
    assert st.dir.endswith("loss_20240607_123456")
    st.push(0, 2.5, 1.0, 1.5)
    st.push_games_played(1200, 33000)
    fs = fight_statistics([1, 2, 0, 1], [True, False, True, False], 800.0, 800.0)
    st.push_fight(True, self_fight=fs, random_fight=fs)
    path = st.save(now)
    assert os.path.basename(path) == "loss_stats_20240624_123456.json"   # the reference's "%Y%m%y" format string, reproduced
    d = json.load(open(path))
    assert list(d) == ["iteration", "loss", "policy_loss", "value_loss", "was_best_change", "fight_statistics", "games_played", "dir"]
    assert d["loss"] == [2.5] and d["value_loss"] == [1.0] and d["policy_loss"] == [1.5] and d["was_best_change"] == [True]
    assert d["games_played"] == [{"games_amnt": 1200, "positions_retrieved": 33000}]
    pit = d["fight_statistics"][0]
    assert list(pit) == ["self_fight", "random_fight", "alphabeta_fight", "mcts_fight"]
    sf = pit["self_fight"]
    assert list(sf) == ["general", "winrate", "color", "color_winrate", "rating_a", "rating_b", "rating_change_history"]
    assert sf["general"] == {"wins": 2, "loses": 1, "draws": 1} and len(sf["rating_change_history"]) == 4
    assert list(sf["rating_change_history"][0]) == ["before_a", "after_a", "before_b", "after_b"]
    assert sf["rating_change_history"][0]["before_a"] == 800.0 and sf["rating_change_history"][0]["after_a"] == 816.0
    assert pit["mcts_fight"]["general"] == {"wins": 0, "loses": 0, "draws": 0}
    again = Stats.load(path)
    assert again.to_dict() == d
