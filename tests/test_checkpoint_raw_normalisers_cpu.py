"""Checkpoints of a run with rl_games' normalisers switched off (normalize_input / normalize_value False).

rl-games 1.5.2's ``ModelA2CContinuousLogStd.Network`` builds ``running_mean_std`` only with normalize_input and
``value_mean_std`` only with normalize_value, so such a run's file has no keys for them, and a strict ``load_state_dict`` of
the network rl_games builds from the pickled run config fails on any surplus key.  The stub network below is built from that
pickled config alone (the same published structure as in test_checkpoint_interop_cpu.py, its own copy); its forward is plain
torch on the raw observations."""
import os
import pickle

import pytest
import torch
import torch.nn as nn

O, A = 18, 2
OFF = ["train.params.config.normalize_input=False", "train.params.config.normalize_value=False"]


class _Network(nn.Module):   # ModelA2CContinuousLogStd.Network with A2CBuilder.Network, for both normalisers off
    def __init__(self, params, config):
        super().__init__()
        net = params["network"]
        assert not config["normalize_input"] and not config["normalize_value"]   # so: no running_mean_std / value_mean_std
        a = nn.Module()
        layers, d = [], config["input_shape"][0]
        for u in net["mlp"]["units"]:
            layers += [nn.Linear(d, u), nn.ELU()]
            d = u
        a.actor_mlp = nn.Sequential(*layers)
        a.rnn_cfg = net.get("rnn")
        if a.rnn_cfg:
            a.rnn = nn.Module()
            a.rnn.rnn = nn.LSTM(d + (config["input_shape"][0] if a.rnn_cfg["concat_input"] else 0), a.rnn_cfg["units"], 1)
            d = a.rnn_cfg["units"]
            a.layer_norm = nn.LayerNorm(d)
        a.value, a.mu, a.sigma = nn.Linear(d, 1), nn.Linear(d, config["actions_num"]), nn.Parameter(torch.zeros(config["actions_num"]))
        self.a2c_network = a

    def forward(self, obs, states=None):
        n = self.a2c_network
        h = n.actor_mlp(obs)                                   # raw observations: no mean, std or clamp
        if n.rnn_cfg:
            out, states = n.rnn.rnn(torch.cat([h, obs], -1)[None], states)
            h = n.layer_norm(out[0])
        return n.mu(h), n.value(h), states


def _write(tmp_path, rnn):
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, rlgames_model_state
    from vine_robot_isaacgymenvs_b200.train import write_run_config
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + OFF + ([] if rnn else ["train.params.network.rnn=null"]) + ["rl_device=cpu"])
    net = cfg["train"]["params"]["network"]
    torch.manual_seed(5)
    model = ActorCritic(O, A, net["mlp"]["units"], rnn=net.get("rnn"))
    exp_dir = tmp_path / "runs" / "Vine5LinkMovingBase"
    pkl = write_run_config(cfg, str(exp_dir), time_str="2022-11-08_11-20-33")
    os.makedirs(exp_dir / "nn", exist_ok=True)
    path = str(exp_dir / "nn" / "Vine5LinkMovingBase.pth")
    torch.save({"model": rlgames_model_state(model, None, None), "epoch": 3}, path)
    return pkl, path


def test_key_and_shape_map_without_normalisers():
    """The exact key -> shape map of the reference network's file with both normalisers off: the network only."""
    from vine_robot_isaacgymenvs_b200.player import REFERENCE_RNN
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, RunningMeanStd, rlgames_model_state
    sd = rlgames_model_state(ActorCritic(O, 2, (256, 128, 64), rnn=REFERENCE_RNN), None, None)
    want = {"a2c_network.sigma": (2,), "a2c_network.actor_mlp.0.weight": (256, O), "a2c_network.actor_mlp.0.bias": (256,),
            "a2c_network.actor_mlp.2.weight": (128, 256), "a2c_network.actor_mlp.2.bias": (128,),
            "a2c_network.actor_mlp.4.weight": (64, 128), "a2c_network.actor_mlp.4.bias": (64,),
            "a2c_network.rnn.rnn.weight_ih_l0": (1024, 64 + O), "a2c_network.rnn.rnn.weight_hh_l0": (1024, 256),
            "a2c_network.rnn.rnn.bias_ih_l0": (1024,), "a2c_network.rnn.rnn.bias_hh_l0": (1024,),
            "a2c_network.layer_norm.weight": (256,), "a2c_network.layer_norm.bias": (256,),
            "a2c_network.mu.weight": (2, 256), "a2c_network.mu.bias": (2,), "a2c_network.value.weight": (1, 256),
            "a2c_network.value.bias": (1,)}
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    # one normaliser on, the other off: only its own three keys appear
    sd = rlgames_model_state(ActorCritic(O, 2, (256, 128, 64), rnn=REFERENCE_RNN), None, RunningMeanStd((1,)))
    assert {k: tuple(v.shape) for k, v in sd.items() if not k.startswith("a2c_network.")} == {
        "value_mean_std.running_mean": (1,), "value_mean_std.running_var": (1,), "value_mean_std.count": ()}


@pytest.mark.parametrize("rnn", [True, False], ids=["reference_network", "mlp_only"])
def test_network_from_the_pickled_config_strict_loads_and_player_acts_on_raw_observations(tmp_path, rnn):
    """The stub network built from the pickled config (normalize_input / normalize_value False) strict-loads the file, and
    PolicyPlayer restores it without an input normaliser: its deterministic action on observations up to |obs| ~ 20 equals the
    plain torch forward on the same raw observations, the LSTM state carried across calls in both."""
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    pkl, path = _write(tmp_path, rnn)
    with open(pkl, "rb") as f:
        params = pickle.load(f)["params"]
    c = params["config"]
    assert c["normalize_input"] is False and c["normalize_value"] is False
    model = _Network(params, {"actions_num": A, "input_shape": (O,), "normalize_input": c["normalize_input"],
                              "normalize_value": c["normalize_value"]})
    model.load_state_dict(torch.load(path, map_location="cpu")["model"])     # strict
    ours = PolicyPlayer(O, device="cpu").restore(path)
    assert not ours.normalize_input
    torch.manual_seed(0)
    states, big = None, 0
    with torch.no_grad():
        for step in range(5):
            obs = torch.randn(1, O) * 8
            big += int((obs.abs() > 5).sum())
            mu, _, states = model(obs, states)
            assert torch.allclose(torch.clamp(mu, -1.0, 1.0), ours.get_action(obs, is_deterministic=True), atol=1e-5), step
    assert big > 0


def test_player_refuses_a_normaliser_the_file_does_not_have(tmp_path):
    """An explicit normalize_input=True on a file without running_mean_std.* is an error, not an identity normaliser
    (which would still divide by sqrt(1 + 1e-5) and clamp at +-5)."""
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    _, path = _write(tmp_path, False)
    with pytest.raises(ValueError, match="running_mean_std"):
        PolicyPlayer(O, device="cpu", normalize_input=True).restore(path)
    assert not PolicyPlayer(O, device="cpu", normalize_input=False).restore(path).normalize_input
