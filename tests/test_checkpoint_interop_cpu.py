"""Checkpoint interop with the reference's deployment script (SURVEY §8 f2): the UNMODIFIED ``BasePlayer`` /
``PpoPlayerContinuous`` / ``VineRobotControlModel`` classes of ``isaacgymenvs/vine_robot_test_model.py`` (executed from
/root/reference, class and function definitions only -- the script's module-level cells hard-code the author's paths) restore a
checkpoint + ``*_rlg_config_dict.pkl`` written by THIS trainer's code and act with it.

rl_games itself is not installable here, so the three names the script imports from it are stubs written in this file from
rl-games 1.5.2's published structure (``ModelBuilder.load -> network.build(config) -> ModelA2CContinuousLogStd.Network`` with
sub-modules ``a2c_network`` / ``running_mean_std`` / ``value_mean_std``; ``torch_ext.load_checkpoint``; ``torch_runner._restore``).
The stub network is built ONLY from the pickled config and restores with a strict ``load_state_dict``: a missing, surplus or
mis-shaped key in our file fails the test.  Its forward is plain torch (no code of this repo), and its deterministic action
must equal ``player.PolicyPlayer``'s on the same file.  The script's part runs only where the reference checkout exists; the
stub network restoring our checkpoint from the pickled config alone runs everywhere.
"""
import ast
import os
import pickle
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

REF = "/root/reference/isaacgymenvs/vine_robot_test_model.py"


# ---------------------------------------------------------------- stand-ins for the three rl_games names the script imports
class _RunningMeanStd(nn.Module):      # rl_games.algos_torch.running_mean_std.RunningMeanStd (eval-mode forward)
    def __init__(self, shape):
        super().__init__()
        self.register_buffer("running_mean", torch.zeros(shape, dtype=torch.float64))
        self.register_buffer("running_var", torch.ones(shape, dtype=torch.float64))
        self.register_buffer("count", torch.ones((), dtype=torch.float64))

    def forward(self, x):
        y = (x - self.running_mean.float()) / torch.sqrt(self.running_var.float() + 1e-5)
        return torch.clamp(y, -5.0, 5.0)


class _LSTMWithDones(nn.Module):       # rl_games.common.layers.recurrent.LSTMWithDones: the nn.LSTM sits under .rnn
    def __init__(self, inp, units):
        super().__init__()
        self.rnn = nn.LSTM(inp, units, 1)


class _A2CNetwork(nn.Module):          # rl_games.algos_torch.network_builder.A2CBuilder.Network for this config
    def __init__(self, params, actions_num, input_shape):
        super().__init__()
        net = params["network"]
        assert net["name"] == "actor_critic" and not net.get("separate", False) and net["mlp"]["activation"] == "elu"
        assert net["space"]["continuous"]["fixed_sigma"]
        layers, d = [], input_shape[0]
        for u in net["mlp"]["units"]:
            layers += [nn.Linear(d, u), nn.ELU()]
            d = u
        self.actor_mlp = nn.Sequential(*layers)
        self.rnn_cfg = net.get("rnn")
        if self.rnn_cfg:
            assert self.rnn_cfg["name"] == "lstm" and not self.rnn_cfg.get("before_mlp", False)
            inp = d + (input_shape[0] if self.rnn_cfg.get("concat_input") else 0)
            self.rnn = _LSTMWithDones(inp, self.rnn_cfg["units"])
            d = self.rnn_cfg["units"]
            if self.rnn_cfg.get("layer_norm"):
                self.layer_norm = nn.LayerNorm(d)
        self.value = nn.Linear(d, 1)
        self.mu = nn.Linear(d, actions_num)
        self.sigma = nn.Parameter(torch.zeros(actions_num))


class _Model(nn.Module):               # ModelA2CContinuousLogStd.Network
    def __init__(self, params, config):
        super().__init__()
        self.a2c_network = _A2CNetwork(params, config["actions_num"], config["input_shape"])
        if config["normalize_input"]:
            self.running_mean_std = _RunningMeanStd(config["input_shape"])
        if config["normalize_value"]:
            self.value_mean_std = _RunningMeanStd((config["value_size"],))

    def forward(self, d):
        n = self.a2c_network
        x = self.running_mean_std(d["obs"])
        h = n.actor_mlp(x)
        states = d.get("rnn_states")
        if n.rnn_cfg:
            inp = torch.cat([h, x], -1) if n.rnn_cfg.get("concat_input") else h
            out, states = n.rnn.rnn(inp[None], states)          # states None: zeros, like a freshly reset player
            h = out[0]
            if n.rnn_cfg.get("layer_norm"):
                h = n.layer_norm(h)
        mu, sigma = n.mu(h), torch.exp(n.sigma)
        return {"mus": mu, "sigmas": sigma, "actions": mu + sigma * torch.randn_like(mu), "values": n.value(h), "rnn_states": states}


def _reference_classes(n_obs, n_actions):
    """Execute the class / function definitions of the reference script (nothing else) with the stubs in scope."""
    class _Builder:
        def load(self, params):
            return types.SimpleNamespace(build=lambda config: _Model(params, config))

    class _Box:
        def __init__(self, low, high):
            self.low, self.high, self.shape = np.asarray(low, np.float32), np.asarray(high, np.float32), np.asarray(low).shape

    if not hasattr(np, "Inf"):
        np.Inf = np.inf                                          # the script predates numpy 2
    ns = {"model_builder": types.SimpleNamespace(ModelBuilder=_Builder),
          "torch_ext": types.SimpleNamespace(load_checkpoint=lambda fn: torch.load(fn, map_location="cpu")),
          "_restore": lambda player, args: player.restore(args["checkpoint"]),
          "spaces": types.SimpleNamespace(Box=_Box), "np": np, "torch": torch, "nn": nn, "pickle": pickle, "os": os,
          "N_OBS": n_obs, "N_ACTIONS": n_actions}                # the script's "PARAMETERS" cell, set for our task
    tree = ast.parse(open(REF).read())
    defs = [node for node in tree.body if isinstance(node, (ast.ClassDef, ast.FunctionDef))]
    assert {d.name for d in defs} >= {"BasePlayer", "PpoPlayerContinuous", "VineRobotControlModel", "rescale_actions"}
    exec(compile(ast.Module(body=defs, type_ignores=[]), REF, "exec"), ns)
    return ns


def _write_checkpoint(tmp_path, rnn):
    """A checkpoint + run config written by this trainer's code -> (path of the pickled config, path of the .pth)."""
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, RunningMeanStd, rlgames_model_state
    from vine_robot_isaacgymenvs_b200.train import write_run_config
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + ([] if rnn else ["train.params.network.rnn=null"]) + ["rl_device=cpu"])
    cfg["train"]["params"]["config"]["device_name"] = "cpu"      # the script defaults to 'cuda'
    O, A = 18, 2
    torch.manual_seed(3)
    net = cfg["train"]["params"]["network"]
    model = ActorCritic(O, A, net["mlp"]["units"], rnn=net.get("rnn"))
    with torch.no_grad():
        model.sigma.fill_(-0.3)
    obs_rms, val_rms = RunningMeanStd((O,)), RunningMeanStd((1,))
    obs_rms.update(torch.randn(4000, O) * 3 + 1)
    val_rms.update(torch.randn(4000) * 2 - 0.5)
    ckpt = {"model": rlgames_model_state(model, obs_rms, val_rms), "epoch": 7, "frame": 7 * 65536, "last_lr": 3e-4}
    exp_dir = tmp_path / "runs" / "Vine5LinkMovingBase"
    pkl = write_run_config(cfg, str(exp_dir), time_str="2022-11-08_11-20-33")
    assert os.path.basename(pkl) == "2022-11-08_11-20-33_rlg_config_dict.pkl" and os.path.exists(exp_dir / "config.yaml")
    os.makedirs(exp_dir / "nn", exist_ok=True)
    path = str(exp_dir / "nn" / "last_Vine5LinkMovingBase_ep_7_rew_1.pth")
    torch.save(ckpt, path)
    return pkl, path


@pytest.mark.parametrize("rnn", [True, False], ids=["reference_network", "mlp_only"])
def test_rl_games_network_built_from_the_pickled_config_restores_and_runs_our_checkpoint(tmp_path, rnn):
    """What rl_games' player does with the two files, minus the script: network from the pickled config, strict load, act."""
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    pkl, path = _write_checkpoint(tmp_path, rnn)
    O, A = 18, 2
    with open(pkl, "rb") as f:
        params = pickle.load(f)["params"]
    model = _Model(params, {"actions_num": A, "input_shape": (O,), "normalize_input": params["config"]["normalize_input"],
                            "normalize_value": params["config"]["normalize_value"], "value_size": 1})
    model.load_state_dict(torch.load(path, map_location="cpu")["model"])     # strict
    model.eval()
    ours = PolicyPlayer(O, device="cpu").restore(path)
    torch.manual_seed(0)
    states = None
    with torch.no_grad():
        for step in range(5):                                    # the LSTM state is carried across calls in both
            obs = torch.randn(1, O) * 2
            out = model({"obs": obs, "rnn_states": states})
            states = out["rnn_states"]
            assert torch.allclose(torch.clamp(out["mus"], -1.0, 1.0), ours.get_action(obs, is_deterministic=True), atol=1e-5), step


@pytest.mark.skipif(not os.path.exists(REF), reason="needs the reference checkout")
@pytest.mark.parametrize("rnn", [True, False], ids=["reference_network", "mlp_only"])
def test_reference_deployment_script_restores_and_runs_our_checkpoint(tmp_path, rnn):
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    pkl, path = _write_checkpoint(tmp_path, rnn)
    O, A = 18, 2
    ns = _reference_classes(O, A)
    control = ns["VineRobotControlModel"](pkl, path, x_range=(-10.0, 10.0), u_range=(-0.1, 3.0))   # strict load_state_dict inside
    player = control.rl_games_player
    assert player.normalize_input and player.normalize_value
    ours = PolicyPlayer(O, device="cpu").restore(path)
    torch.manual_seed(0)
    for step in range(5):                                        # the LSTM state is carried across calls in both
        obs = torch.randn(1, O) * 2
        ref_a = player.get_action(obs, is_determenistic=True)
        assert torch.allclose(ref_a, ours.get_action(obs, is_deterministic=True), atol=1e-5), step
    # and the script's own entry point: 5 observation pieces -> rescaled (rail, pressure) command
    parts = [torch.randn(6), torch.randn(6), torch.randn(3), torch.randn(1), torch.randn(2)]
    out = control.get_action(*parts)
    assert out.shape == (2,) and -10.0 <= float(out[0]) <= 10.0 and -0.1 <= float(out[1]) <= 3.0


def test_checkpoint_key_and_shape_map_is_rl_games():
    """The exact key -> shape map of an rl-games 1.5.2 `continuous_a2c_logstd` model with this network config."""
    from vine_robot_isaacgymenvs_b200.player import REFERENCE_RNN
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, RunningMeanStd, rlgames_model_state
    O = 18
    sd = rlgames_model_state(ActorCritic(O, 2, (256, 128, 64), rnn=REFERENCE_RNN), RunningMeanStd((O,)), RunningMeanStd((1,)))
    want = {"a2c_network.sigma": (2,), "a2c_network.actor_mlp.0.weight": (256, O), "a2c_network.actor_mlp.0.bias": (256,),
            "a2c_network.actor_mlp.2.weight": (128, 256), "a2c_network.actor_mlp.2.bias": (128,),
            "a2c_network.actor_mlp.4.weight": (64, 128), "a2c_network.actor_mlp.4.bias": (64,),
            "a2c_network.rnn.rnn.weight_ih_l0": (1024, 64 + O), "a2c_network.rnn.rnn.weight_hh_l0": (1024, 256),
            "a2c_network.rnn.rnn.bias_ih_l0": (1024,), "a2c_network.rnn.rnn.bias_hh_l0": (1024,),
            "a2c_network.layer_norm.weight": (256,), "a2c_network.layer_norm.bias": (256,),
            "a2c_network.value.weight": (1, 256), "a2c_network.value.bias": (1,),
            "a2c_network.mu.weight": (2, 256), "a2c_network.mu.bias": (2,),
            "running_mean_std.running_mean": (O,), "running_mean_std.running_var": (O,), "running_mean_std.count": (),
            "value_mean_std.running_mean": (1,), "value_mean_std.running_var": (1,), "value_mean_std.count": ()}
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    assert sd["running_mean_std.running_mean"].dtype == torch.float64
