"""The rnn block with rl_games' concat_input and / or layer_norm switched off, on the CPU side: what the kernel-only PPO path
accepts, the checkpoint's key -> shape map, and playback of such a checkpoint.

rl-games 1.5.2's ``A2CBuilder.Network`` reads both switches with ``.get(..., False)``, so a block written the short way
(``rnn: {name: lstm, units: 256, layers: 1}``) has neither.  Without concat_input the LSTM input is the MLP output alone, so
``rnn.rnn.weight_ih_l0`` is [1024, 64]; without layer_norm the network builds no ``layer_norm`` sub-module, so the file has no
``layer_norm.*`` keys.  The rl_games stand-in network of test_checkpoint_interop_cpu.py, built from the pickled run config
alone, strict-loads every file."""
import os
import pickle
import types

import pytest
import torch

from test_checkpoint_interop_cpu import _Model

O, A = 18, 2
COMBOS = {"reference": (True, True), "no_layer_norm": (True, False), "no_concat_input": (False, True), "neither": (False, False)}


def overrides(concat_input, layer_norm):
    return [f"train.params.network.rnn.concat_input={concat_input}", f"train.params.network.rnn.layer_norm={layer_norm}"]


def block(concat_input, layer_norm):
    return {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": concat_input, "layer_norm": layer_norm}


@pytest.mark.parametrize("combo", list(COMBOS))
def test_kernel_path_accepts_both_switches_and_still_refuses_other_widths(combo):
    from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
    ci, ln = COMBOS[combo]
    agent = types.SimpleNamespace(A=A, O=O, has_rnn=True)
    assert PPOAgent._kernel_path_gaps(agent, [256, 128, 64], block(ci, ln)) == []
    why = PPOAgent._kernel_path_gaps(agent, [256, 128, 64], dict(block(ci, ln), units=128))
    assert len(why) == 1 and "units 128" in why[0] and "256" in why[0]
    why = PPOAgent._kernel_path_gaps(agent, [256, 128, 64], dict(block(ci, ln), layers=2))
    assert len(why) == 1 and "layers" in why[0]
    why = PPOAgent._kernel_path_gaps(agent, [256, 128, 64], dict(block(ci, ln), before_mlp=True))
    assert len(why) == 1 and "before_mlp" in why[0]
    # the short form rl_games reads as both switches off
    assert PPOAgent._kernel_path_gaps(agent, [256, 128, 64], {"name": "lstm", "units": 256, "layers": 1}) == []


@pytest.mark.parametrize("combo", list(COMBOS))
def test_key_and_shape_map_follows_rl_games(combo):
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, RunningMeanStd, rlgames_model_state
    ci, ln = COMBOS[combo]
    sd = rlgames_model_state(ActorCritic(O, A, (256, 128, 64), rnn=block(ci, ln)), RunningMeanStd((O,)), RunningMeanStd((1,)))
    want = {"a2c_network.sigma": (2,), "a2c_network.actor_mlp.0.weight": (256, O), "a2c_network.actor_mlp.0.bias": (256,),
            "a2c_network.actor_mlp.2.weight": (128, 256), "a2c_network.actor_mlp.2.bias": (128,),
            "a2c_network.actor_mlp.4.weight": (64, 128), "a2c_network.actor_mlp.4.bias": (64,),
            "a2c_network.rnn.rnn.weight_ih_l0": (1024, 64 + (O if ci else 0)), "a2c_network.rnn.rnn.weight_hh_l0": (1024, 256),
            "a2c_network.rnn.rnn.bias_ih_l0": (1024,), "a2c_network.rnn.rnn.bias_hh_l0": (1024,),
            "a2c_network.value.weight": (1, 256), "a2c_network.value.bias": (1,),
            "a2c_network.mu.weight": (2, 256), "a2c_network.mu.bias": (2,),
            "running_mean_std.running_mean": (O,), "running_mean_std.running_var": (O,), "running_mean_std.count": (),
            "value_mean_std.running_mean": (1,), "value_mean_std.running_var": (1,), "value_mean_std.count": ()}
    if ln:
        want.update({"a2c_network.layer_norm.weight": (256,), "a2c_network.layer_norm.bias": (256,)})
    assert {k: tuple(v.shape) for k, v in sd.items()} == want


def _write(tmp_path, ci, ln):
    """A checkpoint + run config written by this trainer's code for the block (concat_input ci, layer_norm ln)."""
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, RunningMeanStd, rlgames_model_state
    from vine_robot_isaacgymenvs_b200.train import write_run_config
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + overrides(ci, ln) + ["rl_device=cpu"])
    net = cfg["train"]["params"]["network"]
    assert net["rnn"]["concat_input"] is ci and net["rnn"]["layer_norm"] is ln
    torch.manual_seed(11)
    model = ActorCritic(O, A, net["mlp"]["units"], rnn=net["rnn"])
    with torch.no_grad():
        model.sigma.fill_(-0.3)
        model.mu.weight.mul_(4.0)
    obs_rms, val_rms = RunningMeanStd((O,)), RunningMeanStd((1,))
    obs_rms.update(torch.randn(4000, O) * 3 + 1)
    val_rms.update(torch.randn(4000) * 2 - 0.5)
    exp_dir = tmp_path / "runs" / "Vine5LinkMovingBase"
    pkl = write_run_config(cfg, str(exp_dir), time_str="2022-11-08_11-20-33")
    os.makedirs(exp_dir / "nn", exist_ok=True)
    path = str(exp_dir / "nn" / "Vine5LinkMovingBase.pth")
    torch.save({"model": rlgames_model_state(model, obs_rms, val_rms), "epoch": 3}, path)
    return pkl, path, net["rnn"]


@pytest.mark.parametrize("combo", list(COMBOS))
def test_player_infers_the_block_from_the_file_and_acts_like_rl_games(tmp_path, combo):
    """The stand-in rl_games network built from the pickled config strict-loads the file; PolicyPlayer(rnn="auto") reads the
    block from the file (units, concat_input from weight_ih_l0's width, layer_norm from layer_norm.weight) and its
    deterministic actions equal the stand-in's over 5 calls with the LSTM state carried; the run config's own rnn dict is
    accepted, the other switch setting is refused."""
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    ci, ln = COMBOS[combo]
    pkl, path, rnn = _write(tmp_path, ci, ln)
    with open(pkl, "rb") as f:
        params = pickle.load(f)["params"]
    model = _Model(params, {"actions_num": A, "input_shape": (O,), "normalize_input": True, "normalize_value": True, "value_size": 1})
    model.load_state_dict(torch.load(path, map_location="cpu")["model"])     # strict
    model.eval()
    ours = PolicyPlayer(O, device="cpu").restore(path)
    assert ours.model.concat_input is ci and isinstance(ours.model.layer_norm, torch.nn.LayerNorm) is ln
    net = {k[len("a2c_network."):]: v for k, v in torch.load(path, map_location="cpu")["model"].items() if k.startswith("a2c_network.")}
    assert ours.rnn_block(net) == block(ci, ln)
    explicit = PolicyPlayer(O, device="cpu", rnn=rnn).restore(path)
    torch.manual_seed(0)
    states = None
    with torch.no_grad():
        for step in range(5):
            obs = torch.randn(1, O) * 2
            out = model({"obs": obs, "rnn_states": states})
            states = out["rnn_states"]
            ref = torch.clamp(out["mus"], -1.0, 1.0)
            assert torch.allclose(ref, ours.get_action(obs, is_deterministic=True), atol=1e-5), step
            assert torch.allclose(ref, explicit.get_action(obs, is_deterministic=True), atol=1e-5), step
    for wrong in (block(not ci, ln), block(ci, not ln), dict(block(ci, ln), units=128)):
        with pytest.raises(ValueError, match="rnn block"):
            PolicyPlayer(O, device="cpu", rnn=wrong).restore(path)
    # rl_games' short form: both switches off
    short = {"name": "lstm", "units": 256, "layers": 1}
    if combo == "neither":
        PolicyPlayer(O, device="cpu", rnn=short).restore(path)
    else:
        with pytest.raises(ValueError, match="rnn block"):
            PolicyPlayer(O, device="cpu", rnn=short).restore(path)
