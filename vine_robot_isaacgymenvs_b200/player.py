"""Deployment-side inference (SURVEY §8 "next" f4): what the reference's ``isaacgymenvs/vine_robot_test_model.py``
does with rl_games' ``PpoPlayerContinuous`` -- load a checkpoint, feed one observation, get one action, keep the
LSTM state between calls -- without rl_games.

``PolicyPlayer.get_action(obs, is_deterministic)``   == rl_games BasePlayer.get_action (vine_robot_test_model.py:112-131)
``VineRobotControlModel.get_action(q, qd, tip_pos, tip_vel, target_pos)`` == vine_robot_test_model.py:143-177

Checkpoints: the rl_games layout ``PPOAgent.state_dict`` writes (``model`` -> ``a2c_network.*``, ``running_mean_std.*``).
A file without ``running_mean_std.*`` comes from a run with ``normalize_input: False``: the policy then acts on the raw
observations (no mean, std or +-5 clamp), as it did in training.  The rnn block is read from the file too (``rnn="auto"``):
rl_games' ``concat_input`` and ``layer_norm`` default to False, so a block written ``{name: lstm, units: 256, layers: 1}``
has neither the observation columns in ``weight_ih_l0`` nor ``layer_norm.*``.
Runs wherever torch runs (the robot-side host may have no GPU); on a B200 the batched MLP policy can instead go through
``vine_policy_act``.
"""
import torch

from .ppo.ppo import ActorCritic, RunningMeanStd

REFERENCE_RNN = {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": True, "layer_norm": True}


class PolicyPlayer:
    def __init__(self, num_obs, num_actions=2, units=(256, 128, 64), rnn="auto", device="cpu", clip_actions=True,
                 normalize_input="auto"):
        """``normalize_input``: "auto" = whether the checkpoint has the input normaliser (``running_mean_std.*``), or the
        training config's bool (then a file that disagrees is refused).  ``rnn``: "auto" = the block the checkpoint holds
        (``rnn_block``), the training config's ``network.rnn`` dict (then a file that disagrees is refused), or a bool: the
        reference's block / none."""
        self.device, self.clip_actions, self._rnn_arg = torch.device(device), clip_actions, rnn
        self.num_obs, self.num_actions, self.units = num_obs, num_actions, tuple(units)
        self._norm_arg = normalize_input
        self.model = self.obs_rms = self.states = None
        self.normalize_input = True

    def rnn_block(self, net):
        """The rnn block of a checkpoint's network (``net``: its ``a2c_network.*`` entries without the prefix) as rl_games'
        ``network.rnn``, or None when it has none: ``units`` from ``weight_hh_l0``'s width, ``concat_input`` from
        ``weight_ih_l0``'s (mlp ``units[-1] + num_obs`` or ``units[-1]``), ``layer_norm`` from whether ``layer_norm.weight``
        is present."""
        if "rnn.rnn.weight_hh_l0" not in net:
            return None
        d, width = self.units[-1], int(net["rnn.rnn.weight_ih_l0"].shape[1])
        if width not in (d, d + self.num_obs):
            raise ValueError(f"the checkpoint's rnn.rnn.weight_ih_l0 has {width} columns: neither the MLP output ({d}) nor it "
                             f"plus {self.num_obs} observations")
        return dict(REFERENCE_RNN, units=int(net["rnn.rnn.weight_hh_l0"].shape[1]), concat_input=width == d + self.num_obs,
                    layer_norm="layer_norm.weight" in net)

    def _rnn_for(self, net):
        found = self.rnn_block(net)
        if isinstance(self._rnn_arg, dict):   # the training config's block: it must be the file's (rl_games' defaults: False)
            arg = self._rnn_arg
            same = found is not None and str(arg.get("name", "lstm")).lower() == "lstm" and all(
                bool(arg.get(k, False)) == found[k] for k in ("concat_input", "layer_norm")) and int(arg.get("units", 0)) == found["units"]
            if not same:
                raise ValueError(f"rnn={arg} but the checkpoint's rnn block is {found}")
            return arg
        if self._rnn_arg == "auto":
            return found
        return REFERENCE_RNN if self._rnn_arg else None

    def _build(self, rnn):
        self.model = ActorCritic(self.num_obs, self.num_actions, self.units, rnn=rnn).to(self.device).eval()
        self.obs_rms = RunningMeanStd((self.num_obs,)).to(self.device)
        self.reset()

    def restore(self, fn_or_state):
        ck = torch.load(fn_or_state, map_location=self.device) if isinstance(fn_or_state, (str, bytes)) or hasattr(fn_or_state, "__fspath__") else fn_or_state
        model = ck["model"]
        net = {k[len("a2c_network."):]: v for k, v in model.items() if k.startswith("a2c_network.")}
        self._build(self._rnn_for(net))
        self.model.load_state_dict(net)
        rms = {k[len("running_mean_std."):]: v for k, v in model.items() if k.startswith("running_mean_std.")}
        if not rms and "running_mean_std" in ck:          # vine_robot_test_model.py:137-139
            rms = ck["running_mean_std"]
        self.normalize_input = bool(rms) if self._norm_arg == "auto" else bool(self._norm_arg)
        if bool(rms) != self.normalize_input:
            raise ValueError(f"normalize_input={self.normalize_input} but the checkpoint {'has' if rms else 'lacks'} running_mean_std.*")
        if rms:
            self.obs_rms.load_state_dict({k: v.to(torch.float64) for k, v in rms.items()})
        return self

    def reset(self, batch=1):
        """Zero LSTM state (rl_games player.reset / init_rnn)."""
        if self.model is not None and self.model.has_rnn:
            H = self.model.rnn_units
            self.states = (torch.zeros(batch, H, device=self.device), torch.zeros(batch, H, device=self.device))
        else:
            self.states = None

    @torch.no_grad()
    def get_action(self, obs, is_deterministic=False):
        obs = torch.as_tensor(obs, dtype=torch.float32, device=self.device)
        squeeze = obs.dim() == 1
        obs = obs.reshape(-1, self.num_obs)
        if self.states is not None and self.states[0].shape[0] != obs.shape[0]:
            self.reset(obs.shape[0])
        x = self.obs_rms(obs) if self.normalize_input else obs
        mu, logstd, _, self.states = self.model(x, self.states)
        action = mu if is_deterministic else mu + torch.exp(logstd) * torch.randn_like(mu)
        if self.clip_actions:
            action = torch.clamp(action, -1.0, 1.0)
        return action[0] if squeeze else action


class VineRobotControlModel(torch.nn.Module):
    """vine_robot_test_model.py:143-177: actions rescaled from [-1, 1] to the hardware ranges."""

    def __init__(self, checkpoint_path, x_range, u_range, num_obs, device="cpu", deterministic=False, **player_kw):
        """``deterministic=False`` is what the reference script does: its ``forward`` calls ``get_action(obs)`` whose
        ``is_determenistic`` defaults to False, i.e. it SAMPLES (vine_robot_test_model.py:112-131,170-171).  Pass True to act
        with the mean."""
        super().__init__()
        self.deterministic = bool(deterministic)
        self.rail_force_min, self.rail_force_max = x_range
        self.u_min, self.u_max = u_range
        self.player = PolicyPlayer(num_obs, device=device, **player_kw).restore(checkpoint_path)

    @staticmethod
    def rescale(x, low, high):
        return (x + 1) * (high - low) / 2 + low

    def forward(self, obs):
        return self.player.get_action(obs, is_deterministic=self.deterministic)

    def get_action(self, *parts):
        """``parts``: the observation pieces in the order the policy was trained on (the reference's script passes
        q, qd, tip_pos, tip_vel, target_pos); returns (rail command, pressure command) in hardware units."""
        obs = torch.cat([torch.as_tensor(p, dtype=torch.float32).reshape(-1) for p in parts])[None, ...]
        action = self.forward(obs)[0].clone()
        if action.numel() == 1:
            return self.rescale(action, self.u_min, self.u_max)
        action[0] = self.rescale(action[0], self.rail_force_min, self.rail_force_max)
        action[1] = self.rescale(action[1], self.u_min, self.u_max)
        return action
