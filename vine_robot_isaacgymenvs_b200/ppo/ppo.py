"""PPO for the vine task without rl_games (SURVEY §8 row a14 and "next" f1).

Restates what rl-games 1.5.2's ``A2CAgent`` does for ``cfg/train/Vine5LinkMovingBasePPO.yaml``
(``a2c_continuous`` / ``continuous_a2c_logstd`` / ``actor_critic``): horizon-16 rollouts, GAE
(``vine_gae`` CUDA kernel), running mean/std of observations and values, advantage normalisation,
clipped actor loss, clipped (``clip_value``) critic loss x critic_coef, bound loss, Adam with the adaptive-KL or linear
learning-rate schedule (``lr_schedule``) run per minibatch or per mini-epoch (``schedule_type``), value bootstrap on
``time_outs``, reward shaper (scale, shift, clamp).
In-repo analogue of the same math: isaacgymenvs/learning/common_agent.py:257-314 (rollout),
:319-435 (update), :482-517 (losses).  rl_games itself is not vendored in the reference
(setup.py:22) and not installed here: PARITY UNPINNED, checked by learning curves only.

The whole iteration is free of host synchronisation (episode statistics, KL and the learning rate live on the device), so
the rollout (16 x {policy, fused env step} + GAE) and the update (mini_epochs x minibatches) are each captured into ONE
CUDA graph (``use_graphs=True``).  Three execution paths, chosen per network:

  * reference network (MLP -> LSTM 256 -> LayerNorm -> heads, ``train.params.network.rnn``): hand-written kernels only,
    ``_rollout_native_lstm`` / ``_update_native_lstm`` (launch order: ppo/lstm_native.py; kernels: csrc/vine_lstm_net.cu);
  * MLP actor-critic (``rnn=null``): hand-written kernels only, ``_rollout_fused`` / ``_update_fused`` (csrc/vine_rollout.cu,
    csrc/vine_ppo.cu);
  * ``use_fused_update=False`` (or a network shape the kernels do not cover): torch autograd + cuBLAS + torch Adam, the
    library baseline the kernel paths are tested against (``_rollout`` / ``_update``).

Multi-GPU: one process per GPU, envs sharded; per minibatch ONE all-reduce carrying the flat gradient vector(s) plus the
loss statistics (incl. the KL that drives the adaptive learning rate); per iteration one all-reduce of the f64
running-statistics moments.  On the kernel paths the NCCL calls are captured inside the CUDA graphs.
"""
import ctypes as C
import math
import time

import torch
import torch.nn as nn

from .. import abi, distributed as vd


class RunningMeanStd(nn.Module):
    """rl_games RunningMeanStd (per-feature, eps 1e-5, clamp +-5 on normalised output)."""

    def __init__(self, shape, eps=1e-5):
        super().__init__()
        self.eps = eps
        self.register_buffer("running_mean", torch.zeros(shape, dtype=torch.float64))
        self.register_buffer("running_var", torch.ones(shape, dtype=torch.float64))
        self.register_buffer("count", torch.ones((), dtype=torch.float64))

    @torch.no_grad()
    def update(self, x):
        x = x.reshape(-1, *self.running_mean.shape) if self.running_mean.dim() else x.reshape(-1)
        n = x.shape[0]
        mean = x.mean(0)
        m2 = ((x - mean) ** 2).sum(0)
        n, mean, m2 = vd.merge_moments(n, mean, m2)
        n = float(n)
        var = m2.double() / max(n - 1.0, 1.0)
        mean = mean.double()
        delta = mean - self.running_mean
        tot = self.count + n
        new_mean = self.running_mean + delta * n / tot
        m_a = self.running_var * self.count
        m_b = var * n
        self.running_var.copy_((m_a + m_b + delta ** 2 * self.count * n / tot) / tot)
        self.running_mean.copy_(new_mean)
        self.count.copy_(tot)

    def forward(self, x, unnorm=False):
        mean = self.running_mean.float()
        std = torch.sqrt(self.running_var.float() + self.eps)
        if unnorm:
            return torch.clamp(x, -5.0, 5.0) * std + mean
        return torch.clamp((x - mean) / std, -5.0, 5.0)


class _RnnHolder(nn.Module):
    """Parameter holder named like rl_games' LSTMWithDones wrapper (checkpoint key ``rnn.rnn.weight_ih_l0``)."""

    def __init__(self, input_size, hidden):
        super().__init__()
        self.rnn = nn.LSTM(input_size, hidden, 1)


class ActorCritic(nn.Module):
    """``actor_critic`` network of Vine5LinkMovingBasePPO.yaml:10-40 (rl_games A2CBuilder, separate: False):
    shared MLP [256,128,64] ELU -> (rnn: lstm 256, before_mlp False, concat_input True, layer_norm True)
    -> mu head, value head; state-independent learnable log-std initialised to 0 (fixed_sigma: True).
    Sub-module names follow rl_games' ``a2c_network`` so checkpoints map key for key.

    With the LSTM the training forward is truncated BPTT over ``seq_len`` steps; the hidden state is
    multiplied by (1 - done_t) before consuming observation t, which is what rl_games' rollout does
    when it zeroes the states of finished envs (a2c_common.play_steps_rnn)."""

    def __init__(self, num_obs, num_actions, units=(256, 128, 64), rnn=None):
        super().__init__()
        layers, d = [], num_obs
        for u in units:
            layers += [nn.Linear(d, u), nn.ELU()]
            d = u
        self.actor_mlp = nn.Sequential(*layers)
        self.has_rnn = bool(rnn) and str(rnn.get("name", "lstm")).lower() not in ("none", "")
        self.fused_cell = True    # CUDA only: fused pointwise LSTM kernels (False = the pure-torch restatement)
        if self.has_rnn:
            if str(rnn["name"]).lower() != "lstm" or int(rnn.get("layers", 1)) != 1 or rnn.get("before_mlp", False):
                raise ValueError("only the reference's rnn block is supported: lstm, 1 layer, before_mlp False")
            self.concat_input = bool(rnn.get("concat_input", False))
            self.rnn_units = int(rnn["units"])
            self.rnn = _RnnHolder(d + (num_obs if self.concat_input else 0), self.rnn_units)
            d = self.rnn_units
            self.layer_norm = nn.LayerNorm(d) if rnn.get("layer_norm", False) else nn.Identity()
        self.mu = nn.Linear(d, num_actions)
        self.value = nn.Linear(d, 1)
        self.sigma = nn.Parameter(torch.zeros(num_actions))

    def forward(self, obs, states=None, not_done=None):
        """obs [L, S, O] (or [S, O] == L=1); states (h, c) each [S, H]; not_done [L, S] or None.
        Returns mu [L*S, A], logstd, value [L*S, 1], new states."""
        if not self.has_rnn:
            x = obs.reshape(-1, obs.shape[-1])
            h = self.actor_mlp(x)
            return self.mu(h), self.sigma.expand(x.shape[0], -1), self.value(h), None
        if obs.dim() == 2:
            obs = obs.unsqueeze(0)
        L, S, O = obs.shape
        x = obs.reshape(L * S, O)
        m = self.actor_mlp(x)
        inp = torch.cat([m, x.to(m.dtype)], -1) if self.concat_input else m
        r = self.rnn.rnn
        h, c = states
        if self.fused_cell and inp.is_cuda:   # pointwise work in csrc/vine_lstm.cu, GEMMs in bf16
            from .lstm_ops import lstm_seq
            hs, (h, c) = lstm_seq(inp.view(L, S, -1), r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0 + r.bias_hh_l0, h, c, not_done)
            out = self.layer_norm(hs.reshape(L * S, -1))
            return self.mu(out), self.sigma.expand(L * S, -1), self.value(out), (h, c)
        gi = torch.nn.functional.linear(inp, r.weight_ih_l0, r.bias_ih_l0 + r.bias_hh_l0).view(L, S, -1)
        outs = []
        for t in range(L):
            if not_done is not None:
                nd = not_done[t].unsqueeze(-1)
                h, c = h * nd, c * nd
            g = gi[t] + torch.nn.functional.linear(h.to(gi.dtype), r.weight_hh_l0)
            i, f, gg, o = g.float().chunk(4, -1)                         # torch gate order: i, f, g, o
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            outs.append(h)
        out = self.layer_norm(torch.stack(outs).reshape(L * S, -1))
        return self.mu(out), self.sigma.expand(L * S, -1), self.value(out), (h, c)


def neglogp(x, mean, std, logstd):
    return 0.5 * (((x - mean) / std) ** 2).sum(-1) + 0.5 * math.log(2.0 * math.pi) * x.shape[-1] + logstd.sum(-1)


def policy_kl(p0_mu, p0_sigma, p1_mu, p1_sigma):
    c1 = torch.log(p1_sigma / p0_sigma + 1e-5)
    c2 = (p0_sigma ** 2 + (p1_mu - p0_mu) ** 2) / (2.0 * (p1_sigma ** 2 + 1e-5))
    return (c1 + c2 - 0.5).sum(-1).mean()


LR_MIN, LR_MAX = 1e-6, 1e-2   # rl_games AdaptiveScheduler's bounds; LinearScheduler's min_lr is LR_MIN too


NORMALISER_KEYS = ("running_mean_std", "value_mean_std")   # checkpoint prefixes of the input / value normaliser


def rlgames_model_state(model, obs_rms, val_rms):
    """The ``model`` entry of an rl-games 1.5.2 checkpoint (``A2CBase.get_full_state_weights`` -> ``model.state_dict()`` of
    ``ModelA2CContinuousLogStd.Network``): the network under ``a2c_network.*``, the input normaliser under
    ``running_mean_std.*`` ([O], [O], []) and the value normaliser under ``value_mean_std.*`` ([1], [1], []).
    A normaliser passed as None is off (normalize_input / normalize_value False): rl_games builds no such sub-module, so the
    file has none of its keys."""
    sd = {"a2c_network." + k: v.detach().clone() for k, v in model.state_dict().items()}
    for name, rms in zip(NORMALISER_KEYS, (obs_rms, val_rms)):
        if rms is None:
            continue
        for k, v in rms.state_dict().items():
            sd[f"{name}.{k}"] = v.detach().clone()
    return sd


class PPOAgent:
    PDL_MAX_ENVS = 4096   # envs per GPU up to which the rollout is launched with programmatic dependent launch

    def __init__(self, env, train_cfg, device=None, seed=42, use_graphs=False, use_fused_policy=True,
                 use_fused_update=True, grad_allreduce="p2p"):
        c = train_cfg["params"]["config"]
        net = train_cfg["params"]["network"]
        self.env, self.c = env, c
        self.device = device or env.device
        self.n, self.T = env.num_envs, int(c["horizon_length"])
        self.O, self.A = env.num_obs, env.num_acts
        self.gamma, self.tau = float(c["gamma"]), float(c["tau"])
        self.e_clip, self.critic_coef = float(c["e_clip"]), float(c["critic_coef"])
        self.entropy_coef, self.bounds_coef = float(c["entropy_coef"]), float(c["bounds_loss_coef"])
        self.mini_epochs = int(c["mini_epochs"])
        self.batch = self.n * self.T
        self.minibatch = min(int(c["minibatch_size"]), self.batch)
        assert self.batch % self.minibatch == 0, "batch must be a multiple of minibatch_size"
        # rl_games flattens the rollout env-major (swap_and_flatten01), so a minibatch is a slice of envs x all T steps
        assert self.minibatch % self.T == 0, "minibatch_size must be a multiple of horizon_length"
        self.mb_envs = self.minibatch // self.T
        self.kl_threshold = float(c["kl_threshold"])
        opts = self.update_options(train_cfg)
        self.adaptive, self.linear_lr, self.schedule_standard = opts["adaptive"], opts["linear"], opts["standard"]
        self.max_epochs, self.clip_value, self.lr0 = opts["max_epochs"], opts["clip_value"], float(c["learning_rate"])
        self.reward_scale, self.reward_shift = opts["reward_scale"], opts["reward_shift"]
        self.reward_min, self.reward_max = opts["reward_min"], opts["reward_max"]
        self.reward_clamp = self.reward_min > -math.inf or self.reward_max < math.inf
        self.value_bootstrap = bool(c.get("value_bootstrap", False))
        self.normalize_input, self.normalize_value = bool(c["normalize_input"]), bool(c["normalize_value"])
        self.normalize_advantage = bool(c["normalize_advantage"])
        # the kernels' flags of a normaliser that is off (named for the off state: 0 = rl_games' default, normaliser on)
        self._raw_flags = dict(raw_obs=int(not self.normalize_input), raw_value=int(not self.normalize_value))
        self.truncate_grads, self.grad_norm = bool(c.get("truncate_grads", False)), float(c.get("grad_norm", 1.0))
        self.bf16 = bool(c.get("mixed_precision", False))
        # an episode counts as a success when the "Position Success" term (1000 x its weight, V5:1507, V5:186-203) fired in
        # its last step: half of that bonus separates it from every other term at any weight; no weight, no success signal
        w_succ = float(env.cfg["env"].get("POSITION_SUCCESS_REWARD_WEIGHT", 1.0)) if hasattr(env, "cfg") else 1.0
        self.success_threshold = 500.0 * w_succ if w_succ > 0 else float("inf")
        units = net["mlp"]["units"]
        torch.manual_seed(seed)
        dev = self.device
        self.model = ActorCritic(self.O, self.A, units, rnn=net.get("rnn")).to(dev)
        self.has_rnn = self.model.has_rnn
        self.layer_norm = self.has_rnn and isinstance(self.model.layer_norm, nn.LayerNorm)   # rnn.layer_norm
        self.seq_len = int(c.get("seq_len", 4)) if self.has_rnn else 1
        assert self.T % self.seq_len == 0, "horizon_length must be a multiple of seq_len"
        self.obs_rms = RunningMeanStd((self.O,)).to(dev)
        self.val_rms = RunningMeanStd((1,)).to(dev)     # rl_games: RunningMeanStd((value_size,)) -> checkpoint shape [1]
        self.world = vd.rank_world()[1]
        if self.world > 1:  # hvd.setup_algo equivalent: identical parameters on every rank
            for p in self.model.parameters():
                torch.distributed.broadcast(p.data, 0)
        self._want_graphs = bool(use_graphs)
        self._lib = abi.load_library()
        # Both networks run entirely on hand-written sm_100a kernels (tcgen05/TMEM): vine_policy_act / vine_lstm_* for the
        # rollout, vine_ppo_minibatch / vine_lstm_* / vine_ppo_adam for the update.  There is NO silent dispatch: a
        # configuration the kernels do not cover raises here.  torch autograd + cuBLAS/cuDNN + torch Adam exist only as the
        # explicit baseline `use_fused_update=False` (`use_fused_policy=False` additionally takes the policy forward to torch).
        rnn_cfg = net.get("rnn") or {}
        self.fused = self.native_lstm = self.fused_update = False
        if use_fused_update:
            if not use_fused_policy:
                raise ValueError("use_fused_update=True needs use_fused_policy=True (the kernel update reads the kernel rollout's buffers)")
            why = self._kernel_path_gaps(units, rnn_cfg)
            if why:
                raise NotImplementedError(
                    "PPO kernel path does not cover this configuration: " + "; ".join(why) +
                    ". Pass use_fused_update=False for the torch autograd + cuBLAS baseline, or change the configuration.")
            self.native_lstm = self.has_rnn
            self.fused = not self.has_rnn
            self.fused_update = True
        elif use_fused_policy and not self.has_rnn and not self._kernel_path_gaps(units, rnn_cfg, update=False):
            self.fused = True   # baseline update, kernel policy forward (asked for explicitly: use_fused_update=False)
        # CUDA graphs: single GPU always; multi-GPU only for the kernel-only path (its NCCL all-reduces are captured too)
        self.use_graphs = self._want_graphs and (self.world == 1 or (self.fused_update and bool(c.get("graph_nccl", True))))
        # multi-GPU gradient all-reduce of the kernel paths: "p2p" = one-shot over NVLink peer memory inside the reduce / Adam
        # kernels (csrc/vine_p2p.cuh; bit-identical parameters on all ranks), "nccl" = one NCCL all-reduce per minibatch (baseline)
        if grad_allreduce not in ("p2p", "nccl"):
            raise ValueError("grad_allreduce must be 'p2p' or 'nccl'")
        self.grad_allreduce = grad_allreduce if (self.world > 1 and self.fused_update) else "none"
        self._p2p_mlp = self._p2p_lstm = self._p2p_moments = None
        if self.native_lstm:
            self._init_native_lstm(float(c["learning_rate"]))
        elif self.fused_update:
            self._init_fused_update(float(c["learning_rate"]))
        else:
            self.lr_t = torch.tensor(float(c["learning_rate"]), device=dev)   # device-side: no sync in the schedule
            self._epoch_t = torch.zeros((), dtype=torch.float64, device=dev)    # rl_games epoch_num, for the linear schedule
            self.opt = torch.optim.Adam(self.model.parameters(), lr=self.lr_t, eps=1e-8, capturable=True)
        if self.grad_allreduce == "p2p":
            self._p2p_mlp = vd.P2PChannel(self._lib, self._lib.vine_ppo_num_params(self.O) + 4, dev)
            if self.native_lstm:
                self._p2p_lstm = vd.P2PChannel(self._lib, self._lib.vine_lstm_num_params(self.O) + 4, dev)
            self._p2p_moments = vd.P2PChannel(self._lib, 2 * (2 * self.O + 4), dev)   # f64 moments as pairs of 32-bit halves
        T, n = self.T, self.n
        f = lambda *s: torch.zeros(*s, device=dev)  # noqa: E731
        self.b_obs, self.b_act, self.b_mu = f(T, n, self.O), f(T, n, self.A), f(T, n, self.A)
        self.b_nlp, self.b_val, self.b_rew, self.b_done = f(T, n), f(T, n), f(T, n), f(T, n)
        self.b_adv, self.b_ret = f(T, n), f(T, n)
        if self.has_rnn:   # LSTM state of every env, and its snapshots at the start of every seq_len chunk
            H = self.model.rnn_units
            self.rnn_h, self.rnn_c = f(n, H), f(n, H)
            self.b_h, self.b_c = f(T // self.seq_len, n, H), f(T // self.seq_len, n, H)
        self.obs = env.reset()["obs"].clone()
        self.dones = torch.ones(n, device=dev)
        if self.fused_update:   # [T+1, n]: dones seen before step t; row T carries over to the next rollout's row 0
            self._done_ext = torch.ones(T + 1, n, device=dev)
            self.b_done, self.dones = self._done_ext[:T], self._done_ext[T]
        self.last_value = f(n)
        self.epoch = 0
        self.frames = 0
        # device-side statistics: [episodes, successes, return_sum, length_sum] and [a_loss, c_loss, kl, n]
        self.ep_stats = torch.zeros(4, device=dev, dtype=torch.float64)
        self.loss_stats = torch.zeros(4, device=dev, dtype=torch.float64)
        self.ep_ret, self.ep_len = f(n), f(n)
        self._g_rollout = self._g_update = None
        if self.fused or self.native_lstm:   # tcgen05/TMEM policy forward for the rollout
            self._packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=dev)
            if self.native_lstm:
                self._lpacked = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=dev)
            self._obs_mean_f, self._obs_inv_std_f = f(self.O), f(self.O)
            self._val_stats = f(2)
            self._mu_buf, self._val_buf = f(n, self.A), f(n)
            self._refresh_fused(pack=True)

    @staticmethod
    def update_options(train_cfg):
        """The rl_games keys of ``train.params.config`` that select the learning-rate schedule, the value loss and the reward
        shaper, parsed and checked on a plain train-config dict (rl-games 1.5.2 semantics as recalled, DESIGN §9).  Every
        update path (both kernel paths and the torch baseline) implements all of them; a value they cannot honour raises
        here instead of being ignored.  lr_schedule values other than adaptive / linear mean a constant learning rate."""
        c = train_cfg["params"]["config"]
        sched, stype = c.get("lr_schedule"), c.get("schedule_type", "legacy")
        if stype not in ("legacy", "standard"):
            raise ValueError(f"schedule_type {stype!r}: must be 'legacy' (the lr rule after every minibatch) or 'standard' "
                             "(after every mini-epoch, on its mean KL); rl_games would silently keep the learning rate constant")
        max_epochs = int(c.get("max_epochs", -1))
        if sched == "linear" and max_epochs <= 0:
            raise ValueError(f"lr_schedule 'linear' decays the learning rate over max_epochs iterations: max_epochs must be > 0, "
                             f"got {max_epochs}")
        if c.get("schedule_entropy", False):
            raise NotImplementedError("schedule_entropy: True (a linear schedule of entropy_coef) is not implemented: the "
                                      "kernels read entropy_coef as a constant. Set schedule_entropy: False")
        shaper = c.get("reward_shaper") or {}
        if shaper.get("log_val", False):
            raise NotImplementedError("reward_shaper.log_val: True (log of the shifted reward) is not implemented by the rollout "
                                      "kernels or the torch rollout. Remove log_val or set it to False")
        return {"adaptive": sched == "adaptive", "linear": sched == "linear", "standard": stype == "standard",
                "max_epochs": max_epochs, "clip_value": bool(c.get("clip_value", True)),
                "reward_scale": float(shaper.get("scale_value", 1.0)), "reward_shift": float(shaper.get("shift_value", 0.0)),
                "reward_min": float(shaper.get("min_val", -math.inf)), "reward_max": float(shaper.get("max_val", math.inf))}

    def _shaper_fields(self):
        """Reward-shaper fields of VineRolloutPost."""
        return dict(reward_scale=self.reward_scale, reward_shift=self.reward_shift, reward_min=self.reward_min,
                    reward_max=self.reward_max, reward_clamp=int(self.reward_clamp))

    def _schedule_fields(self, mini_epoch, slot):
        """Learning-rate schedule and value-loss fields of the vine_ppo_minibatch launch of (mini-epoch, minibatch slot)."""
        return dict(adaptive_lr=int(self.adaptive), lr_linear=int(self.linear_lr), schedule_standard=int(self.schedule_standard),
                    epoch_begin=int(mini_epoch == 0 and slot == 0), mini_epoch_begin=int(slot == 0),
                    max_epochs=max(self.max_epochs, 0), lr0=self.lr0, kl_threshold=self.kl_threshold, lr_min=LR_MIN,
                    lr_max=LR_MAX, value_loss_unclipped=int(not self.clip_value))

    def _kernel_path_gaps(self, units, rnn_cfg, update=True):
        """Why the hand-written kernel path cannot run this configuration (empty list: it can)."""
        why = []
        if list(units) != [256, 128, 64]:
            why.append(f"network.mlp.units {list(units)} (kernels are built for [256, 128, 64])")
        if self.A != 2:
            why.append(f"{self.A} actions (kernels: 2)")
        if self.O > (30 if self.has_rnn else 31):
            why.append(f"{self.O} observations (kernels: <= {30 if self.has_rnn else 31})")
        if self.has_rnn:   # concat_input and layer_norm may each be on or off
            if int(rnn_cfg.get("units", 0)) != 256:
                why.append(f"network.rnn.units {rnn_cfg.get('units')} (kernels are built for an LSTM of 256 units)")
            if int(rnn_cfg.get("layers", 1)) != 1 or rnn_cfg.get("before_mlp", False):
                why.append("network.rnn with layers != 1 or before_mlp True (kernels: one LSTM layer after the MLP)")
        return why

    def _param_order(self):
        """The flat parameter order of include/vine_b200.h (vine_ppo_*)."""
        m = self.model
        return [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias,
                m.actor_mlp[4].weight, m.actor_mlp[4].bias, m.mu.weight, m.mu.bias, m.value.weight, m.value.bias, m.sigma]

    @torch.no_grad()
    def _init_fused_update(self, lr):
        dev, lib = self.device, self._lib
        order = self._param_order()
        P = lib.vine_ppo_num_params(self.O)
        self.flat = torch.cat([p.detach().reshape(-1) for p in order]).contiguous()
        assert self.flat.numel() == P
        o = 0
        for p in order:   # the torch modules become views of the flat vector the kernels update
            p.data = self.flat[o:o + p.numel()].view_as(p)
            o += p.numel()
        self.adam_m, self.adam_v = torch.zeros(P, device=dev), torch.zeros(P, device=dev)
        self.ppo_state = torch.zeros(abi.PPO_STATE_FLOATS, device=dev)
        self.ppo_state[0] = lr
        self.lr_t = self.ppo_state[0]                                      # 0-dim view: the device-side learning rate
        self._ctas = lib.vine_ppo_max_ctas()
        self._ws = torch.empty(self._ctas, abi.PPO_WS_FLOATS, device=dev)
        self._flat_grads = torch.zeros(P + 4, device=dev)
        self._logstd_old = torch.zeros(self.n // self.mb_envs, 2, device=dev)   # per minibatch slot (update_mu_sigma)
        z = lambda: torch.zeros(self.T, self.n, device=dev)  # noqa: E731
        self._val_old_n, self._ret_n, self._adv_n = z(), z(), z()
        self._mb_structs = self._roll_structs = None
        self._rng_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self._moments = torch.zeros(2 * self.O + 4, dtype=torch.float64, device=dev)
        self._adv_stats = torch.zeros(2, device=dev)
        self._clip_ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=dev) if self.truncate_grads else None

    # ------------------------------------------------------------------ reference network on kernels only
    def _lstm_param_order(self):
        """Flat parameter order of the recurrent half (include/vine_b200.h, vine_lstm_*): the tensors whose storage is the flat
        vector.  The layout is the same with either switch of the rnn block off; the slots the torch block then lacks hold
        tensors of their own that start at 0 and get a gradient of exactly 0, so Adam never moves them: LayerNorm gamma / beta
        with layer_norm off, and with concat_input off the observation columns of W_ih, whose whole [1024, 64 + O] slot is
        _lstm_wih (the torch weight_ih_l0 [1024, 64] is its first 64 columns)."""
        m, r = self.model, self.model.rnn.rnn
        return [self._lstm_wih, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, *self._lstm_ln, m.mu.weight, m.mu.bias,
                m.value.weight, m.value.bias, m.sigma]

    @torch.no_grad()
    def _init_native_lstm(self, lr):
        from .lstm_native import NativeLstmPath
        dev, lib, m = self.device, self._lib, self.model
        z = lambda *s: torch.zeros(*s, device=dev)  # noqa: E731
        # MLP half: the flat layout of vine_ppo_* with the (unused) 64-wide heads kept as zeros
        mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
               m.actor_mlp[4].bias]
        self._mlp_dummy = [z(2, 64), z(2), z(1, 64), z(1), z(2)]
        self.flat = torch.cat([p.detach().reshape(-1) for p in mlp + self._mlp_dummy]).contiguous()
        assert self.flat.numel() == lib.vine_ppo_num_params(self.O)
        o = 0
        for p in mlp + self._mlp_dummy:
            p.data = self.flat[o:o + p.numel()].view_as(p)
            o += p.numel()
        r, H = m.rnn.rnn, m.rnn_units
        self._lstm_wih = r.weight_ih_l0 if m.concat_input else torch.cat([r.weight_ih_l0.detach(), z(4 * H, self.O)], 1)
        self._lstm_ln = [m.layer_norm.weight, m.layer_norm.bias] if self.layer_norm else [z(H), z(H)]
        order = self._lstm_param_order()
        self.flat_l = torch.cat([p.detach().reshape(-1) for p in order]).contiguous()
        assert self.flat_l.numel() == lib.vine_lstm_num_params(self.O)
        o = 0
        for p in order:
            p.data = self.flat_l[o:o + p.numel()].view_as(p)
            o += p.numel()
        if not m.concat_input:   # the torch weight: a strided view of the MLP columns of the flat W_ih
            r.weight_ih_l0.data = self._lstm_wih[:, :r.input_size]
        self.adam_m, self.adam_v = torch.zeros_like(self.flat), torch.zeros_like(self.flat)
        self.adam_ml, self.adam_vl = torch.zeros_like(self.flat_l), torch.zeros_like(self.flat_l)
        self.ppo_state = torch.zeros(abi.PPO_STATE_FLOATS, device=dev)
        self.ppo_state[0] = lr
        self.lr_t = self.ppo_state[0]
        self._logstd_old = z(self.n // self.mb_envs, 2)                           # per minibatch slot (update_mu_sigma)
        zz = lambda: z(self.T, self.n)  # noqa: E731
        self._val_old_n, self._ret_n, self._adv_n = zz(), zz(), zz()
        self._mb_structs = self._roll_structs = None
        self._rng_counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self._moments = torch.zeros(2 * self.O + 4, dtype=torch.float64, device=dev)
        self._adv_stats = z(2)
        self._clip_ws = z(abi.GRAD_CLIP_WS_FLOATS) if self.truncate_grads else None
        L, chunks, tiles_n = self.seq_len, self.T // self.seq_len, -(-self.n // 128)
        hyper = dict(e_clip=self.e_clip, critic_coef=self.critic_coef, entropy_coef=self.entropy_coef,
                     bounds_loss_coef=self.bounds_coef, clip_value=self.clip_value, schedule=self._schedule_fields)
        self._path = NativeLstmPath(self.O, L, chunks * self.mb_envs, dev, hyper, layer_norm=self.layer_norm,
                                    concat_input=m.concat_input)
        from .lstm_native import TB
        bf = lambda *s: torch.zeros(*s, dtype=torch.bfloat16, device=dev)  # noqa: E731
        self._r_U, self._r_HM = bf(tiles_n, TB), bf(tiles_n, 2, TB)
        self._r_HH = [bf(tiles_n, 2, TB), bf(tiles_n, 2, TB)]          # current / next hidden state tiles
        self._r_C = [z(self.n, 256), z(self.n, 256)]
        self._r_cur = 0
        self._HH_saved, self._C_saved = bf(chunks, tiles_n, 2, TB), z(chunks, self.n, 256)
        self._nd_ext = torch.zeros(self.T + 1, self.n, device=dev)       # 1 - dones before step t
        self._ones_n = torch.ones(self.n, device=dev)
        self._scal = z(self.T, self.n, 8)
        R = self._path.R                                                 # minibatch rows per step (padded to whole tiles)
        self._mb_obs, self._mb_scal, self._mb_nd = z(L, R, self.O), z(L, R, 8), z(L, R)

    @torch.no_grad()
    def _rollout_native_lstm(self):
        """Rollout of the recurrent policy on kernels only: per step vine_policy_act (MLP -> U tiles, obs copy), vine_lstm_mask,
        vine_lstm_step, vine_lstm_head (LayerNorm, heads, sampling, buffer writes), the fused env step, vine_rollout_post."""
        env, lib, T, n, L = self.env, self._lib, self.T, self.n, self.seq_len
        ptr = lambda x: x.data_ptr()  # noqa: E731
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        common = dict(packed=ptr(self._packed), obs=ptr(env._obs_clamped), n=n, num_obs=self.O, **self._stat_ptrs(),
                      **self._raw_flags, u_no_obs=int(not self.model.concat_input))
        no_ln = int(not self.layer_norm)
        seed, goff = int(env._seed) ^ 0x5DEECE66D, int(env._global_env_offset)
        vstats = common["value_stats"]
        self._done_ext[0].copy_(self._done_ext[T])
        torch.sub(self._ones_n, self._done_ext[0], out=self._nd_ext[0])   # later rows are written by vine_rollout_post
        for t in range(T + 1):
            cur, nxt = self._r_cur, self._r_cur ^ 1
            last = t == T
            if not last and t % L == 0:   # LSTM state at the start of every seq_len chunk (truncated BPTT restarts here)
                self._HH_saved[t // L].copy_(self._r_HH[cur])
                self._C_saved[t // L].copy_(self._r_C[cur])
            act = abi.VinePolicyAct(u_out=ptr(self._r_U), obs_copy=None if last else ptr(self.b_obs[t]), **common)
            assert lib.vine_policy_act(C.byref(act), stream) == 0
            assert lib.vine_lstm_mask(C.c_void_p(ptr(self._r_HH[cur])), C.c_void_p(ptr(self._nd_ext[t])), n,
                                      C.c_void_p(ptr(self._r_HM)), stream) == 0
            st = abi.VineLstmStep(params=ptr(self._lpacked), u=ptr(self._r_U), hm=ptr(self._r_HM), c_prev=ptr(self._r_C[cur]),
                                  not_done=ptr(self._nd_ext[t]), c=ptr(self._r_C[nxt]), hh=ptr(self._r_HH[nxt]), n=n)
            assert lib.vine_lstm_step(C.byref(st), stream) == 0
            if last:   # bootstrap value of the final observation: the persistent state is NOT advanced
                hd = abi.VineLstmHead(params=ptr(self._lpacked), hh=ptr(self._r_HH[nxt]), value_stats=vstats,
                                      value=ptr(self.last_value), n=n, raw_value=self._raw_flags["raw_value"],
                                      no_layer_norm=no_ln)
                assert lib.vine_lstm_head(C.byref(hd), stream) == 0
                break
            hd = abi.VineLstmHead(params=ptr(self._lpacked), hh=ptr(self._r_HH[nxt]), value_stats=vstats,
                                  mu=ptr(self.b_mu[t]), value=ptr(self.b_val[t]), logstd=ptr(self.model.sigma),
                                  rng_counter=ptr(self._rng_counter), actions=ptr(self.b_act[t]), neglogp=ptr(self.b_nlp[t]),
                                  env_actions=ptr(env.actions), n=n, seed=seed, global_env_offset=goff,
                                  raw_value=self._raw_flags["raw_value"], no_layer_norm=no_ln)
            assert lib.vine_lstm_head(C.byref(hd), stream) == 0
            self._r_cur = nxt
            env.step_device()
            post = abi.VineRolloutPost(rewards=ptr(env.rew_buf), resets=ptr(env.reset_buf), timeouts=ptr(env.timeout_buf),
                                       values=ptr(self.b_val[t]), shaped_rewards=ptr(self.b_rew[t]), dones_next=ptr(self._done_ext[t + 1]),
                                       ep_return=ptr(self.ep_ret), ep_length=ptr(self.ep_len), ep_stats=ptr(self.ep_stats),
                                       rng_counter=ptr(self._rng_counter), n=n, gamma=self.gamma,
                                       value_bootstrap=int(self.value_bootstrap), success_reward_threshold=self.success_threshold,
                                       not_done_next=ptr(self._nd_ext[t + 1]), **self._shaper_fields())
            assert lib.vine_rollout_post(C.byref(post), stream) == 0
        if self._r_cur != 0:   # odd horizon: keep the persistent state in buffer 0 so a captured graph can be replayed
            self._r_HH[0].copy_(self._r_HH[1])
            self._r_C[0].copy_(self._r_C[1])
            self._r_cur = 0
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        rc = lib.vine_gae(p(self.b_rew), p(self.b_val), p(self.b_done), p(self.last_value), p(self.dones),
                          T, n, self.gamma, self.tau, p(self.b_adv), p(self.b_ret), stream)
        assert rc == 0

    @torch.no_grad()
    def _update_native_lstm(self):
        """Update of the recurrent policy on kernels only (ppo/lstm_native.py lists the launches of one minibatch)."""
        T, n, L, E, lib = self.T, self.n, self.seq_len, self.mb_envs, self._lib
        chunks = T // L
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        ptr = lambda x: x.data_ptr()  # noqa: E731
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        if self._mb_structs is None:
            self._prologue = self._prologue_struct()
            self._mb_structs = True
        assert lib.vine_ppo_moments(C.byref(self._prologue), stream) == 0
        self._allreduce_moments(stream)
        assert lib.vine_ppo_finalize(C.byref(self._prologue), stream) == 0
        self._logstd_old.copy_(self.model.sigma.expand_as(self._logstd_old))
        # per-row scalars of the loss, once per iteration: action(2), mu_old(2), neglogp_old, value_old, return, advantage
        torch.cat([self.b_act, self.b_mu, self.b_nlp.unsqueeze(-1), self._val_old_n.unsqueeze(-1), self._ret_n.unsqueeze(-1),
                   self._adv_n.unsqueeze(-1)], dim=-1, out=self._scal)
        path = self._path
        pm = self._p2p_mlp.ptr if self._p2p_mlp is not None else None
        pl = self._p2p_lstm.ptr if self._p2p_lstm is not None else None
        for k in range(self.mini_epochs):
            for e0 in range(0, n, E):
                # rows of the minibatch ordered [step in chunk][chunk, env] + the initial LSTM state of every sequence: one launch
                ga = abi.VineLstmGather(obs=ptr(self.b_obs), scalars=ptr(self._scal), not_done=ptr(self._nd_ext),
                                        c_saved=ptr(self._C_saved), hh_saved=ptr(self._HH_saved), mb_obs=ptr(self._mb_obs),
                                        mb_scalars=ptr(self._mb_scal), mb_not_done=ptr(self._mb_nd), c0=ptr(path.C0),
                                        hm0=ptr(path.HM[0]), seq_len=L, chunks=chunks, num_envs=n, env_begin=e0, env_count=E,
                                        num_obs=self.O, step_rows=path.R)
                assert lib.vine_lstm_gather(C.byref(ga), stream) == 0
                obs_stats = (self._obs_mean_f, self._obs_inv_std_f) if self.normalize_input else (None, None)   # None: off
                path.gradients(self._packed, self._lpacked, self._mb_obs, self._mb_scal, self._mb_nd, *obs_stats,
                               self._val_stats if self.normalize_value else None, self.model.sigma, self._logstd_old[e0 // E],
                               self.ppo_state, writeback=(self._scal, L, chunks, n, e0, E), p2p=(pm, pl), position=(k, e0 // E))
                if self.grad_allreduce == "nccl":   # baseline: ONE NCCL all-reduce per minibatch (gradients + loss statistics)
                    torch.distributed.all_reduce(path.flat_g)
                sc = 1.0 / self.world                # p2p: the Adam kernels add the ranks' buffers themselves (vine_p2p.cuh)
                if self.truncate_grads:
                    self._clip_and_adam_native_lstm(path, sc, pm, pl, stream)
                    continue
                assert lib.vine_ppo_adam(p(path.flat_g_mlp), sc, p(self.flat), p(self.adam_m), p(self.adam_v), p(self._packed),
                                         p(self.ppo_state), self.O, 0.9, 0.999, 1e-8, 0, pm, stream) == 0
                assert lib.vine_lstm_adam(p(path.flat_g_lstm), sc, p(self.flat_l), p(self.adam_ml), p(self.adam_vl), p(self._lpacked),
                                          p(self.ppo_state), self.O, 0.9, 0.999, 1e-8, pl, stream) == 0

    def _clip_and_adam_native_lstm(self, path, sc, pm, pl, stream):
        """truncate_grads: ONE norm over both gradient vectors (the MLP half without its unused head slots, the whole
        recurrent half), then both Adam launches with the coefficient.  With peer memory the clip kernel consumes both
        channels and leaves the rank sums in flat_g_*, so Adam runs without a channel.  The norm is that of exactly
        ActorCritic's parameters with either rnn switch off too: the recurrent slots the block then lacks (W_ih's observation
        columns, LayerNorm gamma / beta; _lstm_param_order) carry a gradient of exactly 0."""
        lib = self._lib
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        P, PL = path.P_mlp, path.P_lstm
        counted = P - sum(t.numel() for t in self._mlp_dummy)
        assert lib.vine_grad_clip(p(path.flat_g_mlp), counted, P + 4, p(path.flat_g_lstm), PL, PL + 4, sc, self.grad_norm,
                                  p(self.ppo_state), p(self._clip_ws), pm, pl, stream) == 0
        coef = C.c_void_p(self.ppo_state.data_ptr() + abi.PPO_STATE_CLIP_COEF * 4)
        assert lib.vine_ppo_adam_clipped(p(path.flat_g_mlp), sc, p(self.flat), p(self.adam_m), p(self.adam_v), p(self._packed),
                                         p(self.ppo_state), self.O, 0.9, 0.999, 1e-8, 0, coef, None, stream) == 0
        assert lib.vine_lstm_adam_clipped(p(path.flat_g_lstm), sc, p(self.flat_l), p(self.adam_ml), p(self.adam_vl), p(self._lpacked),
                                          p(self.ppo_state), self.O, 0.9, 0.999, 1e-8, coef, None, stream) == 0

    def _stat_ptrs(self, value=True):
        """Device pointers of the normalisation statistics the kernels read, as struct fields; a normaliser that is off passes
        None (its kernel flag is set, nothing is read).  value=False: only the observation statistics."""
        ptrs = dict(obs_mean=self._obs_mean_f.data_ptr() if self.normalize_input else None,
                    obs_inv_std=self._obs_inv_std_f.data_ptr() if self.normalize_input else None)
        if value:
            ptrs["value_stats"] = self._val_stats.data_ptr() if self.normalize_value else None
        return ptrs

    def _prologue_struct(self):
        """VinePpoPrologue of the kernel update: running statistics, normalised value targets and advantages."""
        ptr = lambda x: x.data_ptr()  # noqa: E731
        io, iv = self.normalize_input, self.normalize_value
        obs_fields = dict(obs=ptr(self.b_obs), obs_mean=ptr(self.obs_rms.running_mean), obs_var=ptr(self.obs_rms.running_var),
                          obs_count=ptr(self.obs_rms.count), obs_mean_f=ptr(self._obs_mean_f),
                          obs_inv_std_f=ptr(self._obs_inv_std_f)) if io else {}
        val_fields = dict(val_mean=ptr(self.val_rms.running_mean), val_var=ptr(self.val_rms.running_var),
                          val_count=ptr(self.val_rms.count), value_stats=ptr(self._val_stats)) if iv else {}
        return abi.VinePpoPrologue(
            values=ptr(self.b_val), returns=ptr(self.b_ret), moments=ptr(self._moments), adv_stats=ptr(self._adv_stats),
            values_n=ptr(self._val_old_n), returns_n=ptr(self._ret_n), advantages_n=ptr(self._adv_n), count=self.T * self.n,
            num_obs=self.O, world=self.world, normalize_advantage=int(self.normalize_advantage), **obs_fields, **val_fields,
            **self._raw_flags)

    def _allreduce_moments(self, stream):
        """Sum over the ranks of the f64 running-statistics moments (observations, values, advantages), once per iteration:
        over the peer-memory channel (one single-block launch) or, baseline, one NCCL all-reduce."""
        if self.world == 1:
            return
        if self._p2p_moments is not None:
            assert self._lib.vine_p2p_allreduce_f64(self._p2p_moments.ptr, C.c_void_p(self._moments.data_ptr()),
                                                    self._moments.numel(), stream) == 0
        else:
            torch.distributed.all_reduce(self._moments)

    @torch.no_grad()
    def _refresh_fused(self, pack=False):
        """Refresh the normalisation statistics the kernels read; ``pack``: also re-pack the weights (bf16, tensor-core
        operand layout) -- only needed when something other than vine_ppo_adam changed them."""
        if self.normalize_input:   # a normaliser that is off has no statistics the kernels read
            self._obs_mean_f.copy_(self.obs_rms.running_mean.float())
            self._obs_inv_std_f.copy_(torch.rsqrt(self.obs_rms.running_var.float() + self.obs_rms.eps))
        if self.normalize_value:
            self._val_stats.copy_(torch.cat([self.val_rms.running_mean.float().reshape(1),
                                             torch.sqrt(self.val_rms.running_var.float() + self.val_rms.eps).reshape(1)]))
        if pack:
            p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            if self.native_lstm:
                m = self.model
                mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias,
                       m.actor_mlp[4].weight, m.actor_mlp[4].bias] + self._mlp_dummy[:4]
                assert self._lib.vine_mlp_pack(*[p(t) for t in mlp], self.O, p(self._packed), st) == 0
                assert self._lib.vine_lstm_pack(*[p(t) for t in self._lstm_param_order()[:10]], self.O, p(self._lpacked), st) == 0
            else:
                args = [p(t) for t in self._param_order()[:10]]
                assert self._lib.vine_mlp_pack(*args, self.O, p(self._packed), st) == 0

    @property
    def lr(self):
        return float(self.lr_t)

    # ------------------------------------------------------------------ acting
    @torch.no_grad()
    def _policy(self, obs, states=None):
        """mu, logstd, de-normalised value and the next LSTM state for one observation per env."""
        if self.fused and obs.shape[0] == self.n:
            p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
            s = self._stat_ptrs()   # NULL statistics: that normaliser is off
            rc = self._lib.vine_mlp_forward(p(self._packed), p(obs), s["obs_mean"], s["obs_inv_std"], self.n, self.O,
                                            s["value_stats"], p(self._mu_buf), p(self._val_buf),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            return self._mu_buf, self.model.sigma.detach().expand(self.n, -1), self._val_buf, None
        x = self.obs_rms(obs) if self.normalize_input else obs
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.bf16):
            mu, logstd, value, states = self.model(x, states)
        mu, logstd, value = mu.float(), logstd.float(), value.float().squeeze(-1)
        if self.normalize_value:
            value = self.val_rms(value, unnorm=True)
        return mu, logstd, value, states

    @torch.no_grad()
    def _rollout_fused(self):
        """The rollout on hand-written kernels only: per control step vine_policy_act (normalise, MLP on tcgen05,
        sample, neglogp, all rollout-buffer writes), the fused env step, vine_rollout_post; then the last value and GAE."""
        env, lib, T, n = self.env, self._lib, self.T, self.n
        if self._roll_structs is None:
            ptr = lambda x: x.data_ptr()  # noqa: E731
            common = dict(packed=ptr(self._packed), obs=ptr(env._obs_clamped), n=n, num_obs=self.O,
                          seed=int(env._seed) ^ 0x5DEECE66D, global_env_offset=int(env._global_env_offset),
                          **self._stat_ptrs(), **self._raw_flags)
            acts = [abi.VinePolicyAct(mu=ptr(self.b_mu[t]), value=ptr(self.b_val[t]), logstd=ptr(self.model.sigma),
                                      rng_counter=ptr(self._rng_counter), actions=ptr(self.b_act[t]),
                                      neglogp=ptr(self.b_nlp[t]), obs_copy=ptr(self.b_obs[t]), env_actions=ptr(env.actions),
                                      **common) for t in range(T)]
            posts = [abi.VineRolloutPost(rewards=ptr(env.rew_buf), resets=ptr(env.reset_buf), timeouts=ptr(env.timeout_buf),
                                         values=ptr(self.b_val[t]), shaped_rewards=ptr(self.b_rew[t]),
                                         dones_next=ptr(self._done_ext[t + 1]), ep_return=ptr(self.ep_ret),
                                         ep_length=ptr(self.ep_len), ep_stats=ptr(self.ep_stats),
                                         rng_counter=ptr(self._rng_counter), n=n, gamma=self.gamma,
                                         value_bootstrap=int(self.value_bootstrap), success_reward_threshold=self.success_threshold,
                                         **self._shaper_fields()) for t in range(T)]
            last = abi.VinePolicyAct(mu=ptr(self._mu_buf), value=ptr(self.last_value), **common)
            self._roll_structs = (acts, posts, last)
        acts, posts, last = self._roll_structs
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self._done_ext[0].copy_(self._done_ext[T])
        for t in range(T):
            assert lib.vine_policy_act(C.byref(acts[t]), stream) == 0
            env.step_device()
            assert lib.vine_rollout_post(C.byref(posts[t]), stream) == 0
        assert lib.vine_policy_act(C.byref(last), stream) == 0
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        rc = lib.vine_gae(p(self.b_rew), p(self.b_val), p(self.b_done), p(self.last_value), p(self.dones),
                          T, n, self.gamma, self.tau, p(self.b_adv), p(self.b_ret), stream)
        assert rc == 0

    @torch.no_grad()
    def _rollout(self):
        if self.native_lstm or self.fused_update:
            # programmatic dependent launch for the rollout's chain of few-microsecond kernels (6 per env step at 4096 envs:
            # rollout 0.842 -> 0.806 ms); it does not pay for longer kernels (16,384 envs: rollout 1.37 -> 1.71 ms; the update
            # at any size), so it is on only here and only for small batches.  Captured graphs keep the mode of their capture.
            pdl = self.n <= self.PDL_MAX_ENVS
            before = self._lib.vine_set_programmatic_launch(1 if pdl else 0)
            try:
                return self._rollout_native_lstm() if self.native_lstm else self._rollout_fused()
            finally:
                self._lib.vine_set_programmatic_launch(before)
        env = self.env
        for t in range(self.T):
            states = None
            if self.has_rnn:
                if t % self.seq_len == 0:
                    self.b_h[t // self.seq_len], self.b_c[t // self.seq_len] = self.rnn_h, self.rnn_c
                states = (self.rnn_h, self.rnn_c)
            mu, logstd, value, states = self._policy(self.obs, states)
            sigma = torch.exp(logstd)
            action = mu + sigma * torch.randn_like(mu)
            self.b_obs[t], self.b_act[t], self.b_mu[t] = self.obs, action, mu
            self.b_nlp[t], self.b_val[t], self.b_done[t] = neglogp(action, mu, sigma, logstd), value, self.dones
            env.actions.copy_(torch.clamp(action, -1.0, 1.0))                  # rl_games preprocess_actions
            env.step_device()                                                  # ONE fused kernel launch
            rew, dones, timeouts = env.rew_buf, env.reset_buf, env.timeout_buf
            shaped = self._shape_rewards(rew)
            if self.value_bootstrap:                                           # Vine5LinkMovingBasePPO.yaml:56
                shaped = shaped + self.gamma * value * timeouts.float()
            self.b_rew[t] = shaped
            # episode statistics; success == the 1000-point "Position Success" term fired (V5:1507)
            self.ep_ret += rew
            self.ep_len += 1
            d = dones.to(torch.float32)
            self.ep_stats += torch.stack([d.sum(), (d * (rew > self.success_threshold)).sum(), (d * self.ep_ret).sum(),
                                          (d * self.ep_len).sum()]).double()
            self.ep_ret *= 1.0 - d
            self.ep_len *= 1.0 - d
            if self.has_rnn:   # finished envs start their next episode from a zero state
                nd = (1.0 - d).unsqueeze(-1)
                self.rnn_h.copy_(states[0] * nd)
                self.rnn_c.copy_(states[1] * nd)
            self.obs.copy_(env._obs_clamped)
            self.dones.copy_(d)
        _, _, last_value, _ = self._policy(self.obs, (self.rnn_h, self.rnn_c) if self.has_rnn else None)
        self.last_value.copy_(last_value)
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        rc = self._lib.vine_gae(p(self.b_rew), p(self.b_val), p(self.b_done), p(self.last_value), p(self.dones),
                                self.T, self.n, self.gamma, self.tau, p(self.b_adv), p(self.b_ret),
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0

    def play_steps(self):
        if self._g_rollout is not None:
            self._g_rollout.replay()
        else:
            self._rollout()
        self.frames += self.T * self.n * self.world

    @torch.no_grad()
    def evaluate(self, steps, deterministic=True):
        """Play mode (reference: train.py test=True -> rl_games player.run, `deterministic: True` by default): roll the policy
        without learning; deterministic = act with the mean.  The rollout kernels sample mu + exp(logstd) eps, so the mean
        action is obtained by running them with logstd = -40 (sigma = 4e-18, below f32 resolution of any mu)."""
        sigma = self.model.sigma.data
        keep = sigma.clone()
        if deterministic:
            sigma.fill_(-40.0)
        try:
            self.pop_stats()
            for _ in range(max(1, steps // self.T)):
                self._rollout()
            torch.cuda.synchronize(self.device)
        finally:
            sigma.copy_(keep)
        return self.pop_stats()

    def _shape_rewards(self, rew):
        """rl_games DefaultRewardsShaper without log_val: clamp((r + shift) * scale, min_val, max_val); the shift is added only
        when non-zero and the clamp applied only with a finite bound, so the default is exactly r * scale."""
        r = rew + self.reward_shift if self.reward_shift != 0.0 else rew
        r = r * self.reward_scale
        return torch.clamp(r, self.reward_min, self.reward_max) if self.reward_clamp else r

    # ------------------------------------------------------------------ learning
    def _update_lr(self, kl):
        """One run of the learning-rate rule (rl_games scheduler.update) on the device-side lr; kl = the rank-mean KL."""
        if self.adaptive:
            lr = self.lr_t
            lr = torch.where(kl > 2.0 * self.kl_threshold, torch.clamp(lr / 1.5, min=LR_MIN), lr)
            lr = torch.where(kl < 0.5 * self.kl_threshold, torch.clamp(lr * 1.5, max=LR_MAX), lr)
            self.lr_t.copy_(lr)
        elif self.linear_lr:   # LinearScheduler(use_epochs=True), epoch = rl_games epoch_num of this iteration
            left = torch.clamp(self.max_epochs - self._epoch_t, min=0.0)
            self.lr_t.copy_(LR_MIN + (self.lr0 - LR_MIN) * (left / self.max_epochs))

    def _update(self):
        T, n, L = self.T, self.n, self.seq_len
        obs, act, mu_old = self.b_obs, self.b_act, self.b_mu                  # [T, n, .]
        nlp_old, val_old, ret = self.b_nlp, self.b_val, self.b_ret            # [T, n]
        adv = ret - val_old
        with torch.no_grad():
            if self.normalize_input:
                self.obs_rms.update(obs.reshape(T * n, self.O))
                obs = self.obs_rms(obs)
            if self.normalize_value:
                self.val_rms.update(torch.cat([val_old.reshape(-1), ret.reshape(-1)]))
                val_old, ret = self.val_rms(val_old), self.val_rms(ret)
            if self.normalize_advantage:
                s = torch.stack([adv.sum(), (adv * adv).sum()]).double()
                cnt = float(T * n * self.world)
                if self.world > 1:
                    torch.distributed.all_reduce(s)
                mean = s[0] / cnt
                std = torch.sqrt(torch.clamp((s[1] - cnt * mean * mean) / (cnt - 1.0), min=0.0))
                adv = (adv - mean.float()) / (std.float() + 1e-8)
            # sigma of the policy each row was last evaluated with, per minibatch slot (rl_games dataset.update_mu_sigma)
            sigma_old = torch.exp(self.model.sigma.detach()).clone().expand(n // self.mb_envs, -1).clone()
            not_done = 1.0 - self.b_done
            self._epoch_t += 1.0
        params = [p for p in self.model.parameters()]
        E = self.mb_envs

        def mb(x, e0):
            """[T, n, ...] -> minibatch rows ordered (chunk, step-in-chunk, env): [L, (T/L)*E, ...] flattened."""
            y = x[:, e0:e0 + E]
            y = y.reshape(T // L, L, E, *x.shape[2:]).transpose(0, 1)
            return y.reshape(L, (T // L) * E, *x.shape[2:])

        for _ in range(self.mini_epochs):
            ep_kls = []
            for e0 in range(0, n, E):
                o_mb = mb(obs, e0)                                             # [L, S, O]
                flat = lambda x: mb(x, e0).reshape(L * (T // L) * E, *x.shape[2:])  # noqa: E731
                states = nd = None
                if self.has_rnn:
                    H = self.model.rnn_units
                    states = (self.b_h[:, e0:e0 + E].reshape(-1, H), self.b_c[:, e0:e0 + E].reshape(-1, H))
                    nd = mb(not_done, e0)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.bf16):
                    mu, logstd, value, _ = self.model(o_mb, states, nd)
                mu, logstd, value = mu.float(), logstd.float(), value.float().squeeze(-1)
                sigma = torch.exp(logstd)
                nlp = neglogp(flat(act), mu, sigma, logstd)
                ratio = torch.exp(flat(nlp_old) - nlp)
                a, vo, r = flat(adv), flat(val_old), flat(ret)
                a_loss = torch.max(-a * ratio, -a * torch.clamp(ratio, 1.0 - self.e_clip, 1.0 + self.e_clip)).mean()
                if self.clip_value:
                    v_clip = vo + (value - vo).clamp(-self.e_clip, self.e_clip)
                    c_loss = torch.max((value - r) ** 2, (v_clip - r) ** 2).mean()
                else:
                    c_loss = ((value - r) ** 2).mean()
                b_loss = (torch.clamp_min(mu - 1.1, 0.0) ** 2 + torch.clamp_max(mu + 1.1, 0.0) ** 2).sum(-1).mean()
                entropy = (0.5 + 0.5 * math.log(2 * math.pi) + logstd).sum(-1).mean()
                loss = a_loss + 0.5 * c_loss * self.critic_coef - self.entropy_coef * entropy + b_loss * self.bounds_coef
                self.opt.zero_grad(set_to_none=False)
                loss.backward()
                with torch.no_grad():
                    kl = policy_kl(mu.detach(), sigma.detach(), flat(mu_old), sigma_old[e0 // E].expand_as(mu))
                    # a2c_common.train_epoch: dataset.update_mu_sigma(cmu, csigma) -- the next mini-epoch's KL is against this pass
                    unmb = mu.detach().reshape(L, T // L, E, -1).transpose(0, 1).reshape(T, E, -1)
                    mu_old[:, e0:e0 + E] = unmb
                    sigma_old[e0 // E] = sigma.detach()[0]
                    if self.world > 1:  # ONE collective per minibatch: gradients + KL
                        g = torch.cat([p.grad.reshape(-1) for p in params])
                        g, extra = vd.allreduce_mean_(g, kl.reshape(1))
                        kl = extra[0]
                        o = 0
                        for p in params:
                            p.grad.copy_(g[o:o + p.numel()].view_as(p))
                            o += p.numel()
                    if self.truncate_grads:
                        nn.utils.clip_grad_norm_(params, self.grad_norm)
                self.opt.step()
                with torch.no_grad():
                    if self.schedule_standard:
                        ep_kls.append(kl)
                    else:
                        self._update_lr(kl)
                    self.loss_stats += torch.stack([a_loss.detach(), c_loss.detach(), kl,
                                                    torch.ones((), device=kl.device)]).double()
            if self.schedule_standard:   # rl_games schedule_type standard: once per mini-epoch, on its mean KL
                with torch.no_grad():
                    self._update_lr(torch.stack(ep_kls).mean())
        if self.fused or self.native_lstm:
            self._refresh_fused(pack=True)

    @torch.no_grad()
    def _update_fused(self):
        """The update on hand-written kernels only: per minibatch ONE fused tcgen05 launch (forward, losses, backward,
        weight gradients), the partial-gradient reduction, [one NCCL all-reduce of grads + loss statistics], Adam."""
        T, n, lib = self.T, self.n, self._lib
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        if self._mb_structs is None:
            self._prologue = self._prologue_struct()
        # running statistics + normalised targets: f64 sufficient statistics, [one all-reduce], finalize
        assert lib.vine_ppo_moments(C.byref(self._prologue), stream) == 0
        self._allreduce_moments(stream)
        assert lib.vine_ppo_finalize(C.byref(self._prologue), stream) == 0
        self._logstd_old.copy_(self.model.sigma.expand_as(self._logstd_old))
        if self._mb_structs is None:
            ptr = lambda x: x.data_ptr()  # noqa: E731
            self._mb_structs = [[abi.VinePpoMinibatch(
                packed=ptr(self._packed), obs=ptr(self.b_obs), actions=ptr(self.b_act), mu_old=ptr(self.b_mu),
                neglogp_old=ptr(self.b_nlp), values_old=ptr(self._val_old_n), returns=ptr(self._ret_n),
                advantages=ptr(self._adv_n), **self._stat_ptrs(value=False), raw_obs=self._raw_flags["raw_obs"],
                logstd=ptr(self.model.sigma), logstd_old=ptr(self._logstd_old[e0 // self.mb_envs]), workspace=ptr(self._ws),
                state=ptr(self.ppo_state), debug_out=None, horizon=T, num_envs=n, env_begin=e0, env_count=self.mb_envs,
                num_obs=self.O, workspace_ctas=self._ctas, e_clip=self.e_clip, critic_coef=self.critic_coef,
                entropy_coef=self.entropy_coef, bounds_loss_coef=self.bounds_coef, **self._schedule_fields(k, e0 // self.mb_envs))
                for e0 in range(0, n, self.mb_envs)] for k in range(self.mini_epochs)]   # one per (mini-epoch, slot): the schedule
                                                                                       # needs to know which launch opens what
        p = lambda x: C.c_void_p(x.data_ptr())  # noqa: E731
        pm = self._p2p_mlp.ptr if self._p2p_mlp is not None else None
        for k in range(self.mini_epochs):
            for slot, mb in enumerate(self._mb_structs[k]):
                # forward + losses + backward; writes this pass's mu over the rows' mu_old (rl_games dataset.update_mu_sigma)
                n_part = lib.vine_ppo_minibatch(C.byref(mb), stream)
                assert n_part > 0, n_part
                assert lib.vine_ppo_reduce(p(self._ws), n_part, self.O, p(self._flat_grads), p(self.model.sigma),
                                           p(self._logstd_old[slot]), pm, stream) == 0
                if self.grad_allreduce == "nccl":   # baseline: ONE NCCL all-reduce per minibatch (gradients + loss statistics)
                    torch.distributed.all_reduce(self._flat_grads)
                if self.truncate_grads:   # the norm of the mean gradient, then Adam with the coefficient (state slot 9)
                    P = self.flat.numel()  # p2p: the clip kernel consumes the channel and leaves the rank sum in _flat_grads
                    assert lib.vine_grad_clip(p(self._flat_grads), P, P + 4, None, 0, 0, 1.0 / self.world, self.grad_norm,
                                              p(self.ppo_state), p(self._clip_ws), pm, None, stream) == 0
                    coef = C.c_void_p(self.ppo_state.data_ptr() + abi.PPO_STATE_CLIP_COEF * 4)
                    assert lib.vine_ppo_adam_clipped(p(self._flat_grads), 1.0 / self.world, p(self.flat), p(self.adam_m),
                                                     p(self.adam_v), p(self._packed), p(self.ppo_state), self.O, 0.9, 0.999, 1e-8,
                                                     1, coef, None, stream) == 0
                    continue
                # p2p: the Adam kernel waits for every rank's buffer and adds them in rank order itself (vine_p2p.cuh)
                assert lib.vine_ppo_adam(p(self._flat_grads), 1.0 / self.world, p(self.flat), p(self.adam_m), p(self.adam_v),
                                         p(self._packed), p(self.ppo_state), self.O, 0.9, 0.999, 1e-8, 1, pm, stream) == 0

    def capture_graphs(self, warmup=3):
        """Warm up eagerly on a side stream, then capture the rollout and the update as two graphs."""
        s = torch.cuda.Stream(self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(warmup):
                self._rollout()
                self._update_any()
                self.frames += self.T * self.n * self.world   # real training iterations: counted like any other
                self.epoch += 1
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        self._g_rollout, self._g_update = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._g_rollout):
            self._rollout()
        with torch.cuda.graph(self._g_update):
            self._update_any()
        torch.cuda.synchronize(self.device)

    def train_epoch(self):
        if self.use_graphs and self._g_rollout is None:
            self.capture_graphs()
        self.play_steps()
        if self._g_update is not None:
            self._g_update.replay()
        else:
            self._update_any()
        self.epoch += 1

    def _update_any(self):
        if self.native_lstm:
            self._update_native_lstm()
        elif self.fused_update:
            self._update_fused()
        else:
            self._update()

    def pop_stats(self):
        e = self.ep_stats.tolist()
        if self.fused_update:   # the Adam kernel keeps the running sums: a_loss, c_loss, kl, b_loss, count
            st = self.ppo_state.tolist()
            l = [st[4], st[5], st[6], st[8]]
            self.ppo_state[4:9] = 0.0
        else:
            l = self.loss_stats.tolist()
            self.loss_stats.zero_()
        self.ep_stats.zero_()
        eps, nmb = max(e[0], 1.0), max(l[3], 1.0)
        return {"episodes": int(e[0]), "success_rate": e[1] / eps, "mean_return": e[2] / eps, "mean_length": e[3] / eps,
                "a_loss": l[0] / nmb, "c_loss": l[1] / nmb, "kl": l[2] / nmb}

    def train(self, max_epochs, log_every=25, log=print, on_epoch=None):
        hist = []
        torch.cuda.synchronize(self.device)
        t0, f0 = time.perf_counter(), self.frames
        last = self.epoch + max_epochs      # the CUDA-graph warm-up iterations of the first call count against max_epochs
        while self.epoch < last:
            before = self.epoch
            self.train_epoch()
            if on_epoch is not None:
                on_epoch(self)
            if any(e % log_every == 0 for e in range(before + 1, self.epoch + 1)) or self.epoch >= last:
                torch.cuda.synchronize(self.device)
                st = self.pop_stats()
                st.update({"epoch": self.epoch, "frames": self.frames, "lr": self.lr,
                           "fps_total": (self.frames - f0) / (time.perf_counter() - t0)})
                hist.append(st)
                if log:
                    line = " ".join(f"{k}={v:.4g}" if isinstance(v, float) else f"{k}={v}" for k, v in st.items())
                    try:
                        log(line, st)          # loggers that also want the numbers (train.py: scalar writer + observer)
                    except TypeError:
                        log(line)
        return hist

    # ------------------------------------------------------------------ checkpoints
    # Layout of rl-games 1.5.2 ``A2CBase.get_full_state_weights`` -- what the reference's train.py saves under
    # runs/<name>/nn/*.pth and what isaacgymenvs/vine_robot_test_model.py:135-139 reads back: ``model`` holds the
    # network under ``a2c_network.*`` plus the input/value normalisers as ``running_mean_std.*`` / ``value_mean_std.*``
    # (each only when it is on, like rl_games' Network).
    def rlgames_model_state(self):
        return rlgames_model_state(self.model, self.obs_rms if self.normalize_input else None,
                                   self.val_rms if self.normalize_value else None)

    def _optimizer_state(self):
        if self.fused_update:
            sd = {"exp_avg": self.adam_m.clone(), "exp_avg_sq": self.adam_v.clone(), "step": float(self.ppo_state[1])}
            if self.native_lstm:
                sd.update({"exp_avg_lstm": self.adam_ml.clone(), "exp_avg_sq_lstm": self.adam_vl.clone()})
            return {"fused_adam": sd}
        return self.opt.state_dict()

    def state_dict(self):
        sd = {"model": self.rlgames_model_state(), "optimizer": self._optimizer_state(), "epoch": self.epoch,
              "frame": self.frames, "last_lr": self.lr, "last_mean_rewards": 0.0, "env_state": None}
        if self.fused_update:   # Philox stream position of the action noise: a resumed run must not replay it
            sd["vine_rng_counter"] = int(self._rng_counter.item())
        return sd

    def load_state_dict(self, sd):
        model = sd["model"]
        net = {k[len("a2c_network."):]: v for k, v in model.items() if k.startswith("a2c_network.")}
        with torch.no_grad():   # copy in place: with the fused update the parameters are views of one flat vector
            own = self.model.state_dict()
            assert set(own) == set(net), (sorted(set(own) ^ set(net)))
            for k, v in own.items():
                v.copy_(net[k])
        for name, rms, on, key in zip(NORMALISER_KEYS, (self.obs_rms, self.val_rms), (self.normalize_input, self.normalize_value),
                                      ("normalize_input", "normalize_value")):
            sub = {k[len(name) + 1:]: v for k, v in model.items() if k.startswith(name + ".")}
            if not sub and name in sd:          # older layout: normalisers stored beside 'model'
                sub = sd[name]
            if bool(sub) != on:   # rl_games' strict load: a surplus or missing normaliser is an error, not a silent default
                raise ValueError(f"checkpoint {'has' if sub else 'lacks'} {name}.* but {key} is {on}: it was written by a run "
                                 f"with {key} {not on}")
            if sub:   # value_mean_std is [1] in rl_games files; older files of this trainer stored it 0-dim
                own = rms.state_dict()
                rms.load_state_dict({k: v.to(own[k].dtype).reshape(own[k].shape) for k, v in sub.items()})
        opt = sd.get("optimizer")
        if opt and self.fused_update and "fused_adam" in opt:
            self.adam_m.copy_(opt["fused_adam"]["exp_avg"])
            self.adam_v.copy_(opt["fused_adam"]["exp_avg_sq"])
            self.ppo_state[1] = float(opt["fused_adam"]["step"])
            if self.native_lstm and "exp_avg_lstm" in opt["fused_adam"]:
                self.adam_ml.copy_(opt["fused_adam"]["exp_avg_lstm"])
                self.adam_vl.copy_(opt["fused_adam"]["exp_avg_sq_lstm"])
        elif opt and not self.fused_update and "fused_adam" not in opt:
            self.opt.load_state_dict(opt)
        if self.fused_update and "vine_rng_counter" in sd:
            self._rng_counter.fill_(int(sd["vine_rng_counter"]))
        self.epoch, self.frames = sd.get("epoch", 0), sd.get("frame", 0)
        self.lr_t.fill_(float(sd.get("last_lr", self.lr)))
        # the iteration counter of the linear schedule: a resumed run continues its learning-rate sequence
        if self.fused_update:
            self.ppo_state[abi.PPO_STATE_EPOCH] = float(self.epoch)
        else:
            self._epoch_t.fill_(float(self.epoch))
        if self.fused or self.native_lstm:
            self._refresh_fused(pack=True)
