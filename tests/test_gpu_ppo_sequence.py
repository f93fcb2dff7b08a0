"""GPU: the kernel-only PPO iteration launch by launch -- PPOAgent._rollout_fused (the MLP network's rollout) and the update
sequences _update_fused / _update_native_lstm -- against float64 chains built from the rollout buffers.

The per-kernel float64 references live with the kernels' own tests (test_gpu_mlp_update.py, test_gpu_lstm_update.py,
test_gpu_lstm_block_options.py, test_gpu_lstm_rollout.py).  What they cannot see is the wiring of an iteration: which
buffer a launch reads, which state it shares with the launches around it.  SequenceRecorder (test_gpu_lstm_rollout's
RecordingLib, extended) stands in for the agent's library handle and clones, on the launch stream, what each launch of
interest reads and writes; the tests below rebuild every quantity from the rollout buffers in float64 and compare:

  rollout  b_obs[t] = the observation vine_policy_act read; b_done[t] = the resets of step t - 1 (row 0: the previous
           rollout's last row, ones at the very first); env.actions = clamp(b_act[t], +-1); b_rew[t] = the shaped reward
           with the value bootstrap on time-outs, bit for bit; one rng_counter increment per env step; mu / value / neglogp
           and last_value against float64 on the kernel's own h3; b_adv / b_ret = oracle.gae bit for bit; ep_stats against
           a host float64 accumulation.
  update   the running statistics and normalised targets in float64; per minibatch (mini-epoch k, slot) the gradient and
           the loss statistics on the recorded weights, with mu_old / logstd_old from the chain (k = 0: the rollout's mu
           and sigma at update start; else what minibatch (k - 1, slot) wrote and sigma before its Adam step); Adam in
           float64 on the recorded operands, the step count, the learning rate replayed from the rl_games rule, the
           re-packed bf16 weights, and the state block's sums, counters and epoch after the update.

Every bound is stated where it is checked, with its derivation; WORST collects the worst measured value of each (printed)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import vine_robot_isaacgymenvs_b200 as vine
from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200 import config as vcfg
from vine_robot_isaacgymenvs_b200.ppo.ppo import LR_MAX, LR_MIN, ActorCritic, PPOAgent, RunningMeanStd
from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles
from test_gpu_lstm_rollout import RecordingLib, check_u_h3, f32_ulp, set_timeouts
from test_gpu_lstm_update import bf16_ulp, bits
from test_gpu_mlp_update import (KL_LOG_BIAS, TOL_GRAD, TOL_STAT, bf, check_nlp, forward_ref, gradients_ref, loss_ref, u_tile,
                                 value_branches)
from test_gpu_ppo_fused import NAMES

pytestmark = pytest.mark.gpu
DEV = "cuda"
U = 2.0 ** -24                                             # f32 unit roundoff
B1, B2, EPS = (float(np.float32(x)) for x in (0.9, 0.999, 1e-8))   # the f32 constants the Adam kernels receive
MLP = ["train.params.network.rnn=null"]
WORST = {}


def note(key, x):
    WORST[key] = max(WORST.get(key, 0.0), float(x))


def report(tag):
    print(tag, {k: f"{v:.2e}" for k, v in sorted(WORST.items())})


def make_agent(extra=(), n=4096):
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True"] + list(extra))
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=1, use_graphs=False)


# ------------------------------------------------------------------------------------------------------------ the recorder
class SequenceRecorder(RecordingLib):
    """RecordingLib with the launches of the MLP rollout and of both updates recorded as well, into ``log``: (kind, dict)
    in launch order.  It stands in for agent._lib and, on the recurrent network, for the NativeLstmPath's handle.  Every
    snapshot is a clone on the current stream (the agent's launch stream), so it sees exactly what the neighbouring
    launches read and wrote.  The launches are the agent's own, with one addition: vine_lstm_head_train gets a debug_out
    buffer (the per-row mu, value and neglogp the kernel computes anyway), which test 0 shows changes no result."""

    def __init__(self, agent):
        super().__init__(agent)
        self.log = []
        self._path_lib = agent._path.lib if agent.native_lstm else None

    def __enter__(self):
        self._a._lib = self
        if self._path_lib is not None:
            self._a._path.lib = self
        return self

    def __exit__(self, *exc):
        self._a._lib = self._lib
        if self._path_lib is not None:
            self._a._path.lib = self._path_lib
        torch.cuda.synchronize()

    def _tensor(self, ptr):
        """The agent tensor a launch argument points at."""
        a = self._a
        names = ["flat", "adam_m", "adam_v", "_flat_grads", "_packed", "ppo_state", "flat_l", "adam_ml", "adam_vl", "_lpacked"]
        cands = [getattr(a, k) for k in names if hasattr(a, k)]
        if a.native_lstm:
            cands += [a._path.flat_g_mlp, a._path.flat_g_lstm]
        for t in cands:
            if t.data_ptr() == ptr:
                return t
        raise AssertionError(f"unexpected pointer {ptr:#x}")

    def _row_of(self, buf, ptr, row_bytes):
        off = ptr - buf.data_ptr()
        return off // row_bytes if 0 <= off < buf.numel() * buf.element_size() and off % row_bytes == 0 else None

    def vine_lstm_step(self, ref, stream):
        if ref._obj.act:   # the training form (NativeLstmPath.gradients): not part of the rollout's record
            return self._lib.vine_lstm_step(ref, stream)
        return super().vine_lstm_step(ref, stream)

    # ---- MLP rollout
    def vine_policy_act(self, ref, stream):
        a, s = self._a, ref._obj
        if s.u_out and a.native_lstm and s.u_out == a._path.U.data_ptr():   # the training form
            return self._lib.vine_policy_act(ref, stream)
        if s.u_out:
            return super().vine_policy_act(ref, stream)
        rec = dict(obs=a.env._obs_clamped.clone(), ctr=a._rng_counter.clone())
        rc = self._lib.vine_policy_act(ref, stream)
        t = self._row_of(a.b_mu, s.mu, 8 * a.n)
        if t is None:   # the bootstrap launch: value of the final observation, nothing sampled
            assert s.value == a.last_value.data_ptr() and not s.actions and not s.obs_copy and not s.rng_counter
            rec.update(t=None, mu=a._mu_buf.clone(), value=a.last_value.clone())
        else:
            rec.update(t=t, mu=a.b_mu[t].clone(), value=a.b_val[t].clone(), actions=a.b_act[t].clone(),
                       neglogp=a.b_nlp[t].clone(), env_actions=a.env.actions.clone())
        self.log.append(("act", rec))
        return rc

    def vine_rollout_post(self, ref, stream):
        a = self._a
        if a.native_lstm:
            return super().vine_rollout_post(ref, stream)
        rec = dict(ep_ret=a.ep_ret.clone(), ep_len=a.ep_len.clone(), ep_stats=a.ep_stats.clone(), ctr=a._rng_counter.clone())
        rc = self._lib.vine_rollout_post(ref, stream)
        rec.update(rew=a.env.rew_buf.clone(), resets=a.env.reset_buf.clone(), timeouts=a.env.timeout_buf.clone(),
                   t=self._row_of(a.b_rew, ref._obj.shaped_rewards, 4 * a.n))
        self.log.append(("post", rec))
        return rc

    def vine_gae(self, *args):
        rc = self._lib.vine_gae(*args)
        self.log.append(("gae", dict(ptrs=[x.value for x in args[:5]], T=args[5], n=args[6], gamma=args[7], tau=args[8],
                                     out=[x.value for x in args[9:11]])))
        return rc

    # ---- updates
    def vine_ppo_moments(self, ref, stream):
        a = self._a
        names = ["b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "_done_ext"] + (["_nd_ext", "_HH_saved", "_C_saved"]
                                                                                      if a.native_lstm else [])
        rec = {k: getattr(a, k).clone() for k in names}
        rec.update(state=a.ppo_state.clone(), flat=a.flat.clone(), flat_l=a.flat_l.clone() if a.native_lstm else None)
        self.log.append(("update", rec))
        return self._lib.vine_ppo_moments(ref, stream)

    def vine_ppo_finalize(self, ref, stream):
        rc = self._lib.vine_ppo_finalize(ref, stream)
        a = self._a
        self.log.append(("finalize", dict(mean=a._obs_mean_f.clone(), inv_std=a._obs_inv_std_f.clone(), vstats=a._val_stats.clone(),
                                          val_n=a._val_old_n.clone(), ret_n=a._ret_n.clone(), adv_n=a._adv_n.clone())))
        return rc

    def _logstd_old_read(self, ptr):
        a = self._a
        slot = self._row_of(a._logstd_old, ptr, 8)
        return slot, (a._logstd_old[slot].clone() if slot is not None else None)

    def vine_lstm_gather(self, ref, stream):
        a = self._a
        self.log.append(("gather", dict(e0=ref._obj.env_begin, E=ref._obj.env_count, scal=a._scal.clone())))
        return self._lib.vine_lstm_gather(ref, stream)

    def vine_lstm_head_train(self, ref, stream):
        s = ref._obj
        slot, lso = self._logstd_old_read(s.logstd_old)
        assert not s.debug_out
        dbg = torch.zeros(s.n, 4, device=DEV)
        s.debug_out = dbg.data_ptr()
        try:
            rc = self._lib.vine_lstm_head_train(ref, stream)
        finally:
            s.debug_out = None
        self.log.append(("head_train", dict(slot=slot, logstd_old=lso, writeback=bool(s.mu_writeback), dbg=dbg)))
        return rc

    def vine_ppo_minibatch(self, ref, stream):
        a, s = self._a, ref._obj
        slot, lso = self._logstd_old_read(s.logstd_old)
        rec = dict(e0=s.env_begin, E=s.env_count, slot=slot, logstd_old=lso, state_before=a.ppo_state.clone(),
                   flat=a.flat.clone(), packed=a._packed.clone(), ext=bool(s.dh3_ext))
        if not s.dh3_ext:
            rec.update(mu_old=a.b_mu.clone(), mu_old_is_b_mu=s.mu_old == a.b_mu.data_ptr())
        else:
            rec.update(flat_l=a.flat_l.clone())
        rc = self._lib.vine_ppo_minibatch(ref, stream)
        rec.update(state=a.ppo_state.clone())
        if not s.dh3_ext:
            rec.update(mu_new=a.b_mu.clone())
        self.log.append(("minibatch", rec))
        return rc

    def vine_ppo_reduce(self, ws, n_part, O, flat, logstd, logstd_old, ch, stream):
        rc = self._lib.vine_ppo_reduce(ws, n_part, O, flat, logstd, logstd_old, ch, stream)
        self.log.append(("reduce", dict(g=self._tensor(flat.value).clone(), logstd_old=self._a._logstd_old.clone())))
        return rc

    def vine_lstm_reduce(self, *args):
        rc = self._lib.vine_lstm_reduce(*args)
        self.log.append(("lstm_reduce", dict(g=self._tensor(args[5].value).clone(), scal=self._a._scal.clone())))
        return rc

    def vine_grad_clip(self, *args):
        rc = self._lib.vine_grad_clip(*args)
        self.log.append(("clip", dict(state=self._a.ppo_state.clone())))
        return rc

    def _adam(self, name, args, clipped, lstm):
        g, w, m, v, packed, state = (self._tensor(x.value) for x in (args[0], args[2], args[3], args[4], args[5], args[6]))
        assert state is self._a.ppo_state
        book = 1 if lstm else args[11]
        coef = args[11 + (0 if lstm else 1)] if clipped else None
        rec = dict(g=g.clone(), w=w.clone(), m=m.clone(), v=v.clone(), state=state.clone(), book=book, lstm=lstm,
                   scale=args[1], coef_ptr=coef.value if coef is not None else None)
        rc = getattr(self._lib, name)(*args)
        rec.update(w_new=w.clone(), m_new=m.clone(), v_new=v.clone(), packed_new=packed.clone(), state_new=state.clone())
        self.log.append(("adam", rec))
        return rc

    def vine_ppo_adam(self, *args):
        return self._adam("vine_ppo_adam", args, False, False)

    def vine_ppo_adam_clipped(self, *args):
        return self._adam("vine_ppo_adam_clipped", args, True, False)

    def vine_lstm_adam(self, *args):
        return self._adam("vine_lstm_adam", args, False, True)

    def vine_lstm_adam_clipped(self, *args):
        return self._adam("vine_lstm_adam_clipped", args, True, True)


# ------------------------------------------------------------------------------------- 0. the recorder changes nothing
STATE_BUFFERS = ["flat", "adam_m", "adam_v", "ppo_state", "_logstd_old", "b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_rew",
                 "b_adv", "b_ret", "_done_ext", "last_value", "ep_ret", "ep_len", "_rng_counter", "_val_old_n", "_ret_n",
                 "_adv_n", "_obs_mean_f", "_obs_inv_std_f", "_val_stats"]


@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_recorder_leaves_the_iteration_bit_identical(net):
    """Two agents from identical state, 4096 envs: one training iteration (rollout + update) each, one through
    SequenceRecorder.  Parameters, Adam moments, the state block, every rollout buffer and the normalised targets are
    bit-identical, and the f64 running statistics agree to 1e-12 (vine_ppo_moments sums in f64 with atomics, whose order
    may vary between any two runs), as does ep_stats (same reason)."""
    extra = MLP if net == "mlp" else []
    agents = [make_agent(extra) for _ in range(2)]
    for k, a in enumerate(agents):
        if k == 1:
            with SequenceRecorder(a) as rec:
                a.train_epoch()
            assert any(kind == "adam" for kind, _ in rec.log)
        else:
            a.train_epoch()
    torch.cuda.synchronize()
    x, y = agents
    names = STATE_BUFFERS + (["flat_l", "adam_ml", "adam_vl", "_scal", "_nd_ext", "_HH_saved", "_C_saved"] if net == "lstm" else [])
    for name in names:
        assert torch.equal(getattr(x, name).view(torch.uint8), getattr(y, name).view(torch.uint8)), name
    for rms in ("obs_rms", "val_rms"):
        for b in ("running_mean", "running_var", "count"):
            u, w = getattr(getattr(x, rms), b), getattr(getattr(y, rms), b)
            assert bool(((u - w).abs() <= 1e-12 * w.abs()).all()), (rms, b)
    assert bool(((x.ep_stats - y.ep_stats).abs() <= 1e-12 * y.ep_stats.abs()).all())


# ----------------------------------------------------------------------------------------------- A. the MLP rollout
def mlp_weights(flat, agent):
    """The flat MLP vector (include/vine_b200.h layout) as the list of test_gpu_mlp_update (torch layouts): W1 b1 W2 b2 W3 b3
    Wmu bmu Wv bv logstd."""
    out, o = [], 0
    for shape in ((256, agent.O), (256,), (128, 256), (128,), (64, 128), (64,), (2, 64), (2,), (1, 64), (1,), (2,)):
        k = math.prod(shape)
        out.append(flat[o:o + k].view(shape))
        o += k
    assert o == flat.numel()
    return out


def check_h3_rows(h3_k, fwd, W, obs):
    """check_u_h3 over the distinct observation rows: right after a reset every env observes the same state, and one
    flipped element of that row would count once per env.  The per-element bound holds on every row; the fraction of
    elements off float64 (< 1 %) is asserted once there are 1000 distinct rows or more."""
    _, inv = torch.unique(obs, dim=0, return_inverse=True)
    first = torch.full((int(inv.max()) + 1,), obs.shape[0], dtype=torch.long, device=obs.device)
    first.scatter_reduce_(0, inv, torch.arange(obs.shape[0], device=obs.device), reduce="amin")
    if first.numel() >= 1000:
        sub = {k: (v[first] if v.dim() and v.shape[0] == obs.shape[0] else v) for k, v in fwd.items()}
        check_u_h3(h3_k[first], sub, W)
        return
    bfd = lambda t: t.detach().float().bfloat16().double()  # noqa: E731
    tol = 2 * bf16_ulp(fwd["h3"]) + (2 * bf16_ulp(fwd["h2"]) + (2 * bf16_ulp(fwd["h1"])) @ bfd(W[2]).abs().t()) @ bfd(W[4]).abs().t()
    d = (h3_k - fwd["h3"]).abs()
    assert bool((d <= tol).all()), float((d - tol).max())


def shaped_reward(agent, rew, timeouts, values):
    """vine_rollout_post's shaped reward in f32 with the kernel's operation order: (r [+ shift]) * scale, clamped, then
    `shaped += gamma * value` on time-outs, which nvcc contracts to one FFMA: the product of two f32 numbers is exact in
    float64, so the float64 sum rounded once to f32 is the fused result."""
    r = rew + agent.reward_shift if agent.reward_shift != 0.0 else rew
    r = r * agent.reward_scale
    if agent.reward_clamp:
        r = torch.clamp(r, agent.reward_min, agent.reward_max)
    if agent.value_bootstrap:
        gamma = float(np.float32(agent.gamma))
        boot = (r.double() + gamma * values.double()).float()
        r = torch.where(timeouts != 0, boot, r)
    return r


def check_policy_launch(agent, rec, W, mean, inv_std, vstats, logstd, tag):
    """One vine_policy_act launch against float64 on its own observation: h3 from the u_out mode of the same weights
    (check_u_h3: bf16 flips on the env's observations), then mu and the raw value on that h3 with the head bound of
    test_gpu_mlp_update.check_heads (1e-5 (sum |w h3| + |b|) + 1e-7), value = fma(clamp(v, +-5), std, mean): within std
    times that bound (clamp is 1-Lipschitz) + one ulp of the value; neglogp from the kernel's own mu (check_nlp)."""
    fwd = forward_ref(W, rec["obs"], mean, inv_std)
    _, u = u_tile(agent._lib, agent._packed, rec["obs"], mean, inv_std)
    check_h3_rows(u[:, :64], fwd, W, rec["obs"])
    h3 = u[:, :64]
    ref = h3 @ fwd["wh"].t() + fwd["bh"]
    tol = 1e-5 * (h3.abs() @ fwd["wh"].abs().t() + fwd["bh"].abs()) + 1e-7
    em = (rec["mu"].double() - ref[:, :2]).abs()
    assert bool((em <= tol[:, :2]).all()), (tag, "mu", float((em - tol[:, :2]).max()))
    note("rollout mu / bound", (em / tol[:, :2]).max())
    vm, vs = float(vstats[0]), float(vstats[1])
    want = ref[:, 2].clamp(-5.0, 5.0) * vs + vm
    ev = (rec["value"].double() - want).abs()
    bv = vs * tol[:, 2] + f32_ulp(rec["value"].double())
    assert bool((ev <= bv).all()), (tag, "value", float((ev - bv).max()))
    note("rollout value / bound", (ev / bv).max())
    if "neglogp" in rec:
        check_nlp(rec["neglogp"], rec["mu"], rec["actions"], logstd)


def check_mlp_rollout(agent, log, done0, ctr0, tag):
    """Every launch of one recorded _rollout_fused; ``done0`` the done row it must start from, ``ctr0`` the rng counter."""
    T, n = agent.T, agent.n
    acts = [d for k, d in log if k == "act"]
    posts = [d for k, d in log if k == "post"]
    gaes = [d for k, d in log if k == "gae"]
    assert len(acts) == T + 1 and len(posts) == T and len(gaes) == 1, (tag, len(acts), len(posts))
    W = mlp_weights(agent.flat.clone(), agent)
    mean, inv_std, vstats = agent._obs_mean_f.clone(), agent._obs_inv_std_f.clone(), agent._val_stats.clone()
    logstd = agent.model.sigma.detach().clone()
    assert torch.equal(agent._done_ext[0], done0), tag
    host = posts[0]["ep_stats"].double().cpu().clone()
    thr = agent.success_threshold
    for t in range(T):
        a, p = acts[t], posts[t]
        assert a["t"] == t and p["t"] == t, (tag, t)
        assert int(a["ctr"]) == ctr0 + t, (tag, t, int(a["ctr"]))
        assert torch.equal(bits(agent.b_obs[t]), bits(a["obs"])), (tag, t, "b_obs")
        for k, buf in (("mu", agent.b_mu), ("value", agent.b_val), ("actions", agent.b_act), ("neglogp", agent.b_nlp)):
            assert torch.equal(bits(buf[t]), bits(a[k])), (tag, t, k)
        assert torch.equal(bits(a["env_actions"]), bits(a["actions"].clamp(-1.0, 1.0))), (tag, t, "env_actions")
        check_policy_launch(agent, a, W, mean, inv_std, vstats, logstd, f"{tag} t={t}")
        d = (p["resets"] != 0).float()
        assert torch.equal(agent._done_ext[t + 1], d), (tag, t, "done")
        want = shaped_reward(agent, p["rew"], p["timeouts"], agent.b_val[t])
        assert torch.equal(bits(agent.b_rew[t]), bits(want)), (tag, t, "b_rew")
        # episode statistics: f32 running return / length, f64 sums of the finished episodes
        er, el = p["ep_ret"] + p["rew"], p["ep_len"] + 1.0
        fin = d != 0
        host += torch.tensor([float(fin.sum()), float((fin & (p["rew"] > thr)).sum()), float(er[fin].double().sum()),
                              float(el[fin].double().sum())], dtype=torch.float64)
        nxt = posts[t + 1] if t + 1 < T else None
        if nxt is not None:
            assert torch.equal(bits(nxt["ep_ret"]), bits(torch.where(fin, 0.0, er))), (tag, t, "ep_ret")
            assert torch.equal(bits(nxt["ep_len"]), bits(torch.where(fin, 0.0, el))), (tag, t, "ep_len")
    assert int(agent._rng_counter) == ctr0 + T
    last = acts[T]
    assert last["t"] is None and torch.equal(bits(agent.last_value), bits(last["value"]))
    check_policy_launch(agent, last, W, mean, inv_std, vstats, logstd, f"{tag} last")
    assert torch.equal(bits(last["obs"]), bits(agent.env._obs_clamped)), tag   # the final observation
    # GAE on the rollout's buffers, bit for bit against the f32 oracle
    g = gaes[0]
    assert g["ptrs"] == [agent.b_rew.data_ptr(), agent.b_val.data_ptr(), agent.b_done.data_ptr(), agent.last_value.data_ptr(),
                         agent._done_ext[T].data_ptr()], tag
    assert (g["T"], g["n"], g["gamma"], g["tau"]) == (T, n, agent.gamma, agent.tau)
    from oracle import oracle
    cpu = lambda x: x.cpu().numpy()  # noqa: E731
    adv, ret = oracle.gae(cpu(agent.b_rew), cpu(agent.b_val), cpu(agent.b_done), cpu(agent.last_value), cpu(agent._done_ext[T]),
                          agent.gamma, agent.tau)
    assert np.array_equal(cpu(agent.b_adv).view(np.int32), adv.view(np.int32)), tag
    assert np.array_equal(cpu(agent.b_ret).view(np.int32), ret.view(np.int32)), tag
    # ep_stats: counts and lengths are integers (exact); the return sum is an f64 sum in another order: 1e-12 relative
    got = agent.ep_stats.cpu()
    for j in (0, 1, 3):
        assert float(got[j]) == float(host[j]), (tag, j, float(got[j]), float(host[j]))
    assert abs(float(got[2]) - float(host[2])) <= 1e-12 * abs(float(host[2])) + 1e-9, (tag, float(got[2]), float(host[2]))
    return float(d.mean())


ROLLOUT_CASES = {"4096": (4096, []),
                 "ragged_1000": (1000, ["train.params.config.minibatch_size=4000"]),
                 "4096_shift_clamp": (4096, ["train.params.config.reward_shaper.shift_value=-2.0",
                                             "train.params.config.reward_shaper.min_val=-0.2",
                                             "train.params.config.reward_shaper.max_val=0.5"])}


@pytest.mark.parametrize("case", list(ROLLOUT_CASES))
def test_mlp_rollout_launch_by_launch(case):
    """PPOAgent._rollout_fused on FSTR (rnn=null), the agent's first two rollouts, with non-trivial observation / value
    statistics and log-std and ~1/T of the envs timing out at every step of the second (set_timeouts): at 4096 envs
    (programmatic dependent launch), at 1000 (a ragged last block) and with the reward shaper's shift and clamp on.
    Checked per step on the operands the launches read (SequenceRecorder): b_obs[t] = the observation vine_policy_act
    read, bit for bit; b_mu / b_val / b_act / b_nlp[t] = what it wrote, and against float64 (check_policy_launch);
    env.actions = clamp(b_act[t], +-1); b_done[t] = the resets of step t - 1, row 0 = the previous rollout's last row
    (ones for the first); b_rew[t] = shaped_reward, bit for bit; rng_counter = its start + t at step t; ep_ret / ep_len
    carried or zeroed; last_value = the value of the final observation; b_adv / b_ret = oracle.gae bit for bit; ep_stats
    against a host float64 accumulation."""
    n, extra = ROLLOUT_CASES[case]
    agent = make_agent(MLP + list(extra), n=n)
    assert agent.fused_update and not agent.has_rnn and agent.value_bootstrap
    if "shift" in case:
        assert agent.reward_shift == -2.0 and agent.reward_clamp
    g = torch.Generator(device=DEV).manual_seed(n)
    with torch.no_grad():
        agent.model.sigma.copy_(torch.tensor([-0.4, 0.1], device=DEV))
        agent.model.value.weight.mul_(8.0)
        agent.obs_rms.running_mean.copy_(0.2 * torch.randn(agent.O, device=DEV, generator=g).double())
        agent.obs_rms.running_var.copy_((0.3 + torch.rand(agent.O, device=DEV, generator=g)).double())
        agent.val_rms.running_mean.fill_(0.4)
        agent.val_rms.running_var.fill_(2.5)
    agent._refresh_fused(pack=True)
    done0 = torch.ones(n, device=DEV)
    for it in range(2):
        set_timeouts(agent)
        ctr0 = int(agent._rng_counter)
        with SequenceRecorder(agent) as rec:
            agent._rollout()
        frac = check_mlp_rollout(agent, rec.log, done0, ctr0, f"{case} it={it}")
        done0 = agent._done_ext[agent.T].clone()
        if it == 1:
            assert float(agent._done_ext[0].mean()) < 1.0 and float(agent._done_ext[1:].mean()) > 0.5 / agent.T
            assert float(agent.b_rew.isfinite().double().mean()) == 1.0
        print(f"{case} rollout {it}: resets at the last step {frac:.3f}")
    if "shift" in case:   # both bounds of the clamp are hit (measured: 0.3 % and 1.8 % of the second rollout's rows)
        hi, lo = float((agent.b_rew == 0.5).double().mean()), float((agent.b_rew == -0.2).double().mean())
        print(f"{case}: clamped rewards {hi:.3f} at max_val, {lo:.3f} at min_val")
        assert hi > 0.0 and lo > 0.0
    report(case)


# ------------------------------------------------------------------------------------------------------ B/C. the updates
def group_minibatches(log):
    """The update events of a recorded log, one dict per update: start / finalize, and per minibatch (in launch order)
    its minibatch launch, reduce(s), clip and Adam launch(es)."""
    ups = []
    for kind, d in log:
        if kind == "update":
            ups.append(dict(start=d, mbs=[]))
        elif kind == "finalize":
            ups[-1]["finalize"] = d
        elif kind in ("gather", "minibatch") and (kind == "gather" or not d["ext"]):
            ups[-1]["mbs"].append({kind: d, "adam": []})
        elif ups and ups[-1]["mbs"]:
            mb = ups[-1]["mbs"][-1]
            if kind == "adam":
                mb["adam"].append(d)
            elif kind in mb:
                raise AssertionError(f"two {kind} launches in one minibatch")
            else:
                mb[kind] = d
    return ups


def prologue_reference(agent, start, fin, ref_obs, ref_val, tag):
    """float64 running statistics (RunningMeanStd fed float64 data) and normalised targets from the rollout buffers; the
    f32 statistics the minibatch kernel reads are checked against them (mean: the f32 rounding of the float64 mean
    exactly; rsqrtf of the rounded variance within 2e-6, as test_update_prologue_matches_float64_at_the_training_size).
    values_n / returns_n = clamp((x - mean) / std, +-5): the kernel rounds the mean to f32 and x - mean, / std once each:
    within 6e-8 (|x| + |mean|) / std + 1e-6 (1 + |x_n|); the advantage (returns - values in f32, normalised with the f64
    batch moments): within 1.2e-7 (|ret| + |val|) / std_a + 1e-6 (1 + |a_n|).  -> the float64 targets."""
    T, n = agent.T, agent.n
    if agent.normalize_input:
        ref_obs.update(start["b_obs"].reshape(T * n, agent.O).double())
        assert torch.equal(fin["mean"], ref_obs.running_mean.float()), tag
        assert torch.allclose(fin["inv_std"].double(), torch.rsqrt(ref_obs.running_var.float().double() + 1e-5), rtol=2e-6, atol=0)
    val, ret = start["b_val"].double(), start["b_ret"].double()
    if agent.normalize_value:
        ref_val.update(torch.cat([val.reshape(-1), ret.reshape(-1)]))
        vm, vs = float(ref_val.running_mean), math.sqrt(float(ref_val.running_var) + 1e-5)
        vo_n, ret_n = (((x - vm) / vs).clamp(-5.0, 5.0) for x in (val, ret))
        for x, got in ((val, fin["val_n"]), (ret, fin["ret_n"])):
            want = ((x - vm) / vs).clamp(-5.0, 5.0)
            tol = 6e-8 * (x.abs() + abs(vm)) / vs + 1e-6 * (1 + want.abs())
            assert bool(((got.double() - want).abs() <= tol).all()), (tag, float(((got.double() - want).abs() - tol).max()))
    else:
        vo_n, ret_n = val, ret
    adv = ret - val
    if agent.normalize_advantage:
        std = float(adv.std())
        adv_n = (adv - adv.mean()) / (std + 1e-8)
        tol = 1.2e-7 * (ret.abs() + val.abs()) / std + 1e-6 * (1 + adv_n.abs())
        assert bool(((fin["adv_n"].double() - adv_n).abs() <= tol).all()), tag
    else:
        adv_n = adv
    return vo_n, ret_n, adv_n


def kl_rows(mu, mu_old, ls, lso):
    """The rows of the KL statistic (ppo.policy_kl, as the kernels evaluate it: sigma_old^2 + 1e-5 in the denominator)."""
    sig, so = torch.exp(ls.double()), torch.exp(lso.double())
    return (torch.log(so / sig + 1e-5) + (sig ** 2 + (mu.double() - mu_old.double()) ** 2) / (2 * (so ** 2 + 1e-5)) - 0.5).sum(-1)


def check_adam(rec, lr, t, coef, P, tag):
    """One Adam launch against float64 Adam (torch.optim.Adam: m = b1 m + (1 - b1) g, v = b2 v + (1 - b2) g^2,
    w -= lr / (1 - b1^t) m / (sqrt(v) / sqrt(1 - b2^t) + eps)) on the recorded operands, with the f32 constants.
    Bounds from the kernel's f32 roundings: g = flat * coef rounds once (clipped: dg = u |g|); m within 2u (|b1 m0| +
    |(1 - b1) g|) + (1 - b1) dg; v within 3u (|b2 v0| + (1 - b2) g^2) + (1 - b2) 2 |g| dg; the step within
    |step| u (10 + 4 / bc1 + 2 / bc2) (seven roundings, powf within 4 ulp of b^t < 1, whose error 1 - b^t magnifies, halved
    by the square root for bc2) + lr / bc1 dm / den + |step| dv / (2 v); the parameter within that + one ulp."""
    g = rec["g"][:P].double() * coef
    m0, v0, w0 = rec["m"][:P].double(), rec["v"][:P].double(), rec["w"][:P].double()
    m = B1 * m0 + (1 - B1) * g
    v = B2 * v0 + (1 - B2) * g * g
    bc1, bc2 = 1 - B1 ** t, 1 - B2 ** t
    den = v.sqrt() / math.sqrt(bc2) + EPS
    step = lr / bc1 * m / den
    w = w0 - step
    dg = U * g.abs() if coef != 1.0 else torch.zeros_like(g)
    dm = 2 * U * ((B1 * m0).abs() + ((1 - B1) * g).abs()) + (1 - B1) * dg
    dv = 3 * U * (B2 * v0 + (1 - B2) * g * g) + (1 - B2) * 2 * g.abs() * dg
    ds = step.abs() * U * (10 + 4 / bc1 + 2 / bc2) + lr / bc1 * dm / den + torch.where(v > 0, step.abs() * dv / (2 * v), 0.0)
    for name, got, want, tol in (("m", rec["m_new"], m, dm), ("v", rec["v_new"], v, dv),
                                 ("w", rec["w_new"], w, ds + f32_ulp(w))):
        err = (got[:P].double() - want).abs()
        assert bool((err <= tol).all()), (tag, name, float((err - tol).max()), int((err > tol).sum()))
        note(f"adam {name} / bound", (err / tol.clamp_min(1e-45)).max())


class LrReplay:
    """The rl_games learning-rate rule replayed in float64 from the float64 KL of every minibatch (adaptive: / 1.5 above
    2 kl_threshold, x 1.5 below kl_threshold / 2, clamped to [LR_MIN, LR_MAX]; linear: LR_MIN + (lr0 - LR_MIN) max(0,
    max_epochs - epoch) / max_epochs; legacy: after every minibatch, standard: once per mini-epoch on its mean KL), the
    way vine_ppo_minibatch schedules it: the pending KL of the previous minibatch is applied by the next minibatch launch
    (across iterations too), the epoch counted after.  A decision whose KL lies within ``kl_tol`` of a threshold is taken
    from the kernel (which must then have made one of the two choices) and counted in ``skipped``."""

    def __init__(self, agent):
        self.a = agent
        self.lr = float(np.float32(agent.lr0))
        self.lr_min, self.lr_max = float(np.float32(LR_MIN)), float(np.float32(LR_MAX))
        self.pending, self.ekl, self.epoch, self.decisions, self.skipped = None, [], 0, 0, 0
        self.roundings = 0   # f32 roundings the kernel's lr has been through since it last equalled self.lr exactly

    def _rule(self, kl, kl_tol, kernel_lr):
        a = self.a
        if a.adaptive:
            thr = a.kl_threshold
            up = min(self.lr * 1.5, self.lr_max)
            down = max(self.lr / 1.5, self.lr_min)
            self.decisions += 1
            if abs(kl - 2 * thr) <= kl_tol or abs(kl - 0.5 * thr) <= kl_tol:
                self.skipped += 1
                cands = [self.lr, up, down]
                best = min(cands, key=lambda c: abs(c - kernel_lr))
                assert abs(best - kernel_lr) <= 8 * U * best, (kernel_lr, cands)
                self.lr, self.roundings = kernel_lr, 0
                return
            new = down if kl > 2 * thr else (up if kl < 0.5 * thr else self.lr)
            self.roundings += int(new != self.lr)
            self.lr = new
        elif a.linear_lr:   # in f64 from the f32 constants, one rounding to f32
            self.lr = self.lr_min + (float(np.float32(a.lr0)) - self.lr_min) * max(0.0, a.max_epochs - self.epoch) / a.max_epochs
            self.roundings = 1

    def launch(self, k, slot, kernel_lr):
        """The schedule part of minibatch (k, slot); ``kernel_lr`` the lr the kernel left (used only for a skipped one)."""
        a = self.a
        if self.pending is not None:
            if a.schedule_standard:
                self.ekl.append(self.pending)
            else:
                self._rule(*self.pending, kernel_lr)
            self.pending = None
        if a.schedule_standard and slot == 0 and self.ekl:
            kl = sum(x for x, _ in self.ekl) / len(self.ekl)
            self._rule(kl, max(t for _, t in self.ekl), kernel_lr)
            self.ekl = []
        if k == 0 and slot == 0:
            self.epoch += 1

    def check(self, kernel_lr, tag):
        """The kernel's f32 lr: within one rounding (u) per run of the rule that changed it since the last exact value."""
        tol = U * self.roundings * self.lr
        assert abs(kernel_lr - self.lr) <= tol, (tag, kernel_lr, self.lr)
        note("lr rel err", abs(kernel_lr - self.lr) / self.lr)


def check_state_after(st, up, st0, stats, steps_before, tag):
    """The state block ``st`` after an update: the step count (minibatches since the agent was built), the minibatch count,
    the epoch, the loss sums = st0's plus the per-minibatch statistics in launch order (f32 adds: bit for bit)."""
    M = len(up["mbs"])
    assert float(st[1]) == steps_before + M, (tag, float(st[1]))
    assert float(st[8]) == float(st0[8]) + M, tag
    assert float(st[abi.PPO_STATE_EPOCH]) == float(st0[abi.PPO_STATE_EPOCH]) + 1, tag
    sums = st0[4:8].cpu().numpy().astype(np.float32).copy()
    for s4 in stats:
        sums = (sums + s4.astype(np.float32)).astype(np.float32)
    assert np.array_equal(st[4:8].cpu().numpy().view(np.int32), sums.view(np.int32)), (tag, st[4:8].tolist(), sums)


def run_recorded(agent, iters):
    logs = []
    for _ in range(iters):
        set_timeouts(agent)
        with SequenceRecorder(agent) as rec:
            agent.train_epoch()
        logs.append(rec.log)
    return logs


def mu_write_back_bound(fwd, W):
    """|mu_kernel - mu_float64| per element: the head bound of check_heads on the kernel's h3, plus bf16 flips of h1 / h2 /
    h3 carried through the layers (the bound of check_u_h3) and the heads: 1e-5 (|h3| |wh| + |bh|) + (tol_h3 |wh|)."""
    bfd = lambda t: bf(t.detach().double())  # noqa: E731
    w2, w3 = bfd(W[2]).abs(), bfd(W[4]).abs()
    tol_h3 = 2 * bf16_ulp(fwd["h3"]) + (2 * bf16_ulp(fwd["h2"]) + (2 * bf16_ulp(fwd["h1"])) @ w2.t()) @ w3.t()
    wh = fwd["wh"][:2].abs()
    base = 1e-5 * ((fwd["h3"].abs() + tol_h3) @ wh.t() + fwd["bh"][:2].abs()) + 1e-7
    return base, base + tol_h3 @ wh.t()


def near_boundary_allowance(fwd, W, loss, scal, mu_k, v_tol, logstd, hyp, clip_value, inv_B):
    """What the rows near a branch boundary of the loss may move each gradient tensor by.  On the rollout's own data (no
    planted margins) some rows lie so close to a boundary that the kernel may take the other branch than float64: the
    ratio clip, decided on the kernel's mu, which the write-back gives exactly (a row counts when the side of float64 and
    of the kernel's mu differ, or the latter lies within 1e-5 of the boundary: f32 nlp noise); the value clip
    (| |v - v_old| - e_clip | <= v_tol) and the choice between the two value losses (|c1 - c2| <= 2 v_tol (|e1| + |e2|) +
    v_tol^2), with v_tol the value's bound (test body).  Each such row's head gradient then changes by delta (the actor term
    adv ratio switched on / off; the value term of the other branch); propagated through the backward chain row by row,
    it moves a weight tensor by at most sum_rows |dz_row| |input_row| and a bias by |sum_rows |dz_row||.  -> NAMES order."""
    s = scal.double()
    act, vo, ret, adv = s[:, :2], s[:, 5], s[:, 6], s[:, 7]
    e = hyp["e_clip"]
    sig = torch.exp(logstd.double())
    d = (act - fwd["mu"]) / sig
    ratio = torch.exp(s[:, 4] - loss["nlp"])
    dk = (act - mu_k.double()) / sig
    lr_ = s[:, 4] - loss["nlp"]
    lr_k = s[:, 4] - (0.5 * (dk * dk).sum(-1) + math.log(2 * math.pi) + logstd.double().sum())
    lo, hi = math.log(1 - e), math.log(1 + e)
    near_r = ((lr_ < lo) != (lr_k < lo)) | ((lr_ > hi) != (lr_k > hi)) | ((lr_k - lo).abs() <= 1e-5) | ((lr_k - hi).abs() <= 1e-5)
    g_alt = torch.where(near_r, adv * ratio, torch.zeros_like(adv))     # |change| of d loss / d nlp on such a row
    v = fwd["v"]
    e1, e2 = v - ret, vo + torch.clamp(v - vo, -e, e) - ret
    near_v = ((v - vo).abs() - e).abs() <= v_tol
    if clip_value:   # inside the clip e1 == e2 and both losses give the same gradient: the choice matters only outside
        near_v |= ((v - vo).abs() > e - v_tol) & ((e1 * e1 - e2 * e2).abs() <= 2 * v_tol * (e1.abs() + e2.abs()) + v_tol ** 2)
    dv = torch.where(near_v, 0.5 * hyp["critic_coef"] * 2 * (e1.abs() + e2.abs()), torch.zeros_like(v))
    dmu = g_alt[:, None] * d.abs() / sig
    dls = g_alt[:, None] * (1 + d * d)
    dzh = torch.cat([dmu, dv[:, None]], 1) * inv_B
    h1, h2, h3, x = fwd["h1"], fwd["h2"], fwd["h3"], fwd["x"][:, :W[0].shape[1]]
    dz3 = (dzh @ fwd["wh"].abs()) * elu_grad_bound(h3)
    dz2 = (dz3 @ bf(W[4].double()).abs()) * elu_grad_bound(h2)
    dz1 = (dz2 @ bf(W[2].double()).abs()) * elu_grad_bound(h1)
    nrm = lambda t: t.norm(dim=-1)  # noqa: E731
    wsum = lambda dz, inp: float((nrm(dz) * nrm(inp)).sum())  # noqa: E731
    bsum = lambda dz: float(dz.sum(0).norm())  # noqa: E731
    return [wsum(dz1, x), bsum(dz1), wsum(dz2, h1), bsum(dz2), wsum(dz3, h2), bsum(dz3), wsum(dzh[:, :2], h3),
            bsum(dzh[:, :2]), wsum(dzh[:, 2:], h3), bsum(dzh[:, 2:]), float((dls.sum(0) * inv_B).norm())], \
        dict(ratio=float(near_r.double().mean()), value=float(near_v.double().mean()))


def elu_grad_bound(h):
    return torch.where(h > 0, torch.ones_like(h), (h + 1).abs())


UPDATE_CASES = {"default": (4096, []),
                "truncate_standard": (4096, ["train.params.config.truncate_grads=True", "train.params.config.grad_norm=0.02",
                                              "train.params.config.schedule_type=standard"]),
                "linear": (4096, ["train.params.config.lr_schedule=linear", "train.params.config.max_epochs=10"]),
                "ragged_1000": (1000, ["train.params.config.minibatch_size=4000"])}


@pytest.mark.parametrize("case", list(UPDATE_CASES))
def test_mlp_update_sequence_against_float64(case):
    """_update_fused for two iterations (so that the normalisers, sigma and Adam's step count are non-trivial) at 4096 envs
    x 16 steps with minibatch 32768 (2 slots x 4 mini-epochs), with truncate_grads + schedule_type standard, with the
    linear schedule, and at 1000 envs (4 slots of 250 envs).  The float64 chain (module docstring) on the recorded
    operands, per minibatch (k, slot):
      mu_old read = the rollout's mu (k = 0) / the write-back of (k - 1, slot), bit for bit; the write-back against
        float64 (mu_write_back_bound, and fewer than 2 % of rows beyond its flip-free part);
      logstd_old read = sigma at update start (k = 0) / sigma before (k - 1, slot)'s Adam step, bit for bit;
      the 11 gradient tensors against gradients_ref on float64 targets: TOL_GRAD (2e-3 relative Frobenius, the bound
        of test_gpu_mlp_update.py) + near_boundary_allowance (the rollout's own rows carry no planted margin from the loss's
        branch boundaries: at most 2.5e-4 of the rows lie near the ratio clip and 1.6e-2 near the value clip, measured);
        a_loss, kl and b_loss against float64 rows on the kernel's own mu (the write-back): TOL_STAT of the mean |row| (kl +
        KL_LOG_BIAS); c_loss against float64 v: its rows move by 2 |v - r| dv + dv^2 with dv the value's bound;
      clip (truncate_grads): state[10] = the f64 norm of the recorded gradient within 1e-5 relative (an f32 sum of
        ~50k squares), the coefficient min(1, grad_norm / (norm + 1e-6)) likewise;
      Adam: check_adam, the step count = minibatches since the agent was built, lr = LrReplay within 2u per rule run,
        the re-packed weights = vine_mlp_pack(new parameters) bit for bit.
    After each update: check_state_after; b_mu = the last mini-epoch's write-back and _logstd_old[slot] = sigma before
    the last Adam step of the slot, bit for bit."""
    n, extra = UPDATE_CASES[case]
    agent = make_agent(MLP + list(extra), n=n)
    assert agent.fused_update and not agent.has_rnn
    lib, T, O, E = agent._lib, agent.T, agent.O, agent.mb_envs
    M = agent.n // E
    P = agent.flat.numel()
    hyp = dict(e_clip=agent.e_clip, critic_coef=agent.critic_coef, entropy_coef=agent.entropy_coef,
               bounds_loss_coef=agent.bounds_coef)
    ref_obs, ref_val = RunningMeanStd((O,)).to(DEV), RunningMeanStd(()).to(DEV)
    replay = LrReplay(agent)
    steps = 0
    clipped_seen = 0
    logs = run_recorded(agent, 2)
    for it, log in enumerate(logs):
        ups = group_minibatches(log)
        assert len(ups) == 1
        up = ups[0]
        st0 = up["start"]["state"]
        vo_n, ret_n, adv_n = prologue_reference(agent, up["start"], up["finalize"], ref_obs, ref_val, f"{case} it={it}")
        mean, inv_std = up["finalize"]["mean"], up["finalize"]["inv_std"]
        sigma0 = up["start"]["flat"][P - 2:P].clone()
        assert len(up["mbs"]) == agent.mini_epochs * M
        written, sigma_before_adam, stats = {}, {}, []
        for i, mb in enumerate(up["mbs"]):
            k, slot = divmod(i, M)
            tag = f"{case} it={it} k={k} slot={slot}"
            rec = mb["minibatch"]
            e0 = rec["e0"]
            assert (e0, rec["E"], rec["slot"]) == (slot * E, E, slot), (tag, e0, rec["slot"])
            rows = lambda x: x[:, e0:e0 + E].reshape(T * E, *x.shape[2:])  # noqa: E731
            # the chain's mu_old and logstd_old, bit for bit
            mu_old = rows(up["start"]["b_mu"]) if k == 0 else written[slot]
            assert rec["mu_old_is_b_mu"], tag
            assert torch.equal(bits(rows(rec["mu_old"])), bits(mu_old)), (tag, "mu_old")
            lso = sigma0 if k == 0 else sigma_before_adam[slot]
            assert rec["logstd_old"] is not None and torch.equal(bits(rec["logstd_old"]), bits(lso)), (tag, "logstd_old")
            # the kernel schedule: step and epoch counters
            steps += 1
            assert float(rec["state"][1]) == steps, (tag, float(rec["state"][1]))
            assert float(rec["state"][abi.PPO_STATE_EPOCH]) == it + 1, tag
            # forward on the recorded weights, write-back of mu
            W = mlp_weights(rec["flat"], agent)
            obs = rows(up["start"]["b_obs"])
            fwd = forward_ref(W, obs, mean, inv_std)
            mu_k = rows(rec["mu_new"])
            written[slot] = mu_k.clone()
            base, full = mu_write_back_bound(fwd, W)
            em = (mu_k.double() - fwd["mu"]).abs()
            assert bool((em <= full).all()), (tag, "write-back", float((em - full).max()))
            flips = float((em > base).any(-1).double().mean())
            assert flips < 2e-2, (tag, flips)
            note("mu write-back rows beyond the flip-free bound", flips)
            # gradients and statistics against float64
            scal = torch.cat([rows(up["start"]["b_act"]).double(), mu_old.double(), rows(up["start"]["b_nlp"]).double()[:, None],
                              rows(vo_n)[:, None], rows(ret_n)[:, None], rows(adv_n)[:, None]], 1)
            ls = W[10]
            loss = loss_ref(fwd["mu"], fwd["v"], scal, ls, lso, hyp, agent.clip_value)
            grads = gradients_ref(fwd, W, loss, 1.0 / (T * E))
            # the value's bound: the flip-free head bound, and on the rows whose mu shows a bf16 flip below the heads the
            # flip-inclusive one (a flip moves mu and v together)
            v_base = 1e-5 * (fwd["h3"].abs() @ fwd["wh"][2].abs() + fwd["bh"][2].abs()) + 1e-7
            v_full = v_base + (2 * bf16_ulp(fwd["h3"]) + (2 * bf16_ulp(fwd["h2"]) + (2 * bf16_ulp(fwd["h1"])) @
                               bf(W[2].double()).abs().t()) @ bf(W[4].double()).abs().t()) @ fwd["wh"][2].abs()
            v_tol = torch.where((em > base).any(-1), v_full, v_base)
            allow, near = near_boundary_allowance(fwd, W, loss, scal, mu_k, v_tol, W[10], hyp, agent.clip_value,
                                                  1.0 / (T * E))
            note("rows near a ratio-clip boundary", near["ratio"])
            note("rows near a value-loss boundary", near["value"])
            g = mb["reduce"]["g"]
            got = mlp_weights(g[:P].double(), agent)
            for name, x, y, al in zip(NAMES, got, grads, allow):
                err = float((x - y).norm())
                bound = TOL_GRAD * float(y.norm()) + al
                note(f"grad {name} rel", err / float(y.norm()))
                note(f"grad {name} / bound", err / bound)
                assert err <= bound, (tag, name, err / float(y.norm()), err, bound)
            rows_k = loss_ref(mu_k.double(), fwd["v"], scal, ls, lso, hyp, agent.clip_value)["rows"]
            for j, key in enumerate(("a_loss", "c_loss", "kl", "b_loss")):
                r = rows_k[key]
                scale = float(r.abs().mean()) + 1e-30
                err = abs(float(g[P + j]) - float(r.mean()))
                if key == "c_loss":
                    dv = v_tol
                    e1 = (fwd["v"] - scal[:, 6]).abs() + (fwd["v"] - scal[:, 5]).abs() + 2 * agent.e_clip
                    tol = float((2 * e1 * dv + dv * dv).mean()) + TOL_STAT * scale
                else:
                    tol = TOL_STAT * scale + (KL_LOG_BIAS if key == "kl" else 0.0)
                note(f"stat {key} / bound", err / tol)
                assert err <= tol, (tag, key, err, tol)
            kl64, kl_tol = float(rows_k["kl"].mean()), TOL_STAT * float(rows_k["kl"].abs().mean()) + KL_LOG_BIAS
            stats.append(g[P:P + 4].cpu().numpy())
            assert torch.equal(bits(mb["reduce"]["logstd_old"][slot]), bits(rec["flat"][P - 2:P])), (tag, "sigma copy")
            # learning-rate schedule (the kernel's lr is what Adam reads)
            adam = mb["adam"]
            assert len(adam) == 1 and not adam[0]["lstm"] and adam[0]["book"] == 1, tag
            ad = adam[0]
            kernel_lr = float(ad["state"][0])
            replay.launch(k, slot, kernel_lr)
            replay.check(kernel_lr, tag)
            replay.pending = (kl64, kl_tol)
            # clip and Adam
            coef = 1.0
            if agent.truncate_grads:
                cs = mb["clip"]["state"]
                norm = float(g[:P].double().norm())
                assert abs(float(cs[abi.PPO_STATE_GRAD_NORM]) - norm) <= 1e-5 * norm, (tag, float(cs[10]), norm)
                want = min(1.0, agent.grad_norm / (norm + 1e-6))
                coef = float(cs[abi.PPO_STATE_CLIP_COEF])
                assert abs(coef - want) <= 1e-5 * want, (tag, coef, want)
                assert ad["coef_ptr"] == agent.ppo_state.data_ptr() + 4 * abi.PPO_STATE_CLIP_COEF
                clipped_seen += int(coef < 1.0)
            assert torch.equal(bits(ad["w"]), bits(rec["flat"])), (tag, "Adam reads the minibatch's parameters")
            assert float(ad["state"][1]) == steps
            check_adam(ad, kernel_lr, steps, coef, P, tag)
            sigma_before_adam[slot] = ad["w"][P - 2:P].clone()
            ref_pack = torch.zeros_like(ad["packed_new"])
            Wn = [x.contiguous() for x in mlp_weights(ad["w_new"], agent)[:10]]
            assert lib.vine_mlp_pack(*[C.c_void_p(x.data_ptr()) for x in Wn], O, C.c_void_p(ref_pack.data_ptr()), None) == 0
            torch.cuda.synchronize()
            assert torch.equal(ad["packed_new"], ref_pack), (tag, "re-pack")
            # Adam's bookkeeping: sums, count, KL, pending
            sn, so = ad["state_new"], ad["state"]
            assert float(sn[2]) == float(g[P + 2]) and float(sn[3]) == 1.0 and float(sn[8]) == float(so[8]) + 1
        st_end = group_minibatches(logs[it + 1])[0]["start"]["state"] if it + 1 < len(logs) else agent.ppo_state
        check_state_after(st_end, up, st0, stats, steps - len(up["mbs"]), f"{case} it={it}")
        if it == len(logs) - 1:
            for slot in range(M):
                assert torch.equal(bits(agent.b_mu[:, slot * E:(slot + 1) * E].reshape(T * E, 2)), bits(written[slot])), slot
                assert torch.equal(bits(agent._logstd_old[slot]), bits(sigma_before_adam[slot])), slot
    assert replay.skipped <= max(1, replay.decisions // 10), (replay.skipped, replay.decisions)
    if agent.truncate_grads:   # grad_norm 0.02 lies below the gradient norm of some minibatches: the coefficient < 1 is exercised
        print(f"{case}: {clipped_seen} of {steps} minibatches clipped")
        assert clipped_seen > 0
    print(f"{case}: {replay.decisions} lr decisions, {replay.skipped} within rounding of a threshold")
    report(case)


# ------------------------------------------------------------------------------------------- C. the recurrent update
SUMS = ("b_mu", "b_v", "logstd")   # sums over the rows of terms of both signs (test_gpu_lstm_block_options.SUMS)
LSTM_NAMES = ["W_ih", "W_hh", "b_ih", "b_hh", "ln_g", "ln_b", "W_mu", "b_mu", "W_v", "b_v", "logstd"]
MLP_DUMMY = 197                    # the 64-wide heads and log-std of the MLP layout, unused by the recurrent network


def lstm_rows(x, L, e0, E):
    """[T, n, ...] -> [L, chunks * E, ...]: the minibatch's rows [step in chunk][chunk, env] (ppo.PPOAgent._update's mb)."""
    ch = x.shape[0] // L
    return x[:, e0:e0 + E].reshape(ch, L, E, *x.shape[2:]).transpose(0, 1).reshape(L, ch * E, *x.shape[2:])


def lstm_reference_model(agent, flat, flat_l):
    """fp32 ppo.ActorCritic (pure-torch cell) holding the recorded parameters, its 2-D weights rounded to bf16 as the kernels
    see them (test_gpu_lstm_update.native_problem)."""
    m = ActorCritic(agent.O, agent.A, (256, 128, 64), rnn=dict(name="lstm", units=256, layers=1, before_mlp=False,
                                                               concat_input=True, layer_norm=True)).to(DEV)
    m.fused_cell = False
    r = m.rnn.rnn
    mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
           m.actor_mlp[4].bias]
    rec = [r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight, m.layer_norm.bias, m.mu.weight,
           m.mu.bias, m.value.weight, m.value.bias, m.sigma]
    with torch.no_grad():
        for vec, prms in ((flat, mlp), (flat_l, rec)):
            o = 0
            for prm in prms:
                prm.copy_(vec[o:o + prm.numel()].view_as(prm))
                o += prm.numel()
                if prm.dim() == 2 and prm.shape[0] > 3:
                    prm.copy_(prm.bfloat16().float())
        assert o == flat_l.numel()
    return m, mlp, rec


def check_lstm_minibatch(agent, up, mb, fin, targets, mu_old, lso, hyp, tag):
    """Gradients of both halves and a_loss / c_loss against fp32 autograd of ActorCritic on the recorded parameters, with
    the float64 targets and the chain's mu_old: the bounds of test_gpu_lstm_block_options.test_minibatch_matches_autograd
    (4e-2 relative Frobenius per tensor, 2e-1 for the sums of both signs SUMS, 3e-2 on a_loss / c_loss; bf16 operands
    through a 4-step recurrence), its mean |mu - mu_autograd| < 2e-2 on the write-back; the KL statistic against float64
    rows on the kernel's own mu (the write-back) with the TOL_STAT / KL_LOG_BIAS bound of the MLP minibatch.
    -> (the write-back mu rows, the float64 KL, its tolerance)."""
    T, L, O = agent.T, agent.seq_len, agent.O
    e0, E = mb["gather"]["e0"], mb["gather"]["E"]
    ch = T // L
    S = ch * E
    rec = mb["minibatch"]
    m, mlp, lst = lstm_reference_model(agent, rec["flat"], rec["flat_l"])
    start = up["start"]
    x = torch.clamp((lstm_rows(start["b_obs"], L, e0, E) - fin["mean"]) * fin["inv_std"], -5.0, 5.0)
    h0 = torch.cat([from_tiles(start["_HH_saved"][c], agent.n)[e0:e0 + E] for c in range(ch)]).float()
    c0 = torch.cat([start["_C_saved"][c][e0:e0 + E] for c in range(ch)])
    nd = lstm_rows(start["_nd_ext"][:T], L, e0, E)
    mu, _, v, _ = m(x, (h0, c0), nd)
    v = v.squeeze(-1)
    f = lambda t: lstm_rows(t, L, e0, E).reshape(L * S, *t.shape[2:])  # noqa: E731
    vo_n, ret_n, adv_n = (f(t).float() for t in targets)
    act, nlpo = f(start["b_act"]), f(start["b_nlp"])
    e = agent.e_clip
    nlp = 0.5 * (((act - mu) / torch.exp(m.sigma)) ** 2).sum(-1) + math.log(2 * math.pi) + m.sigma.sum()
    ratio = torch.exp(nlpo - nlp)
    # the actor term's branch as the kernel's own mu (the write-back) decides it: the fp32 mu is ~1e-2 off the kernel's, which
    # on the rollout's data (no planted margins) would move rows across the ratio clip
    mu_k = f(mb["lstm_reduce"]["scal"][..., 2:4])
    ls = lst[10].detach()
    dk = (act.double() - mu_k.double()) / torch.exp(ls.double())
    ratio_k = torch.exp(nlpo.double() - (0.5 * (dk * dk).sum(-1) + math.log(2 * math.pi) + ls.double().sum()))
    on = ((ratio_k >= 1 - e) & (ratio_k <= 1 + e)) | (-adv_n.double() * ratio_k > -adv_n.double() * ratio_k.clamp(1 - e, 1 + e))
    a_loss = torch.where(on, -adv_n * ratio, (-adv_n * ratio_k.clamp(1 - e, 1 + e)).float()).mean()
    # likewise the value loss's branch, decided on the kernel's own v (debug_out, normalised): torch.max's choice, its
    # half / half split on a tie, and clamp's pass-through inside the clip
    R = mb["head_train"]["dbg"].shape[0] // L
    v_k = mb["head_train"]["dbg"].view(L, R, 4)[:, :S, 2].reshape(L * S)
    gt, lt, pass2 = value_branches(v_k, vo_n, ret_n, e)
    e1 = v - ret_n
    e2 = torch.where(pass2, v - ret_n, vo_n + (v_k - vo_n).clamp(-e, e) - ret_n)
    if agent.clip_value:
        c_loss = torch.where(gt, e1 ** 2, torch.where(lt, e2 ** 2, 0.5 * (e1 ** 2 + e2 ** 2))).mean()
    else:
        c_loss = (e1 ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + m.sigma).sum()
    (a_loss + 0.5 * c_loss * hyp["critic_coef"] - hyp["entropy_coef"] * entropy + b_loss * hyp["bounds_loss_coef"]).backward()
    gm, gl = mb["reduce"]["g"].double(), mb["lstm_reduce"]["g"].double()
    errs, o = {}, 0
    for name, prm in zip(LSTM_NAMES, lst):
        errs[name] = float((gl[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    o = 0
    for name, prm in zip(NAMES[:6], mlp):
        errs[name] = float((gm[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    for k_, e_ in errs.items():
        note(f"lstm grad {k_}", e_)
    # the sums of both signs: each row's term is within the 4e-2 of the other tensors, so their sum is within 4e-2 of the
    # sum of the rows' magnitudes (computed on the kernel's mu and v), whichever is looser than 2e-1 of the net sum
    B = L * S
    sig = torch.exp(ls.double())
    g_nlp = torch.where(on, adv_n.double() * ratio_k, torch.zeros_like(ratio_k))
    dv_rows = hyp["critic_coef"] * torch.maximum((v_k - ret_n).abs(), (e2.detach() - 0).abs()).double()
    mags = {"b_mu": float((g_nlp[:, None] * dk.abs() / sig).abs().sum(0).norm()) / B + hyp["bounds_loss_coef"] * 2.2,
            "b_v": float(dv_rows.sum()) / B,
            "logstd": float((g_nlp[:, None].abs() * (1 + dk * dk)).sum(0).norm()) / B + 2 * hyp["entropy_coef"]}
    for k_ in SUMS:
        prm = lst[LSTM_NAMES.index(k_)]
        errs[k_] = errs[k_] * float(prm.grad.double().norm()) / max(float(prm.grad.double().norm()), 0.2 * mags[k_])
    shown = ", ".join(f"{k_} {e_:.2e}" for k_, e_ in errs.items())
    assert max(e_ for k_, e_ in errs.items() if k_ not in SUMS) < 4e-2, (tag, shown)
    assert max(errs[k_] for k_ in SUMS) < 2e-1, (tag, shown)
    PL = gl.numel() - 4
    assert abs(float(gl[PL]) - float(a_loss)) < 3e-2 * abs(float(a_loss)) + 1e-4, (tag, float(gl[PL]), float(a_loss))
    assert abs(float(gl[PL + 1]) - float(c_loss)) < 3e-2 * float(c_loss), (tag, float(gl[PL + 1]), float(c_loss))
    note("lstm a_loss rel", abs(float(gl[PL]) - float(a_loss)) / (abs(float(a_loss)) + 1e-4))
    note("lstm c_loss rel", abs(float(gl[PL + 1]) - float(c_loss)) / float(c_loss))
    dmu = float((mu_k - mu.detach()).abs().mean())
    assert dmu < 2e-2, (tag, dmu)
    note("lstm write-back mean |mu - mu_autograd|", dmu)
    kl = kl_rows(mu_k, mu_old, lst[10].detach(), lso)
    kl_tol = TOL_STAT * float(kl.abs().mean()) + KL_LOG_BIAS
    err = abs(float(gl[PL + 2]) - float(kl.mean()))
    assert err <= kl_tol, (tag, "kl", err, kl_tol)
    note("lstm stat kl / bound", err / kl_tol)
    return mu_k, float(kl.mean()), kl_tol


LSTM_CASES = {"4096": (4096, []), "ragged_1000": (1000, ["train.params.config.minibatch_size=4000"])}


@pytest.mark.parametrize("case", list(LSTM_CASES))
def test_lstm_update_sequence_against_float64(case):
    """_update_native_lstm (reference network) for two iterations at 4096 envs (2 slots of 2048 envs x 4 mini-epochs) and
    at 1000 envs (4 slots of 250 envs: 1000 sequences padded to 1024 rows per step), with the sequence invariants of
    test_mlp_update_sequence_against_float64 -- the float64 targets (prologue_reference), mu_old in the scalars = the rollout's
    mu / the previous mini-epoch's write-back bit for bit, logstd_old as read by vine_lstm_head_train and vine_ppo_minibatch
    = the chain's, each minibatch's gradients against autograd (check_lstm_minibatch), both Adam launches against float64
    (check_adam) and their re-packs bit for bit, the step count, LrReplay, the state block after the update -- and the
    recurrent path's own facts: both Adam launches of a minibatch read the same lr and step; the MLP half's Adam leaves the
    state block untouched (bookkeeping 0) and vine_lstm_adam adds the loss statistics, counts the minibatch and sets the
    pending KL; the 197 unused MLP head slots stay exactly 0 in the parameters, both moments and the gradient."""
    n, extra = LSTM_CASES[case]
    agent = make_agent(list(extra), n=n)
    assert agent.native_lstm and agent.layer_norm and agent.model.concat_input
    lib, T, O, E, L = agent._lib, agent.T, agent.O, agent.mb_envs, agent.seq_len
    M = agent.n // E
    P, PL = agent.flat.numel(), agent.flat_l.numel()
    hyp = dict(e_clip=agent.e_clip, critic_coef=agent.critic_coef, entropy_coef=agent.entropy_coef,
               bounds_loss_coef=agent.bounds_coef)
    ref_obs, ref_val = RunningMeanStd((O,)).to(DEV), RunningMeanStd(()).to(DEV)
    replay = LrReplay(agent)
    steps = 0
    logs = run_recorded(agent, 2)
    for it, log in enumerate(logs):
        up = group_minibatches(log)[0]
        st0 = up["start"]["state"]
        fin = up["finalize"]
        targets = prologue_reference(agent, up["start"], fin, ref_obs, ref_val, f"{case} it={it}")
        sigma0 = up["start"]["flat_l"][PL - 2:PL].clone()
        assert len(up["mbs"]) == agent.mini_epochs * M
        written, sigma_before_adam, stats = {}, {}, []
        for i, mb in enumerate(up["mbs"]):
            k, slot = divmod(i, M)
            tag = f"{case} it={it} k={k} slot={slot}"
            e0 = mb["gather"]["e0"]
            assert (e0, mb["gather"]["E"]) == (slot * E, E), tag
            rows = lambda x: lstm_rows(x, L, e0, E).reshape(-1, *x.shape[2:])  # noqa: E731
            scal = mb["gather"]["scal"]
            mu_old = rows(up["start"]["b_mu"]) if k == 0 else written[slot]
            assert torch.equal(bits(rows(scal)[:, 2:4].contiguous()), bits(mu_old)), (tag, "mu_old")
            if k == 0:   # the other scalars: the rollout's actions / neglogp and the prologue's targets, as finalize left them
                for j, src in ((0, up["start"]["b_act"][..., 0]), (1, up["start"]["b_act"][..., 1]), (4, up["start"]["b_nlp"]),
                               (5, fin["val_n"]), (6, fin["ret_n"]), (7, fin["adv_n"])):
                    assert torch.equal(bits(rows(scal)[:, j].contiguous()), bits(rows(src))), (tag, j)
            lso = sigma0 if k == 0 else sigma_before_adam[slot]
            for kind in ("head_train", "minibatch"):
                assert mb[kind]["slot"] == slot and torch.equal(bits(mb[kind]["logstd_old"]), bits(lso)), (tag, kind)
            assert mb["head_train"]["writeback"], tag
            rec = mb["minibatch"]
            steps += 1
            assert float(rec["state"][1]) == steps and float(rec["state"][abi.PPO_STATE_EPOCH]) == it + 1, tag
            mu_k, kl64, kl_tol = check_lstm_minibatch(agent, up, mb, fin, targets, mu_old, lso, hyp, tag)
            written[slot] = mu_k.clone()
            g_l = mb["lstm_reduce"]["g"]
            stats.append(g_l[PL:PL + 4].cpu().numpy())
            assert torch.equal(bits(mb["reduce"]["logstd_old"][slot]), bits(rec["flat_l"][PL - 2:PL])), (tag, "sigma copy")
            # the two Adam launches: same lr and step, bookkeeping by vine_lstm_adam only
            am, al = mb["adam"]
            assert not am["lstm"] and am["book"] == 0 and al["lstm"], tag
            assert torch.equal(bits(am["state"]), bits(al["state"])) and torch.equal(bits(am["state_new"]), bits(am["state"])), tag
            kernel_lr = float(al["state"][0])
            replay.launch(k, slot, kernel_lr)
            replay.check(kernel_lr, tag)
            replay.pending = (kl64, kl_tol)
            sn, so = al["state_new"], al["state"]
            assert float(sn[2]) == float(g_l[PL + 2]) and float(sn[3]) == 1.0 and float(sn[8]) == float(so[8]) + 1, tag
            assert float(so[1]) == steps
            for ad, w0, PP in ((am, rec["flat"], P), (al, rec["flat_l"], PL)):
                assert torch.equal(bits(ad["w"]), bits(w0)), tag
                check_adam(ad, kernel_lr, steps, 1.0, PP, tag)
            for vec in (am["w_new"], am["m_new"], am["v_new"], am["g"][:P]):
                assert bool((vec[P - MLP_DUMMY:P] == 0).all()), (tag, "dummy MLP head slots")
            sigma_before_adam[slot] = al["w"][PL - 2:PL].clone()
            # re-packs bit for bit
            pm, pl = torch.zeros_like(am["packed_new"]), torch.zeros_like(al["packed_new"])
            wm = [x.contiguous() for x in mlp_weights(am["w_new"], agent)[:10]]
            assert lib.vine_mlp_pack(*[C.c_void_p(x.data_ptr()) for x in wm], O, C.c_void_p(pm.data_ptr()), None) == 0
            wl, o = [], 0
            for prm in agent._lstm_param_order()[:10]:
                wl.append(al["w_new"][o:o + prm.numel()].view_as(prm).contiguous())
                o += prm.numel()
            assert lib.vine_lstm_pack(*[C.c_void_p(x.data_ptr()) for x in wl], O, C.c_void_p(pl.data_ptr()), None) == 0
            torch.cuda.synchronize()
            assert torch.equal(am["packed_new"], pm) and torch.equal(al["packed_new"], pl), (tag, "re-pack")
        st_end = group_minibatches(logs[it + 1])[0]["start"]["state"] if it + 1 < len(logs) else agent.ppo_state
        check_state_after(st_end, up, st0, stats, steps - len(up["mbs"]), f"{case} it={it}")
        if it == len(logs) - 1:
            for slot in range(M):
                got = lstm_rows(agent._scal, L, slot * E, E).reshape(-1, 8)[:, 2:4]
                assert torch.equal(bits(got.contiguous()), bits(written[slot])), slot
                assert torch.equal(bits(agent._logstd_old[slot]), bits(sigma_before_adam[slot])), slot
    assert replay.skipped <= max(1, replay.decisions // 10), (replay.skipped, replay.decisions)
    print(f"{case}: {replay.decisions} lr decisions, {replay.skipped} within rounding of a threshold")
    report(case)
