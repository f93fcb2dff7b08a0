"""GPU: rl_games' lr_schedule (adaptive / linear), schedule_type (legacy / standard), clip_value and reward_shaper in the
kernel-only PPO update, against their closed forms and the torch baseline.

The learning-rate schedule runs in block 0 of vine_ppo_minibatch, between optimiser steps, so the lr each Adam launch applies
is state[0] right after that launch.  The tests record it with a proxy around the agent's library handle that copies
state[0] into a buffer after every vine_ppo_adam(_clipped) launch, on the same stream: eager and graph-replayed alike (in a
captured graph the copies are captured too)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from vine_robot_isaacgymenvs_b200 import abi

pytestmark = pytest.mark.gpu
DEV = "cuda"
MLP = ["train.params.network.rnn=null"]
LR0 = 3e-4
LR_MIN = float(np.float32(1e-6))


def p(t):
    return C.c_void_p(t.data_ptr())


def make_agent(extra, graphs=False, n=512, **kw):
    import vine_robot_isaacgymenvs_b200 as vine
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", "train.params.config.minibatch_size=4096",
                                              f"train.params.config.learning_rate={LR0}"] + extra)
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=1, use_graphs=graphs, **kw)


def sched(lr_schedule, schedule_type, max_epochs=3, kl_threshold=None):
    out = [f"train.params.config.lr_schedule={lr_schedule}", f"train.params.config.schedule_type={schedule_type}",
           f"train.params.config.max_epochs={max_epochs}"]
    return out + ([f"train.params.config.kl_threshold={kl_threshold}"] if kl_threshold is not None else [])


class LrRecorder:
    """Stands in for the agent's library handle: after every MLP-half Adam launch (one per minibatch on both networks) it
    copies state[0] -- the lr that launch applied -- into buf[i mod per_iter], in stream order."""

    def __init__(self, agent):
        self._lib, self.agent = agent._lib, agent
        self.per_iter = agent.mini_epochs * (agent.n // agent.mb_envs)
        self.buf = torch.zeros(self.per_iter, device=DEV)
        self.i = 0
        agent._lib = self

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name not in ("vine_ppo_adam", "vine_ppo_adam_clipped"):
            return fn

        def recorded(*args):
            rc = fn(*args)
            self.buf[self.i % self.per_iter].copy_(self.agent.ppo_state[0])
            self.i += 1
            return rc
        return recorded


def record_torch_lr(agent):
    """The torch baseline: lr_t right before every optimiser step."""
    per_iter = agent.mini_epochs * (agent.n // agent.mb_envs)
    buf, step, st = torch.zeros(per_iter, device=DEV), agent.opt.step, {"i": 0}

    def recorded(*a, **k):
        buf[st["i"] % per_iter].copy_(agent.lr_t)
        st["i"] += 1
        return step(*a, **k)
    agent.opt.step = recorded
    return buf


def linear_f(epoch, max_epochs):
    lr0 = float(np.float32(LR0))
    return LR_MIN + (lr0 - LR_MIN) * max(0, max_epochs - epoch) / max_epochs


def expected_linear(epoch, max_epochs, K, M, standard):
    """lr of every Adam step of iteration `epoch` (rl_games epoch_num, 1-based): the first step (legacy) or the first mini-epoch
    (standard) still runs with the previous iteration's f(epoch - 1), every later one with f(epoch)."""
    return [linear_f(epoch - 1 if (k == 0 and (standard or j == 0)) else epoch, max_epochs) for k in range(K) for j in range(M)]


def expected_forced_adaptive(epoch, K, M, standard):
    """A kl_threshold every KL exceeds twice: every run of the rule divides by 1.5 (f32, like both implementations)."""
    out = []
    lr = np.float32(LR0)
    for e in range(1, epoch + 1):
        for k in range(K):
            for j in range(M):
                if e == epoch:
                    out.append(float(lr))
                if not standard or j == M - 1:
                    lr = max(np.float32(lr / np.float32(1.5)), np.float32(1e-6))
    return out


def assert_within_one_ulp(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        assert abs(g - w) <= float(np.spacing(np.float32(w))), (what, i, g, w, got, want)


# ---------------------------------------------------------------------------------------------- 1. lr sequence, closed form
@pytest.mark.parametrize("net", ["mlp", "lstm"])
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
@pytest.mark.parametrize("stype", ["legacy", "standard"])
def test_linear_lr_sequence_matches_the_closed_form(net, graphs, stype):
    """lr_schedule linear: the lr of every Adam launch over several iterations, into the floor, is
    f(e) = 1e-6 + (lr0 - 1e-6) max(0, max_epochs - e) / max_epochs at the cadence of schedule_type, within 1 f32 ulp.
    With graphs, the first train_epoch runs three eager warm-up iterations before the first replay; max_epochs is longer
    there so that the replays still see the decay."""
    max_epochs = 6 if graphs else 3
    a = make_agent((MLP if net == "mlp" else []) + sched("linear", stype, max_epochs), graphs)
    assert a.linear_lr and a.schedule_standard == (stype == "standard") and a.fused_update
    rec = LrRecorder(a)
    K, M = a.mini_epochs, a.n // a.mb_envs
    assert (K, M) == (4, 2)
    seen = 0
    for _ in range(4):
        a.train_epoch()
        torch.cuda.synchronize()
        got = rec.buf.tolist()
        assert_within_one_ulp(got, expected_linear(a.epoch, max_epochs, K, M, stype == "standard"), (net, a.epoch))
        seen = max(seen, a.epoch)
    assert seen > max_epochs                                         # reached the floor
    assert float(a.ppo_state[abi.PPO_STATE_EPOCH]) == a.epoch
    assert abs(rec.buf[-1].item() - LR_MIN) <= float(np.spacing(np.float32(LR_MIN)))


@pytest.mark.parametrize("net", ["mlp", "lstm"])
@pytest.mark.parametrize("case", ["linear-legacy", "linear-standard", "adaptive-standard"])
def test_kernel_and_torch_paths_apply_the_same_lr_sequence(net, case):
    """The kernel path and the torch baseline apply the same lr at every Adam step over three iterations (within 1 f32 ulp), and
    both equal the closed form: linear x {legacy, standard}, and adaptive x standard with a kl_threshold every KL exceeds
    twice, so that every run of the rule divides by 1.5 -- once per mini-epoch, not once per minibatch."""
    lr_schedule, stype = case.split("-")
    extra = (MLP if net == "mlp" else []) + sched(lr_schedule, stype, 3, kl_threshold=1e-9 if lr_schedule == "adaptive" else None)
    a = make_agent(extra, use_fused_update=True)
    b = make_agent(extra, use_fused_update=False)
    assert a.fused_update and not b.fused_update
    rec, buf_b = LrRecorder(a), record_torch_lr(b)
    K, M = a.mini_epochs, a.n // a.mb_envs
    for _ in range(3):
        a.train_epoch()
        b.train_epoch()
        torch.cuda.synchronize()
        ga, gb = rec.buf.tolist(), buf_b.tolist()
        want = (expected_linear(a.epoch, 3, K, M, stype == "standard") if lr_schedule == "linear"
                else expected_forced_adaptive(a.epoch, K, M, True))
        assert_within_one_ulp(ga, want, ("kernel", a.epoch))
        if lr_schedule == "linear":   # f64 closed form, one rounding to f32 on both paths
            assert_within_one_ulp(gb, want, ("torch", b.epoch))
            assert_within_one_ulp(ga, gb, ("kernel vs torch", a.epoch))
        else:                         # torch divides by a scalar as a multiplication by its f32 reciprocal: an ulp per step
            assert all(abs(x - y) <= 1e-6 * y for x, y in zip(gb, want)), (gb, want)


# ------------------------------------------------------------------------------------ 2. standard acts on the mean KL (ABI)
def test_standard_schedule_acts_on_the_mean_kl_of_the_mini_epoch():
    """vine_ppo_minibatch driven directly, the KL of each minibatch written into state[2] / state[3] between launches as the
    Adam bookkeeping would: KLs of 3x and 0.1x kl_threshold in one mini-epoch.  legacy: /1.5 after the first, x1.5 after the
    second.  standard: the mean (1.55x) is inside the band, the lr stays; a mean of 2.5x divides once, when the next
    mini-epoch opens.  Each launch with epoch_begin counts one iteration in state[11]."""
    a = make_agent(MLP)
    a._rollout()
    a._update_any()            # builds the per-(mini-epoch, slot) launch structs
    torch.cuda.synchronize()
    thr = a.kl_threshold
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(standard, kls):
        state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
        state[0] = 1e-3
        lrs = []
        flags = [(1, 1)] + [(0, 0)] * (len(kls) - 1) + [(0, 1)]      # (epoch_begin, mini_epoch_begin) of each launch
        for i, (eb, mb_begin) in enumerate(flags):
            mb = abi.VinePpoMinibatch.from_buffer_copy(a._mb_structs[0][0])
            mb.state, mb.schedule_standard, mb.epoch_begin, mb.mini_epoch_begin = state.data_ptr(), int(standard), eb, mb_begin
            assert mb.adaptive_lr == 1 and mb.lr_linear == 0
            assert a._lib.vine_ppo_minibatch(C.byref(mb), stream) > 0
            torch.cuda.synchronize()
            lrs.append(float(state[0]))
            if i < len(kls):
                state[2], state[3] = kls[i] * thr, 1.0
        assert float(state[abi.PPO_STATE_EPOCH]) == 1.0 and float(state[1]) == len(flags)
        return lrs, state

    f32 = np.float32
    lrs, _ = run(False, [3.0, 0.1])
    assert lrs == [float(f32(1e-3)), float(f32(1e-3) / f32(1.5)), float((f32(1e-3) / f32(1.5)) * f32(1.5))]
    lrs, st = run(True, [3.0, 0.1])
    assert lrs == [float(f32(1e-3))] * 3
    assert float(st[abi.PPO_STATE_EPOCH_KL_SUM]) == 0.0 and float(st[abi.PPO_STATE_EPOCH_KL_COUNT]) == 0.0
    lrs, _ = run(True, [3.0, 2.0])
    assert lrs == [float(f32(1e-3))] * 2 + [float(f32(1e-3) / f32(1.5))]


# -------------------------------------------------------------------------------------------------- 3. agent level, standard
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_adaptive_standard_update_follows_the_torch_update(net):
    """Same rollout, adaptive + standard, 4 mini-epochs x 2 minibatches, two iterations: the kernel path and the torch path
    take the same x1.5 / /1.5 decisions up to one (bf16 GEMMs may move one borderline mean across a threshold, as in
    test_full_update_kl_and_learning_rate_follow_the_torch_update), and the kernel's lr only changes between mini-epochs."""
    extra = (MLP if net == "mlp" else []) + sched("adaptive", "standard")
    a = make_agent(extra, use_fused_update=True)
    b = make_agent(extra, use_fused_update=False)
    b.load_state_dict(a.state_dict())
    rec = LrRecorder(a)
    for _ in range(2):
        a._rollout()
        for name in ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "b_adv", "b_done"):
            getattr(b, name).copy_(getattr(a, name))
        if net == "lstm":
            from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles
            for ck in range(a.T // a.seq_len):
                b.b_h[ck].copy_(from_tiles(a._HH_saved[ck], a.n))
                b.b_c[ck].copy_(a._C_saved[ck])
        a.pop_stats(); b.pop_stats()
        a._update_any()
        b._update_any()
        a.epoch += 1
        b.epoch += 1
        torch.cuda.synchronize()
        sa, sb = a.pop_stats(), b.pop_stats()
        assert abs(sa["kl"] - sb["kl"]) <= 0.15 * sb["kl"] + 2e-5, (sa["kl"], sb["kl"])
        # the kernel applies the last mini-epoch's decision when the next update opens: compare after applying it by hand
        st = a.ppo_state
        lr_a = float(st[0])
        mean_kl = (float(st[abi.PPO_STATE_EPOCH_KL_SUM]) + float(st[2]) * float(st[3])) / (float(st[abi.PPO_STATE_EPOCH_KL_COUNT]) + float(st[3]))
        if mean_kl > 2 * a.kl_threshold:
            lr_a = max(lr_a / 1.5, 1e-6)
        elif mean_kl < 0.5 * a.kl_threshold:
            lr_a = min(lr_a * 1.5, 1e-2)
        assert abs(math.log(lr_a / b.lr) / math.log(1.5)) <= 1.01, (lr_a, b.lr)
        lrs = rec.buf.view(a.mini_epochs, -1)
        assert bool((lrs == lrs[:, :1]).all()), lrs                # constant within every mini-epoch
        b.load_state_dict(a.state_dict())
        b.lr_t.fill_(lr_a)


# -------------------------------------------------------------------------------------------------- 4. clip_value False
HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.0, bounds_loss_coef=1e-4)


def mlp_reference_unclipped(W, buf, mean, inv_std, e0, E, hyp):
    """fp32 autograd restatement of the torch update's loss with clip_value False (weights rounded to bf16 like the kernel)."""
    leaves = [w.clone().requires_grad_(True) for w in W]
    w1, b1, w2, b2, w3, b3, wmu, bmu, wv, bv, logstd = leaves
    sl = lambda t: t[:, e0:e0 + E].reshape(-1, *t.shape[2:])  # noqa: E731
    q = lambda w: w + (w.bfloat16().float() - w).detach()  # noqa: E731
    x = torch.clamp((sl(buf["obs"]) - mean) * inv_std, -5, 5)
    h = torch.nn.functional.elu(x @ q(w1).t() + b1)
    h = torch.nn.functional.elu(h @ q(w2).t() + b2)
    h = torch.nn.functional.elu(h @ q(w3).t() + b3)
    mu, v = h @ q(wmu).t() + bmu, (h @ q(wv).t() + bv).squeeze(-1)
    sigma = torch.exp(logstd)
    act, adv, ret = sl(buf["act"]), sl(buf["adv"]), sl(buf["ret"])
    nlp = 0.5 * (((act - mu) / sigma) ** 2).sum(-1) + 0.5 * math.log(2 * math.pi) * 2 + logstd.sum()
    ratio = torch.exp(sl(buf["nlp_old"]) - nlp)
    a_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - hyp["e_clip"], 1 + hyp["e_clip"])).mean()
    c_loss = ((v - ret) ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + logstd).sum()
    loss = a_loss + 0.5 * c_loss * hyp["critic_coef"] - hyp["entropy_coef"] * entropy + b_loss * hyp["bounds_loss_coef"]
    loss.backward()
    return [l.grad for l in leaves], c_loss.item()


@pytest.mark.parametrize("T,N,e0,E,O", [(16, 256, 0, 128, 18), (8, 600, 100, 333, 28)])
def test_unclipped_value_loss_minibatch_gradients_match_autograd(T, N, e0, E, O):
    """value_loss_unclipped = 1: every gradient tensor within 3e-2 relative Frobenius norm of autograd with (ret - v)^2 and
    c_loss within 2e-2 (the tolerances of test_fused_minibatch_gradients_match_autograd).  The inputs have rows with
    |v - v_old| > e_clip; the clipped and unclipped value gradients differ by exactly what those rows contribute to the value
    bias; and with v_old = v on every row (nothing clipped) the two flags give the same bits."""
    from test_gpu_ppo_fused import NAMES, make_problem, run_kernel, split
    lib = abi.load_library()
    W, buf, mean, inv_std, logstd_old = make_problem(T, N, O, seed=7 * T + O)
    un = dict(HYP, value_loss_unclipped=1)
    _, _, _, out_u, dbg, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, un, O, T, N)
    _, _, _, out_c, _, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, HYP, O, T, N)
    grads, c_loss = mlp_reference_unclipped(W, buf, mean, inv_std, e0, E, HYP)
    P = lib.vine_ppo_num_params(O)
    errs = {k: float((g - r).norm() / (r.norm() + 1e-12)) for k, g, r in zip(NAMES, split(out_u[:P], W), grads)}
    assert max(errs.values()) < 3e-2, errs
    assert abs(float(out_u[P + 1]) - c_loss) <= 2e-2 * c_loss + 1e-5
    # rows where clipping changes the value gradient: |v - v_old| > e_clip and the clipped error is the larger one
    sl = lambda t: t[:, e0:e0 + E].reshape(-1)  # noqa: E731
    v, vo, ret = dbg[:, 2].double(), sl(buf["val_old"]).double(), sl(buf["ret"]).double()
    e = HYP["e_clip"]
    vc = vo + (v - vo).clamp(-e, e)
    rows = ((v - vo).abs() > e) & ((vc - ret) ** 2 > (v - ret) ** 2)
    assert 0.05 < float(rows.double().mean()) < 0.95
    B = v.numel()
    i_bv = P - 3                                                     # the value bias: sum over rows of d(loss)/dv
    want = float((HYP["critic_coef"] * (v - ret))[rows].sum() / B)
    assert abs(float(out_u[i_bv] - out_c[i_bv]) - want) <= 2e-2 * abs(want), (float(out_u[i_bv] - out_c[i_bv]), want)
    # nothing clipped: same bits
    buf["val_old"][:, e0:e0 + E] = dbg[:, 2].view(T, E)
    _, _, st_u, out_u, _, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, un, O, T, N)
    _, _, st_c, out_c, _, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, HYP, O, T, N)
    assert torch.equal(out_u.view(torch.int32), out_c.view(torch.int32))


def head_reference_unclipped(Pd, hq, scal, logstd_old, hyp):
    leaves = {k: Pd[k].clone().requires_grad_(True) for k in ("ln_g", "ln_b", "w_mu", "b_mu", "w_v", "b_v", "logstd")}
    hr = hq.clone().requires_grad_(True)
    y = torch.nn.functional.layer_norm(hr, (256,), leaves["ln_g"], leaves["ln_b"], 1e-5)
    mu, v = y @ leaves["w_mu"].t() + leaves["b_mu"], (y @ leaves["w_v"].t() + leaves["b_v"])[:, 0]
    ls = leaves["logstd"]
    act, nlpo, ret, adv = scal[:, :2], scal[:, 4], scal[:, 6], scal[:, 7]
    nlp = 0.5 * (((act - mu) / torch.exp(ls)) ** 2).sum(-1) + math.log(2 * math.pi) + ls.sum()
    ratio = torch.exp(nlpo - nlp)
    e = hyp["e_clip"]
    a_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - e, 1 + e)).mean()
    c_loss = ((v - ret) ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + ls).sum()
    loss = a_loss + 0.5 * hyp["critic_coef"] * c_loss - hyp["entropy_coef"] * entropy + hyp["bounds_loss_coef"] * b_loss
    loss.backward()
    return v.detach(), hr.grad, {k: t.grad for k, t in leaves.items()}, c_loss.item()


def test_unclipped_value_loss_head_train_matches_float64():
    """vine_lstm_head_train with value_loss_unclipped = 1 against the float64 reference of test_gpu_lstm_update.py with
    (ret - v)^2 (same tolerances), and per row: dh differs from the clipped launch exactly on the rows whose value is clipped
    with the clipped error the larger one."""
    from test_gpu_lstm_update import HEAD_HYP, SENT_BF16, bf16_ulp, from_tiles, head_problem, pack, rel
    lib = abi.load_library()
    n = 32768
    P, HH, hq, scal, logstd_old = head_problem(n, 900, HEAD_HYP)
    lp = pack(lib, P, 18)
    outs = {}
    for unclipped in (0, 1):
        DH = torch.full_like(HH, SENT_BF16)
        gparts = torch.zeros(abi.LSTM_HEAD_GRAD_PARTS, abi.LSTM_HEAD_GRAD_FLOATS, device=DEV)
        ht = abi.VineLstmHeadTrain(params=lp.data_ptr(), hh=HH.data_ptr(), scalars=scal.data_ptr(), logstd=P["logstd"].data_ptr(),
                                   logstd_old=logstd_old.data_ptr(), dh=DH.data_ptr(), grads=gparts.data_ptr(), n=n, inv_B=1.0 / n,
                                   value_loss_unclipped=unclipped, **HEAD_HYP)
        nparts = lib.vine_lstm_head_train(C.byref(ht), None)
        assert nparts > 0
        torch.cuda.synchronize()
        outs[unclipped] = (from_tiles(DH, n).double(), gparts[:nparts].double().sum(0))
    Pd = {k: P[k].double() for k in P}
    v, dh_ref, grads, c_loss = head_reference_unclipped(Pd, hq, scal.double(), logstd_old, HEAD_HYP)
    dh, gs = outs[1]
    row_max = dh_ref.abs().amax(-1, keepdim=True)
    tol = bf16_ulp(dh_ref) + 1e-4 * row_max + 1e-5 * row_max.median()
    assert bool(((dh - dh_ref).abs() <= tol).all()), float(((dh - dh_ref).abs() - tol).max())
    errs = {"ln_g": rel(gs[0:256], grads["ln_g"]), "ln_b": rel(gs[256:512], grads["ln_b"]),
            "w_v": rel(gs[1024:1280], grads["w_v"].reshape(-1)), "b_v": rel(gs[1282:1283], grads["b_v"]),
            "w_mu": rel(gs[512:1024], grads["w_mu"].reshape(-1)), "c_loss": abs(float(gs[1287]) - c_loss) / c_loss}
    assert max(errs.values()) < 1e-4, errs
    e = HEAD_HYP["e_clip"]
    vo, ret = scal[:, 5].double(), scal[:, 6].double()
    vc = vo + (v - vo).clamp(-e, e)
    rows = ((v - vo).abs() > e) & ((vc - ret) ** 2 > (v - ret) ** 2)
    assert 0.05 < float(rows.double().mean()) < 0.95
    differ = (outs[0][0] != outs[1][0]).any(-1)
    assert torch.equal(differ, rows), (int(differ.sum()), int(rows.sum()), int((differ ^ rows).sum()))


# ------------------------------------------------------------------------------------------------------- 5. reward shaper
@pytest.mark.parametrize("shift,lo,hi", [(0.5, -1.5, 2.0), (0.0, -math.inf, math.inf), (-3.0, -math.inf, 0.25)])
def test_rollout_post_reward_shaper_matches_torch_bit_for_bit(shift, lo, hi):
    """vine_rollout_post against PPOAgent._shape_rewards (the torch rollout's formula): clamp((r + shift) * scale, min, max),
    bit for bit, with finite bounds that clip a real fraction of rows, a NaN reward that stays NaN and a -0 reward; shift 0
    with infinite bounds is exactly r * scale (-0 stays -0)."""
    from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
    lib = abi.load_library()
    n = 5000
    g = torch.Generator(device=DEV).manual_seed(3)
    rew = torch.randn(n, device=DEV, generator=g) * 400 + 100
    rew[7], rew[8], rew[9] = float("nan"), -0.0, float("inf")
    resets = torch.zeros(n, dtype=torch.int64, device=DEV)
    timeouts = torch.zeros(n, dtype=torch.uint8, device=DEV)
    values = torch.zeros(n, device=DEV)
    shaped, dones = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    ep_ret, ep_len = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    stats = torch.zeros(4, dtype=torch.float64, device=DEV)
    scale = 0.01
    shaper = PPOAgent.__new__(PPOAgent)
    shaper.reward_scale, shaper.reward_shift, shaper.reward_min, shaper.reward_max = scale, shift, lo, hi
    shaper.reward_clamp = lo > -math.inf or hi < math.inf
    a = abi.VineRolloutPost(rewards=rew.data_ptr(), resets=resets.data_ptr(), timeouts=timeouts.data_ptr(), values=values.data_ptr(),
                            shaped_rewards=shaped.data_ptr(), dones_next=dones.data_ptr(), ep_return=ep_ret.data_ptr(),
                            ep_length=ep_len.data_ptr(), ep_stats=stats.data_ptr(), n=n, gamma=0.99, value_bootstrap=0,
                            success_reward_threshold=500.0, **shaper._shaper_fields())
    assert lib.vine_rollout_post(C.byref(a), None) == 0
    torch.cuda.synchronize()
    want = shaper._shape_rewards(rew)
    assert torch.equal(shaped.view(torch.int32), want.view(torch.int32))
    assert math.isnan(float(shaped[7]))
    if shaper.reward_clamp:
        assert float((shaped == hi).double().mean()) > 0.05 or hi == math.inf
        assert float((shaped == lo).double().mean()) > 0.05 or lo == -math.inf
    if shift == 0.0 and not shaper.reward_clamp:
        assert torch.equal(shaped.view(torch.int32), (rew * scale).view(torch.int32))
        assert str(float(shaped[8])) == "-0.0"


# ---------------------------------------------------------------------------------------------------------------- 6. resume
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_resumed_linear_run_continues_the_lr_sequence(net):
    """Save a linear + legacy run after two iterations, load it into a fresh agent: the next iteration's lr values are
    f(2) for the first step and f(3) after, as if the run had not stopped."""
    extra = (MLP if net == "mlp" else []) + sched("linear", "legacy", 5)
    a = make_agent(extra)
    for _ in range(2):
        a.train_epoch()
    sd = a.state_dict()
    b = make_agent(extra)
    b.load_state_dict(sd)
    assert float(b.ppo_state[abi.PPO_STATE_EPOCH]) == 2.0 and b.epoch == 2
    rec = LrRecorder(b)
    b.train_epoch()
    torch.cuda.synchronize()
    K, M = b.mini_epochs, b.n // b.mb_envs
    assert_within_one_ulp(rec.buf.tolist(), expected_linear(3, 5, K, M, False), net)


# ------------------------------------------------------------------------------------------------------------- 7. two GPUs
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs with peer access")
def test_linear_standard_training_keeps_ranks_bit_identical_on_two_gpus():
    import json
    import os
    import subprocess
    import sys
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", os.path.join(repo, "tools", "lr_schedule_multi_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=repo, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    assert d["world"] == 2
    for net in ("mlp", "lstm"):
        for mode in ("p2p", "nccl"):
            res = d[net][mode]
            assert res["params_bit_identical_across_ranks"] and res["lr_bit_identical_across_ranks"] and res["finite"], (net, mode)
            assert abs(res["lr"] - res["lr_expected"]) <= float(np.spacing(np.float32(res["lr_expected"]))), (net, mode, res)
