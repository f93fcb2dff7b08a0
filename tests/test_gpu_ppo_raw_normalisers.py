"""GPU: kernel-only PPO with rl_games' input and/or value normaliser switched off (normalize_input / normalize_value False).

rl_games semantics: without normalize_input the network sees the observations as they are (no mean, std or +-5 clamp; with
concat_input also the x part of the LSTM input); without normalize_value the rollout's value is the value head's output and
the value targets enter the loss unnormalised and unclamped.  The kernels take this from the raw_obs / raw_value flags of
their argument structs and then read no statistics (the pointers are NULL here, or NaN where a read would show).

The env clamps its observations at +-5, so the kernel-level checks feed observations beyond that themselves; values are
planted beyond +-5 through the value head's bias.  Tolerances are those of the tests each check follows, named there."""
import ctypes as C
import math

import pytest
import torch

import vine_robot_isaacgymenvs_b200 as vine
from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200 import config as vcfg
from vine_robot_isaacgymenvs_b200.ppo.lstm_native import NativeLstmPath
from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic, PPOAgent
from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles, to_tiles
from test_gpu_lstm_update import loss_scalars
from test_gpu_mlp_update import MARGIN, bf, check_h3, check_heads, check_nlp, elu, rows_of, set_scalars
from test_gpu_ppo_fused import HYP, NAMES, make_problem, p, run_kernel, split

pytestmark = pytest.mark.gpu
DEV = "cuda"
RNN = {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": True, "layer_norm": True}
RAW = {"input": ["train.params.config.normalize_input=False"], "value": ["train.params.config.normalize_value=False"]}
RAW["both"] = RAW["input"] + RAW["value"]
bits = lambda t: t.contiguous().view(torch.int32)  # noqa: E731


def forward_raw(W, obs):
    """float64 forward on the kernel's bf16 operands with raw observations: x = bf16(obs), no clamp."""
    w1, b1, w2, b2, w3, b3, wmu, bmu, wv, bv = [w.double() for w in W[:10]]
    O = obs.shape[1]
    x = bf(obs)
    h1 = bf(elu(x @ bf(w1).t() + b1))
    h2 = bf(elu(h1 @ bf(w2).t() + b2))
    h3 = bf(elu(h2 @ bf(w3).t() + b3))
    wh, bh = torch.cat([bf(wmu), bf(wv)]), torch.cat([bmu, bv])
    return dict(x=x, h1=h1, h2=h2, h3=h3, wh=wh, bh=bh, O=O)


def act_raw(lib, packed, obs, logstd, n, O, raw_value=1, u_out=None):
    """vine_policy_act with raw_obs and NULL observation statistics (raw_value: NULL value statistics too)."""
    vstats = torch.tensor([0.3, 1.7], device=DEV)
    out = dict(mu=torch.zeros(n, 2, device=DEV), value=torch.zeros(n, device=DEV), actions=torch.zeros(n, 2, device=DEV),
               neglogp=torch.zeros(n, device=DEV), env_actions=torch.zeros(n, 2, device=DEV))
    counter = torch.zeros(1, dtype=torch.int32, device=DEV)
    ptrs = {k: v.data_ptr() for k, v in out.items()} if u_out is None else dict(u_out=u_out.data_ptr())
    a = abi.VinePolicyAct(packed=packed.data_ptr(), obs=obs.data_ptr(), obs_mean=None, obs_inv_std=None,
                          value_stats=None if raw_value else vstats.data_ptr(), logstd=logstd.data_ptr(),
                          rng_counter=counter.data_ptr(), n=n, num_obs=O, seed=99, raw_obs=1, raw_value=raw_value, **ptrs)
    assert lib.vine_policy_act(C.byref(a), None) == 0
    torch.cuda.synchronize()
    return out


def mlp_net(n, O, seed, obs_scale, v_bias=None):
    lib = abi.load_library()
    W, buf, _, _, _ = make_problem(1, n, O, seed=seed)
    if v_bias is not None:
        W[9].fill_(v_bias)
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_mlp_pack(*[p(w.contiguous()) for w in W[:10]], O, p(packed), None) == 0
    return lib, W, (buf["obs"][0] * obs_scale).contiguous(), packed


# ------------------------------------------------------------------------------------------------ 1. vine_policy_act, raw_obs
@pytest.mark.parametrize("O", [18, 28])
def test_policy_act_raw_obs_matches_float64(O):
    """raw_obs with NULL statistics and |obs| up to ~30 (n = 40 tiles + 45 rows): the U tile's x columns are bf16(obs) bit for
    bit (the constant 1 at column 95, zeros between), h3 follows float64 on those operands (check_h3), and the sampling
    launch's mu / raw value follow float64 on the kernel's own h3 (check_heads), neglogp too (check_nlp)."""
    n = 40 * 128 + 45
    lib, W, obs, packed = mlp_net(n, O, 700 + O, 4.0)
    assert float((obs.abs() > 5).double().mean()) > 0.1
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    U = torch.full(((n + 127) // 128, 1, 128 * 128), 7.0, dtype=torch.bfloat16, device=DEV)
    act_raw(lib, packed, obs, logstd, n, O, u_out=U)
    u = from_tiles(U, n).double()
    fwd = forward_raw(W, obs)
    assert torch.equal(u[:, 64:64 + O].float().bfloat16().view(torch.int16), obs.bfloat16().view(torch.int16))
    assert float(u[:, 95].min()) == 1.0 and float(u[:, 64 + O:95].abs().sum()) == 0.0
    frac, worst = check_h3(u[:, :64], fwd, W[4])
    o = act_raw(lib, packed, obs, logstd, n, O)
    check_heads(o["mu"], o["value"], u[:, :64], fwd["wh"], fwd["bh"])
    check_nlp(o["neglogp"], o["mu"], o["actions"], logstd)
    assert torch.equal(o["env_actions"], o["actions"].clamp(-1, 1))
    print(f"O={O}: h3 {frac:.2e} of elements differ from float64, by <= {worst:.1f} bf16 ulp")


def test_policy_act_raw_obs_is_the_identity_normaliser_inside_the_clamp():
    """|obs| <= 5, mean 0, inv_std 1: raw_obs = 0 and 1 give the same bits in every output ((x - 0) * 1 = x and the clamp
    is inactive), through vine_policy_act and through vine_mlp_forward's NULL statistics."""
    n, O = 5000, 18
    lib, W, obs, packed = mlp_net(n, O, 41, 1.0)
    obs.clamp_(-5.0, 5.0)
    mean, inv_std, vstats = torch.zeros(O, device=DEV), torch.ones(O, device=DEV), torch.tensor([0.3, 1.7], device=DEV)
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    outs = []
    for raw in (0, 1):
        out = dict(mu=torch.zeros(n, 2, device=DEV), value=torch.zeros(n, device=DEV), actions=torch.zeros(n, 2, device=DEV),
                   neglogp=torch.zeros(n, device=DEV))
        counter = torch.zeros(1, dtype=torch.int32, device=DEV)
        a = abi.VinePolicyAct(packed=packed.data_ptr(), obs=obs.data_ptr(), obs_mean=None if raw else mean.data_ptr(),
                              obs_inv_std=None if raw else inv_std.data_ptr(), value_stats=vstats.data_ptr(),
                              logstd=logstd.data_ptr(), rng_counter=counter.data_ptr(), n=n, num_obs=O, seed=5, raw_obs=raw,
                              **{k: v.data_ptr() for k, v in out.items()})
        assert lib.vine_policy_act(C.byref(a), None) == 0
        outs.append(out)
    mu2, v2 = torch.zeros(n, 2, device=DEV), torch.zeros(n, device=DEV)
    assert lib.vine_mlp_forward(p(packed), p(obs), None, None, n, O, p(vstats), p(mu2), p(v2), None) == 0
    torch.cuda.synchronize()
    for k in outs[0]:
        assert torch.equal(bits(outs[0][k]), bits(outs[1][k])), k
    assert torch.equal(bits(mu2), bits(outs[0]["mu"])) and torch.equal(bits(v2), bits(outs[0]["value"]))
    # one statistics pointer without the other is refused
    assert lib.vine_mlp_forward(p(packed), p(obs), p(mean), None, n, O, p(vstats), p(mu2), p(v2), None) == abi.ERR_INVALID_ARG


# ---------------------------------------------------------------------------------------------------------- 2. raw_value
@pytest.mark.parametrize("v_bias", [8.0, -8.0])
def test_policy_act_raw_value_is_the_head_output(v_bias):
    """Value bias +-8: the head output is near +-8 on every row; with raw_value the value is that output (check_heads on the
    kernel's own h3), never clamped to 5; vine_mlp_forward with NULL value statistics gives the same bits."""
    n, O = 3000, 18
    lib, W, obs, packed = mlp_net(n, O, 43, 1.0, v_bias=v_bias)
    obs.clamp_(-5.0, 5.0)
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    U = torch.zeros(((n + 127) // 128, 1, 128 * 128), dtype=torch.bfloat16, device=DEV)
    act_raw(lib, packed, obs, logstd, n, O, u_out=U)
    o = act_raw(lib, packed, obs, logstd, n, O)
    u = from_tiles(U, n).double()
    fwd = forward_raw(W, obs)
    assert float((o["value"].abs() > 6).double().mean()) > 0.9 and float(o["value"].sign().mean()) == math.copysign(1, v_bias)
    check_heads(o["mu"], o["value"], u[:, :64], fwd["wh"], fwd["bh"])
    mu2, v2 = torch.zeros(n, 2, device=DEV), torch.zeros(n, device=DEV)
    assert lib.vine_mlp_forward(p(packed), p(obs), None, None, n, O, None, p(mu2), p(v2), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(bits(v2), bits(o["value"])) and torch.equal(bits(mu2), bits(o["mu"]))


def lstm_params(O, seed, v_bias):
    torch.manual_seed(seed)
    m = ActorCritic(O, 2, (256, 128, 64), rnn=RNN).to(DEV)
    with torch.no_grad():
        m.layer_norm.weight.uniform_(0.5, 1.5)
        m.layer_norm.bias.uniform_(-0.2, 0.2)
        m.value.bias.fill_(v_bias)
    r = m.rnn.rnn
    lp = [t.detach().contiguous() for t in (r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight,
                                            m.layer_norm.bias, m.mu.weight, m.mu.bias, m.value.weight, m.value.bias)]
    packed = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert abi.load_library().vine_lstm_pack(*[p(t) for t in lp], O, p(packed), None) == 0
    return m, packed


@pytest.mark.parametrize("v_bias", [8.0, -8.0])
def test_lstm_head_raw_value_is_the_head_output(v_bias):
    """vine_lstm_head (rollout mode, n = 9600: the grid-stride loop) with raw_value and NULL value statistics: the value is the
    value head on the float64 LayerNorm of the bf16 hidden state (biased variance, eps 1e-5), within the check_heads bound
    widened by the LayerNorm's f32 rounding (2e-5 of sum |w y| + |b|), near +-8 and never clamped; mu is the same bits as
    with the normaliser on."""
    O, n = 18, 9600
    lib = abi.load_library()
    m, packed = lstm_params(O, 11, v_bias)
    h = (torch.randn(n, 256, device=DEV) * 0.7).bfloat16().float()
    hh = to_tiles(h)
    vstats = torch.tensor([0.3, 1.7], device=DEV)
    res = []
    for raw in (1, 0):
        mu, val = torch.zeros(n, 2, device=DEV), torch.zeros(n, device=DEV)
        a = abi.VineLstmHead(params=packed.data_ptr(), hh=hh.data_ptr(), value_stats=None if raw else vstats.data_ptr(),
                             mu=mu.data_ptr(), value=val.data_ptr(), n=n, raw_value=raw)
        assert lib.vine_lstm_head(C.byref(a), None) == 0
        res.append((mu, val))
    torch.cuda.synchronize()
    (mu, val), (mu_n, val_n) = res
    hd = h.double()
    y = (hd - hd.mean(-1, keepdim=True)) / torch.sqrt(hd.var(-1, unbiased=False, keepdim=True) + 1e-5)
    y = y * m.layer_norm.weight.double() + m.layer_norm.bias.double()
    w, b = m.value.weight.double()[0], float(m.value.bias)
    ref = y @ w + b
    tol = 2e-5 * (y.abs() @ w.abs() + abs(b)) + 1e-6
    assert bool(((val.double() - ref).abs() <= tol).all()), float(((val.double() - ref).abs() - tol).max())
    assert float((val.abs() > 6).double().mean()) > 0.9
    assert torch.equal(bits(mu), bits(mu_n))
    assert float(val_n.abs().max()) <= 5.0 * 1.7 + 0.3 + 1e-5 < float(val.abs().max())


# ------------------------------------------------------------------------------------------------ 3. vine_ppo_minibatch, raw_obs
def reference_raw(W, buf, logstd_old, e0, E, hyp):
    """fp32 autograd of ppo.PPOAgent._update's loss on raw observations (test_gpu_ppo_fused.reference without the
    normaliser).  Weights and activations enter the GEMMs rounded to bf16 like the kernel's operands (straight-through for
    the gradient): with raw observations up to ~30 the outputs reach |mu| ~ 15, where f32 activations alone would move the
    log-ratio by ~0.2 and send rows near a clip boundary down the other branch of the loss."""
    leaves = [w.clone().requires_grad_(True) for w in W]
    w1, b1, w2, b2, w3, b3, wmu, bmu, wv, bv, logstd = leaves
    sl = lambda t: t[:, e0:e0 + E].reshape(-1, *t.shape[2:])  # noqa: E731
    q = lambda w: w + (w.bfloat16().float() - w).detach()  # noqa: E731
    h = torch.nn.functional.elu(q(sl(buf["obs"])) @ q(w1).t() + b1)
    h = torch.nn.functional.elu(q(h) @ q(w2).t() + b2)
    h = torch.nn.functional.elu(q(h) @ q(w3).t() + b3)
    h = q(h)
    mu = h @ q(wmu).t() + bmu
    v = (h @ q(wv).t() + bv).squeeze(-1)
    sigma = torch.exp(logstd)
    act, adv, vo, ret = sl(buf["act"]), sl(buf["adv"]), sl(buf["val_old"]), sl(buf["ret"])
    nlp = 0.5 * (((act - mu) / sigma) ** 2).sum(-1) + math.log(2 * math.pi) + logstd.sum()
    ratio = torch.exp(sl(buf["nlp_old"]) - nlp)
    a_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - hyp["e_clip"], 1 + hyp["e_clip"])).mean()
    v_clip = vo + (v - vo).clamp(-hyp["e_clip"], hyp["e_clip"])
    c_loss = torch.max((v - ret) ** 2, (v_clip - ret) ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    (a_loss + 0.5 * c_loss * hyp["critic_coef"] + b_loss * hyp["bounds_loss_coef"]).backward()
    return [l.grad for l in leaves], dict(a_loss=a_loss.item(), c_loss=c_loss.item(), b_loss=b_loss.item()), mu.detach(), v.detach()


@pytest.mark.parametrize("T,N,e0,E,O", [(16, 256, 0, 128, 18), (8, 600, 100, 333, 28)])
def test_minibatch_raw_obs_matches_autograd(T, N, e0, E, O):
    """raw_obs with |obs| up to ~30 and NaN observation statistics (a read would poison every gradient): the gradients match
    fp32 autograd on the raw observations within 3e-2, the loss statistics within 2e-2 and mu / v within 1.5e-2 mean error
    relative to 1 + |output| (the bounds of test_fused_minibatch_gradients_match_autograd, the last made relative because the
    outputs reach ~15).  The loss scalars are built around the float64 forward so that every row stays MARGIN away from a
    branch boundary of the loss (test_gpu_mlp_update.mlp_problem); value_old and return are then moved up by 6, so the raw
    value targets lie beyond +5 and enter the loss as they are."""
    lib = abi.load_library()
    W, buf, _, _, logstd_old = make_problem(T, N, O, seed=T * N + O + 1)
    buf["obs"].mul_(4.0)
    fwd = forward_raw(W, rows_of(buf, "obs", e0, E).contiguous())
    head = fwd["h3"] @ fwd["wh"].t() + fwd["bh"]
    scal = loss_scalars(head[:, :2], head[:, 2], W[10], HYP["e_clip"], torch.Generator(device=DEV).manual_seed(T + O), MARGIN)
    scal[:, 5:7] += 6.0
    set_scalars(buf, scal, e0, E)
    assert float((buf["obs"].abs() > 5).double().mean()) > 0.1 and float((rows_of(buf, "ret", e0, E) > 5).double().mean()) > 0.5
    nan = torch.full((O,), float("nan"), device=DEV)
    flat, packed, state, out, dbg, n_part = run_kernel(lib, W, buf, nan, nan, logstd_old, e0, E, dict(HYP, raw_obs=1), O, T, N)
    grads, stats, mu, v = reference_raw(W, buf, logstd_old, e0, E, HYP)
    P = flat.numel()
    assert torch.isfinite(out).all()
    rel = lambda k, r: float(((k - r).abs() / (1 + r.abs())).mean())  # noqa: E731
    assert rel(dbg[:, :2], mu) < 1.5e-2 and rel(dbg[:, 2], v) < 1.5e-2, (rel(dbg[:, :2], mu), rel(dbg[:, 2], v))
    errs = {name: float((g - r).norm() / (r.norm() + 1e-12)) for name, g, r in zip(NAMES, split(out[:P], W), grads)}
    print("relative gradient errors:", {k: f"{e:.2e}" for k, e in errs.items()})
    assert max(errs.values()) < 3e-2, errs
    for j, k in ((0, "a_loss"), (1, "c_loss"), (3, "b_loss")):
        assert abs(float(out[P + j]) - stats[k]) <= 2e-2 * abs(stats[k]) + 1e-5, (k, float(out[P + j]), stats[k])


def test_ragged_recurrent_minibatch_raw_obs_matches_autograd():
    """The recurrent minibatch (S = 200 of R = 256 rows per step, O = 28) with raw observations up to ~30, NULL statistics
    and raw value targets beyond +-5, against fp32 autograd of ppo.ActorCritic on the raw observations (the x part of the
    LSTM input is raw too): 4e-2 per parameter tensor and 3e-2 on a_loss / c_loss, as in
    test_ragged_minibatch_o28_matches_autograd."""
    from test_gpu_lstm_any_shape import HYP as LHYP, native_problem, stage
    O, L, S = 28, 4, 200
    d = native_problem(O, L, S, 34)
    m = d["m"]
    d["obs"] = d["obs"] * 4.0
    assert float((d["obs"].abs() > 5).double().mean()) > 0.1
    with torch.no_grad():
        mu, _, v, _ = m(d["obs"], (d["h0"], d["c0"]), d["nd"])
    g = torch.Generator(device=DEV).manual_seed(35)
    d["scal"] = loss_scalars(mu.double(), v.double().squeeze(-1), m.sigma.detach(), LHYP["e_clip"], g, 0.05).view(L, S, 8)
    d["scal"][..., 5:7] += 6.0    # raw value targets (value_old, return) beyond +5, every row's value clipped by a wide margin
    path = NativeLstmPath(O, L, S, DEV, LHYP)
    obs, scal, nd = stage(path, d, slice(0, S))
    dbg = torch.zeros(L * path.R, 4, device=DEV)
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    path.gradients(d["packed"], d["lpacked"], obs, scal, nd, None, None, None, m.sigma.detach(), d["logstd_old"].clone(), state,
                   debug_out=dbg)
    torch.cuda.synchronize()
    gm, gl = path.flat_g_mlp.double().clone(), path.flat_g_lstm.double().clone()
    dbg = dbg.view(L, path.R, 4)[:, :S].reshape(L * S, 4)
    mu, _, v, _ = m(d["obs"], (d["h0"], d["c0"]), d["nd"])
    mu, v = mu.float(), v.float().squeeze(-1)
    sc = d["scal"].reshape(L * S, 8)
    act, nlpo, vo, ret, adv = sc[:, :2], sc[:, 4], sc[:, 5], sc[:, 6], sc[:, 7]
    nlp = 0.5 * (((act - mu) / torch.exp(m.sigma)) ** 2).sum(-1) + math.log(2 * math.pi) + m.sigma.sum()
    ratio = torch.exp(nlpo - nlp)
    a_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 0.8, 1.2)).mean()
    v_clip = vo + (v - vo).clamp(-0.2, 0.2)
    c_loss = torch.max((v - ret) ** 2, (v_clip - ret) ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    (a_loss + 0.5 * c_loss * 2.0 + b_loss * 1e-4).backward()
    assert float((dbg[:, :2] - mu.detach()).abs().mean()) < 2e-2 and float((dbg[:, 2] - v.detach()).abs().mean()) < 2e-2
    r = m.rnn.rnn
    errs, o = {}, 0
    for name, prm in (("W_ih", r.weight_ih_l0), ("W_hh", r.weight_hh_l0), ("b_ih", r.bias_ih_l0), ("b_hh", r.bias_hh_l0),
                      ("ln_g", m.layer_norm.weight), ("ln_b", m.layer_norm.bias), ("W_mu", m.mu.weight), ("b_mu", m.mu.bias),
                      ("W_v", m.value.weight), ("b_v", m.value.bias), ("logstd", m.sigma)):
        errs[name] = float((gl[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    o = 0
    for name, prm in (("W1", m.actor_mlp[0].weight), ("b1", m.actor_mlp[0].bias), ("W2", m.actor_mlp[2].weight),
                      ("b2", m.actor_mlp[2].bias), ("W3", m.actor_mlp[4].weight), ("b3", m.actor_mlp[4].bias)):
        errs[name] = float((gm[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    print({k: f"{e:.2e}" for k, e in errs.items()})
    P = gl.numel() - 4
    assert abs(float(gl[P]) - float(a_loss)) < 3e-2 * abs(float(a_loss)) + 1e-4
    assert abs(float(gl[P + 1]) - float(c_loss)) < 3e-2 * float(c_loss)
    assert max(errs.values()) < 4e-2, errs


# ----------------------------------------------------------------------------------------------------------- 4. the prologue
@pytest.mark.parametrize("raw_obs,raw_value", [(1, 0), (0, 1), (1, 1)])
def test_prologue_leaves_the_switched_off_statistics_alone(raw_obs, raw_value):
    """Two iterations at 16 x 4096 rows, values and returns up to ~30, against a launch with both normalisers on over the same
    data: the statistics of a normaliser that is off (f64 running statistics and their f32 copies, seeded with sentinels) keep
    their bits and its pointers may be NULL; with raw_value, values_n / returns_n are values / returns bit for bit.  The
    rest (the other normaliser, the advantages) equals the reference launch up to the order of the f64 atomics that sum the
    moments (1e-12 relative on the f64 statistics, 1e-6 on what is derived in f32); the moments end at zero."""
    lib = abi.load_library()
    O, count = 18, 16 * 4096
    g = torch.Generator(device=DEV).manual_seed(17 + 2 * raw_obs + raw_value)
    f = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731

    def buffers():
        b = dict(om=torch.full((O,), 0.25, dtype=torch.float64, device=DEV), ov=torch.full((O,), 3.0, dtype=torch.float64, device=DEV),
                 oc=torch.full((), 7.0, dtype=torch.float64, device=DEV), vm=torch.full((), 0.5, dtype=torch.float64, device=DEV),
                 vv=torch.full((), 2.0, dtype=torch.float64, device=DEV), vc=torch.full((), 9.0, dtype=torch.float64, device=DEV),
                 mf=torch.full((O,), -1.5, device=DEV), inv=torch.full((O,), 0.75, device=DEV), vs=torch.tensor([0.1, 0.2], device=DEV),
                 ast=f(2), vn=f(count), rn=f(count), an=f(count), mom=torch.zeros(2 * O + 4, dtype=torch.float64, device=DEV))
        return b

    def launch(b, obs, val, ret, ro, rv):
        P = lambda k: b[k].data_ptr()  # noqa: E731
        a = abi.VinePpoPrologue(obs=None if ro else obs.data_ptr(), values=val.data_ptr(), returns=ret.data_ptr(), moments=P("mom"),
                                obs_mean=None if ro else P("om"), obs_var=None if ro else P("ov"), obs_count=None if ro else P("oc"),
                                val_mean=None if rv else P("vm"), val_var=None if rv else P("vv"), val_count=None if rv else P("vc"),
                                obs_mean_f=None if ro else P("mf"), obs_inv_std_f=None if ro else P("inv"),
                                value_stats=None if rv else P("vs"), adv_stats=P("ast"), values_n=P("vn"), returns_n=P("rn"),
                                advantages_n=P("an"), count=count, num_obs=O, world=1, normalize_advantage=1, raw_obs=ro, raw_value=rv)
        assert lib.vine_ppo_moments(C.byref(a), None) == 0 and lib.vine_ppo_finalize(C.byref(a), None) == 0

    got, ref = buffers(), buffers()
    start = {k: v.clone() for k, v in got.items()}
    for _ in range(2):
        obs = torch.randn(count, O, device=DEV, generator=g) * 8.0
        val = torch.randn(count, device=DEV, generator=g) * 10.0
        ret = val + torch.randn(count, device=DEV, generator=g) * 4.0
        launch(got, obs, val, ret, raw_obs, raw_value)
        launch(ref, obs, val, ret, 0, 0)
        torch.cuda.synchronize()
        assert float(got["mom"].abs().max()) == 0.0
        same = lambda k: torch.equal(got[k].reshape(-1).view(torch.uint8), start[k].reshape(-1).view(torch.uint8))  # noqa: E731

        def close(k):
            x, y = got[k].double(), ref[k].double()
            rtol = 1e-12 if got[k].dtype == torch.float64 else 1e-6
            return bool(((x - y).abs() <= rtol * (1 + y.abs())).all())
        for k in ("om", "ov", "oc", "mf", "inv"):
            assert same(k) if raw_obs else close(k), k
        for k in ("vm", "vv", "vc", "vs"):
            assert same(k) if raw_value else close(k), k
        if raw_value:
            assert torch.equal(bits(got["vn"]), bits(val)) and torch.equal(bits(got["rn"]), bits(ret))
            assert float(got["rn"].abs().max()) > 5.0
        else:
            assert close("vn") and close("rn")
        assert close("an") and close("ast")


# ------------------------------------------------------------------------------------------------------------- 5. the agent
def agent(n, net, mode, extra=(), graphs=False, fused_update=True, seed=1):
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True"] + RAW[mode] + list(extra)
                       + (["train.params.network.rnn=null"] if net == "mlp" else []))
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=seed, use_graphs=graphs, use_fused_update=fused_update)


def params_of(a):
    m = a.model
    ps = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
          m.actor_mlp[4].bias]
    if m.has_rnn:
        r = m.rnn.rnn
        ps += [r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight, m.layer_norm.bias]
    ps += [m.mu.weight, m.mu.bias, m.value.weight, m.value.bias, m.sigma]
    return torch.cat([t.detach().reshape(-1) for t in ps]).clone()


@pytest.mark.parametrize("mode", ["input", "value", "both"])
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_kernel_update_moves_the_parameters_like_the_torch_update(net, mode):
    """FSTR, 1024 envs, minibatch_size 8192 (two minibatches), one mini-epoch, with the normaliser(s) off: the kernel-only
    update against torch autograd + torch Adam on the same rollout (cosine > 0.9 of the parameter steps, loss statistics
    within 5e-2, as in test_ragged_kernel_update_moves_the_parameters_like_the_torch_update).  A value bias of 6 puts the
    rollout's values beyond +-5 (with the value normaliser off they are not clamped).  The MLP baseline runs the kernel
    policy forward (agent.fused)."""
    one = ["train.params.config.mini_epochs=1", "train.params.config.minibatch_size=8192"]
    a = agent(1024, net, mode, one)
    b = agent(1024, net, mode, one, fused_update=False)
    assert a.fused_update and not b.fused_update and b.fused == (net == "mlp")
    with torch.no_grad():
        a.model.value.bias.fill_(6.0)
    a._refresh_fused(pack=True)
    b.load_state_dict(a.state_dict())
    if mode != "input":
        assert not any(k.startswith("value_mean_std.") for k in a.state_dict()["model"])
    if mode != "value":
        assert not any(k.startswith("running_mean_std.") for k in a.state_dict()["model"])
    start = params_of(a)
    a._rollout()
    torch.cuda.synchronize()
    if mode != "input":
        assert float(a.b_val.abs().max()) > 5.0 or float(a.b_ret.abs().max()) > 5.0
    names = ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "b_adv", "b_done")
    for name in names:
        getattr(b, name).copy_(getattr(a, name))
    if net == "lstm":
        for ck in range(a.T // a.seq_len):
            b.b_h[ck].copy_(from_tiles(a._HH_saved[ck], a.n))
            b.b_c[ck].copy_(a._C_saved[ck])
    a._update_any()
    b._update_any()
    torch.cuda.synchronize()
    da, db = params_of(a) - start, params_of(b) - start
    cos = float((da * db).sum() / (da.norm() * db.norm()))
    print(net, mode, "cos", cos)
    assert cos > 0.9, cos
    sa, sb = a.pop_stats(), b.pop_stats()
    for k in ("a_loss", "c_loss", "kl"):
        assert abs(sa[k] - sb[k]) <= 5e-2 * abs(sb[k]) + 2e-4, (k, sa[k], sb[k])
    if net == "mlp":   # the baseline's kernel forward reads what the torch update left: NULL statistics where a normaliser is off
        mu, _, v, _ = b._policy(b.obs)
        with torch.no_grad():
            ref = b.model(b.obs_rms(b.obs) if b.normalize_input else b.obs)
            vr = ref[2].squeeze(-1)
            vr = b.val_rms(vr, unnorm=True) if b.normalize_value else vr
        assert float((mu - ref[0]).abs().max()) < 5e-2 and float((v - vr).abs().max()) < 5e-2 * (1 + float(vr.abs().max()))


# ------------------------------------------------------------------------------------------------------- 6. graph replay
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_graph_replay_equals_eager_launches_with_both_normalisers_off(net):
    """n = 200 (two minibatches of 100 envs), both normalisers off: after the same number of training iterations, graph
    replay and eager launches leave bit-identical parameters and optimiser state."""
    extra = ["train.params.config.minibatch_size=1600"]
    g, e = agent(200, net, "both", extra, graphs=True), agent(200, net, "both", extra)
    for _ in range(2):
        g.train_epoch()
    for _ in range(g.epoch):
        e.train_epoch()
    torch.cuda.synchronize()
    assert g.epoch == e.epoch == 5
    assert torch.equal(g.flat, e.flat) and torch.equal(g.ppo_state, e.ppo_state)
    if net == "lstm":
        assert torch.equal(g.flat_l, e.flat_l)


# --------------------------------------------------------------------------------------------------- 7. train and play back
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_train_and_play_back_with_both_normalisers_off(net, tmp_path, monkeypatch):
    """``train.launch`` with both normalisers off trains a few iterations and writes a checkpoint without normaliser keys; the
    trainer plays it back (test=True), PolicyPlayer restores it as raw-observation policy, and an agent with the normalisers
    on refuses it."""
    from vine_robot_isaacgymenvs_b200 import train
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    monkeypatch.chdir(tmp_path)
    base = vcfg.FSTR_OVERRIDES + ["num_envs=128", "headless=True", "train.params.config.minibatch_size=1024"] + RAW["both"]
    base += ["train.params.network.rnn=null"] if net == "mlp" else []
    hist = train.launch(base + ["max_iterations=4"])
    assert len(hist) >= 1 and hist[-1]["epoch"] >= 4
    ck = tmp_path / "runs" / "Vine5LinkMovingBase" / "nn" / "Vine5LinkMovingBase.pth"
    sd = torch.load(ck, map_location=DEV)
    assert sd["model"] and not any(k.startswith(("running_mean_std.", "value_mean_std.")) for k in sd["model"])
    stats = train.launch(base + ["test=True", f"checkpoint={ck}", "play_steps=64"])
    assert stats["episodes"] > 0 and 0.0 <= stats["success_rate"] <= 1.0
    pl = PolicyPlayer(18, device=DEV).restore(str(ck))
    assert not pl.normalize_input
    on = agent(128, net, "value", ["train.params.config.minibatch_size=1024"])   # normalize_input on
    with pytest.raises(ValueError, match="running_mean_std"):
        on.load_state_dict(sd)
