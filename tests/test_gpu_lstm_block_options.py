"""GPU: kernel-only PPO with the rnn block's layer_norm and / or concat_input switched off (rl_games network.rnn; both default
to False in rl_games' A2CBuilder, so the short block ``{name: lstm, units: 256, layers: 1}`` has neither).

How the kernels take the switches:
  - layer_norm off: vine_lstm_head / vine_lstm_head_train with no_layer_norm act on y = h (no mean, rstd, gamma, beta); the
    training backward is dh = sum_j d_j w_j and the gamma / beta slots of every gradient partial are exactly 0;
  - concat_input off: vine_policy_act with u_no_obs writes U = [MLP output | 0 ... 0 | 1 | 0]: the observation columns are 0,
    the constant-1 column of the gate-bias gradient stays;
  - the flat parameter vector keeps its layout: the slots the torch block lacks (gamma / beta, the observation columns of W_ih)
    start at 0 and get a gradient of exactly 0, so Adam never moves them.
Tolerances are those of the tests each check follows, named there."""
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
from test_gpu_lstm_any_shape import run
from test_gpu_lstm_rollout import f32_ulp, fused_value
from test_gpu_lstm_update import SENT_BF16, SENT_F32, bf16_ulp, loss_scalars, make_params, pack, rel
from test_gpu_ppo_fused import make_problem, p

pytestmark = pytest.mark.gpu
DEV = "cuda"
TB = abi.LSTM_TILE_BYTES // 2
HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.0, bounds_loss_coef=1e-4)
HEAD_HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.01, bounds_loss_coef=0.05)
COMBOS = {"no_layer_norm": (True, False), "no_concat_input": (False, True), "neither": (False, False)}   # (concat_input, layer_norm)
SUMS = ("b_mu", "b_v", "logstd")   # gradients that are sums over the rows of terms of both signs


def bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def block(ci, ln):
    return {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": ci, "layer_norm": ln}


def combo_agent(n, ci, ln, extra=(), graphs=False, fused_update=True, seed=1):
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", f"train.params.network.rnn.concat_input={ci}",
                                              f"train.params.network.rnn.layer_norm={ln}"] + list(extra))
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=seed, use_graphs=graphs, use_fused_update=fused_update)


# ------------------------------------------------------------------------------------ 1. head kernels without LayerNorm
def head_reference_no_ln(Pd, hq, scal, logstd_old, hyp):
    """float64 heads on y = h -> the PPO loss of ppo.PPOAgent (test_gpu_lstm_update.head_reference without the LayerNorm)."""
    leaves = {k: Pd[k].clone().requires_grad_(True) for k in ("w_mu", "b_mu", "w_v", "b_v", "logstd")}
    hr = hq.clone().requires_grad_(True)
    mu = hr @ leaves["w_mu"].t() + leaves["b_mu"]
    v = (hr @ leaves["w_v"].t() + leaves["b_v"])[:, 0]
    ls = leaves["logstd"]
    act, muo, nlpo, vo, ret, adv = scal[:, :2], scal[:, 2:4], scal[:, 4], scal[:, 5], scal[:, 6], scal[:, 7]
    nlp = 0.5 * (((act - mu) / torch.exp(ls)) ** 2).sum(-1) + math.log(2 * math.pi) + ls.sum()
    ratio = torch.exp(nlpo - nlp)
    e = hyp["e_clip"]
    a_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - e, 1 + e)).mean()
    v_clip = vo + (v - vo).clamp(-e, e)
    c_loss = torch.max((v - ret) ** 2, (v_clip - ret) ** 2).mean()
    b_loss = (torch.clamp_min(mu - 1.1, 0) ** 2 + torch.clamp_max(mu + 1.1, 0) ** 2).sum(-1).mean()
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + ls).sum()
    loss = a_loss + 0.5 * hyp["critic_coef"] * c_loss - hyp["entropy_coef"] * entropy + hyp["bounds_loss_coef"] * b_loss
    loss.backward()
    so, s = torch.exp(logstd_old.double()), torch.exp(ls.detach())
    kl = (torch.log(so / s + 1e-5) + (s ** 2 + (muo - mu.detach()) ** 2) / (2 * (so ** 2 + 1e-5)) - 0.5).sum(-1).mean()
    stats = torch.stack([a_loss.detach(), c_loss.detach(), kl, b_loss.detach()])
    return mu.detach(), v.detach(), nlp.detach(), ratio.detach(), hr.grad, {k: t.grad for k, t in leaves.items()}, stats


def head_train(lib, lp, HH, scal, P, logstd_old, n, R, S):
    DH = torch.full_like(HH, SENT_BF16)
    gparts = torch.full((abi.LSTM_HEAD_GRAD_PARTS, abi.LSTM_HEAD_GRAD_FLOATS), SENT_F32, device=DEV)
    dbg = torch.full((n, 4), SENT_F32, device=DEV)
    ht = abi.VineLstmHeadTrain(params=lp.data_ptr(), hh=HH.data_ptr(), scalars=scal.data_ptr(), logstd=P["logstd"].data_ptr(),
                               logstd_old=logstd_old.data_ptr(), dh=DH.data_ptr(), grads=gparts.data_ptr(), debug_out=dbg.data_ptr(),
                               n=n, inv_B=1.0 / (n // R * S), step_rows=R if R != S else 0, step_seqs=S, no_layer_norm=1,
                               **HEAD_HYP)
    nparts = lib.vine_lstm_head_train(C.byref(ht), None)
    torch.cuda.synchronize()
    return nparts, DH, gparts, dbg


def rollout_head(lib, lp, HH, n, raw_value, no_ln, vstats, logstd, seed=0x5DEECE66D ^ 42, ctr=3):
    o = {k: torch.full(s, SENT_F32, device=DEV) for k, s in (("mu", (n, 2)), ("value", (n,)), ("actions", (n, 2)),
                                                             ("neglogp", (n,)), ("env_actions", (n, 2)))}
    counter = torch.tensor([ctr], dtype=torch.int32, device=DEV)
    hd = abi.VineLstmHead(params=lp.data_ptr(), hh=HH.data_ptr(), value_stats=None if raw_value else vstats.data_ptr(),
                          mu=o["mu"].data_ptr(), value=o["value"].data_ptr(), logstd=logstd.data_ptr(), rng_counter=counter.data_ptr(),
                          actions=o["actions"].data_ptr(), neglogp=o["neglogp"].data_ptr(), env_actions=o["env_actions"].data_ptr(),
                          n=n, seed=seed, global_env_offset=0, raw_value=raw_value, no_layer_norm=no_ln)
    assert lib.vine_lstm_head(C.byref(hd), None) == 0
    torch.cuda.synchronize()
    return o


@pytest.mark.parametrize("S", [8192, 8000], ids=["aligned", "padded"])
def test_head_kernels_without_layer_norm_match_float64(S):
    """The training minibatch shape, 4 steps x R = 8192 rows (S real sequences per step: all, or 8000 with 192 padded rows),
    above the 296-block clamp, every loss branch taken by a real fraction of rows, NaN in every padded row's h and scalars.
    vine_lstm_head_train with no_layer_norm against float64 heads on y = h (head_reference_no_ln) with the tolerances of
    test_lstm_head_train_matches_float64_above_the_block_clamp: mu, v within 2e-5 + 1e-5 |x|, neglogp 2e-5 (1 + |x|), dh one
    bf16 ulp + 1e-4 of the row's largest |dh| + 1e-5 of the median row's, the summed head / logstd gradients and loss
    statistics 1e-4 relative.  The LayerNorm slots of every partial are exactly 0, padded rows get dh = 0 and no debug row,
    and a second launch with zeros instead of NaN in the padded rows gives the same bits.
    vine_lstm_head (rollout) on the same tiles, raw_value 1 and 0: mu and the value head's v equal the training kernel's bit
    for bit (the hand-off claim: the same sums in the same order), the de-normalised value is fma(clamp(v), std, mean); its
    sampling draws the noise of the LayerNorm launch (same Philox key): neglogp the same bits, actions - mu the same within a
    few ulp, env_actions = clamp(actions)."""
    lib = abi.load_library()
    R, L = 8192, 4
    n = L * R
    g = torch.Generator(device=DEV).manual_seed(900 + S)
    P = make_params(18, 900 + S)
    h = torch.tanh(torch.randn(n, 256, device=DEV, generator=g) * 0.9 + 0.3 * torch.randn(n, 1, device=DEV, generator=g))
    real = torch.arange(n, device=DEV) % R < S
    HH_clean = to_tiles(h * real[:, None])
    hq = from_tiles(HH_clean, n).double()
    Pd = {k: P[k].double() for k in P}
    mu_r, v_r = hq @ Pd["w_mu"].t() + Pd["b_mu"], (hq @ Pd["w_v"].t() + Pd["b_v"])[:, 0]
    scal_clean = torch.zeros(n, 8, device=DEV)
    scal_clean[real] = loss_scalars(mu_r[real], v_r[real], P["logstd"], HEAD_HYP["e_clip"], g, 0.01)
    logstd_old = P["logstd"] + 0.05
    lp = pack(lib, dict(P, ln_g=torch.full_like(P["ln_g"], float("nan")), ln_b=torch.full_like(P["ln_b"], float("nan"))), 18)
    HH, scal = HH_clean.clone(), scal_clean.clone()
    if S < R:   # NaN in every padded row
        hn = from_tiles(HH, n)
        hn[~real] = float("nan")
        HH = to_tiles(hn)
        scal[~real] = float("nan")
    nparts, DH, gparts, dbg = head_train(lib, lp, HH, scal, P, logstd_old, n, R, S)
    assert nparts == 296
    mu, v, nlp, ratio, dh_ref, grads, stats = head_reference_no_ln(Pd, hq[real], scal_clean[real].double(), logstd_old, HEAD_HYP)
    e = HEAD_HYP["e_clip"]
    fr = {"ratio_low": float((ratio < 1 - e).double().mean()), "ratio_high": float((ratio > 1 + e).double().mean()),
          "value_clipped": float(((v - scal_clean[real][:, 5].double()).abs() > e).double().mean()),
          "mu_bound": float(((mu.abs() > 1.1).any(-1)).double().mean())}
    assert min(fr.values()) > 0.05, fr
    dr = dbg[real].double()
    assert bool(((dr[:, :2] - mu).abs() <= 2e-5 + 1e-5 * mu.abs()).all()), float((dr[:, :2] - mu).abs().max())
    assert bool(((dr[:, 2] - v).abs() <= 2e-5 + 1e-5 * v.abs()).all()), float((dr[:, 2] - v).abs().max())
    assert bool(((dr[:, 3] - nlp).abs() <= 2e-5 * (1 + nlp.abs())).all()), float((dr[:, 3] - nlp).abs().max())
    assert bool((dbg[~real] == SENT_F32).all())
    dh = from_tiles(DH, n).double()
    row_max = dh_ref.abs().amax(-1, keepdim=True)
    tol = bf16_ulp(dh_ref) + 1e-4 * row_max + 1e-5 * row_max.median()
    assert bool(((dh[real] - dh_ref).abs() <= tol).all()), float(((dh[real] - dh_ref).abs() - tol).max())
    assert bool((dh[~real] == 0).all())
    assert bool((gparts[:nparts, :512] == 0).all())                   # d(gamma), d(beta): exactly 0
    gs = gparts[:nparts].double().sum(0)
    errs = {"w_mu": rel(gs[512:1024], grads["w_mu"].reshape(-1)), "w_v": rel(gs[1024:1280], grads["w_v"].reshape(-1)),
            "b_mu": rel(gs[1280:1282], grads["b_mu"]), "b_v": rel(gs[1282:1283], grads["b_v"]), "logstd": rel(gs[1284:1286], grads["logstd"])}
    errs.update({k: abs(float(gs[1286 + j]) - float(stats[j])) / abs(float(stats[j])) for j, k in enumerate(["a_loss", "c_loss", "kl", "b_loss"])})
    print(S, fr, {k: f"{x:.1e}" for k, x in errs.items()})
    assert max(errs.values()) < 1e-4, errs
    if S < R:   # the padded rows' contents change no bit
        _, DH2, gparts2, dbg2 = head_train(lib, lp, HH_clean, scal_clean, P, logstd_old, n, R, S)
        assert torch.equal(bits(DH), bits(DH2)) and torch.equal(bits(gparts[:nparts]), bits(gparts2[:nparts]))
        assert torch.equal(bits(dbg), bits(dbg2))
    # the rollout kernel on the same tiles
    vstats = torch.tensor([0.4, 1.6], device=DEV)
    logstd = torch.tensor([-0.4, 0.1], device=DEV)
    lp_ln = pack(lib, P, 18)
    ref = rollout_head(lib, lp_ln, HH_clean, n, 0, 0, vstats, logstd)             # with LayerNorm: the same noise
    for raw_value in (1, 0):
        o = rollout_head(lib, lp, HH_clean, n, raw_value, 1, vstats, logstd)
        assert torch.equal(bits(o["mu"][real]), bits(dbg[real, :2]))
        want = dbg[real, 2] if raw_value else fused_value(dbg[real, 2], vstats)
        assert torch.equal(bits(o["value"][real]), bits(want)), raw_value
        assert torch.equal(bits(o["neglogp"]), bits(ref["neglogp"]))
        # a = fma(sigma, z, mu) rounds once: a - mu (exact in float64) is sigma z within half an ulp of a, in both launches
        d_new, d_ref = o["actions"].double() - o["mu"].double(), ref["actions"].double() - ref["mu"].double()
        bound = 0.5 * (f32_ulp(o["actions"].double()) + f32_ulp(ref["actions"].double()))
        assert bool(((d_new - d_ref).abs() <= bound).all()), float(((d_new - d_ref).abs() - bound).max())
        assert torch.equal(o["env_actions"], o["actions"].clamp(-1.0, 1.0))
    assert float((o["value"][real] - (v_r[real].float().clamp(-5, 5) * 1.6 + 0.4)).abs().max()) < 1e-3


# ------------------------------------------------------------------------- 2. vine_policy_act without the observation in U
@pytest.mark.parametrize("form", ["rollout", "minibatch"])
def test_policy_act_u_without_the_observation(form):
    """vine_policy_act with u_out, u_no_obs 1 against 0 on the same inputs (normalised observations, O = 18): the rollout form
    (n = 40 tiles + 45 rows, with the observation copy) and the minibatch form (4 steps of 256 rows, 200 real).  U's MLP
    columns 0..63 and the observation copy are the same bits; columns 64..94 are exactly 0, column 95 is what it was (1 on
    every real row, 0 on padded rows and rows past n), 96..127 are 0, and nothing is left unwritten.  u_no_obs without u_out is
    refused."""
    lib = abi.load_library()
    O = 18
    n = 40 * 128 + 45 if form == "rollout" else 4 * 256
    W, buf, mean, inv_std, _ = make_problem(1, n, O, seed=77 + n)
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_mlp_pack(*[p(w.contiguous()) for w in W[:10]], O, p(packed), None) == 0
    obs = buf["obs"][0].contiguous()
    vstats = torch.tensor([0.3, 1.7], device=DEV)
    tiles = (n + 127) // 128
    step = dict(u_step_rows=256, u_step_seqs=200) if form == "minibatch" else {}

    def launch(flag):
        U = torch.full((tiles, TB), float("nan"), dtype=torch.bfloat16, device=DEV)
        copy = torch.full((n, O), SENT_F32, device=DEV)
        a = abi.VinePolicyAct(packed=packed.data_ptr(), obs=obs.data_ptr(), obs_mean=mean.data_ptr(), obs_inv_std=inv_std.data_ptr(),
                              value_stats=vstats.data_ptr(), n=n, num_obs=O, u_out=U.data_ptr(), u_no_obs=flag,
                              obs_copy=copy.data_ptr() if form == "rollout" else None, **step)
        assert lib.vine_policy_act(C.byref(a), None) == 0
        torch.cuda.synchronize()
        return from_tiles(U.view(tiles, 1, TB), tiles * 128), copy

    u0, c0 = launch(0)
    u1, c1 = launch(1)
    valid = torch.arange(tiles * 128, device=DEV) < n
    if step:
        valid &= torch.arange(tiles * 128, device=DEV) % 256 < 200
    assert bool(torch.isfinite(u1).all()) and bool(torch.isfinite(u0).all())
    assert torch.equal(bits(u1[:, :64]), bits(u0[:, :64])) and torch.equal(bits(c1), bits(c0))
    assert float(u0[valid, 64:64 + O].abs().sum()) > 0                           # the flag-0 launch does carry x
    assert bool((u1[:, 64:95] == 0).all()) and bool((u1[:, 96:] == 0).all())
    assert torch.equal(bits(u1[:, 95]), bits(u0[:, 95]))
    assert bool((u1[valid, 95] == 1).all()) and bool((u1[~valid, 95] == 0).all())
    mu, val = torch.zeros(n, 2, device=DEV), torch.zeros(n, device=DEV)
    a = abi.VinePolicyAct(packed=packed.data_ptr(), obs=obs.data_ptr(), obs_mean=mean.data_ptr(), obs_inv_std=inv_std.data_ptr(),
                          value_stats=vstats.data_ptr(), n=n, num_obs=O, mu=mu.data_ptr(), value=val.data_ptr(), u_no_obs=1)
    assert lib.vine_policy_act(C.byref(a), None) == abi.ERR_INVALID_ARG


# ------------------------------------------------------------------------------------ 3. whole minibatch against autograd
def native_problem(O, L, S, seed, ci, ln):
    """test_gpu_lstm_any_shape.native_problem for the block (concat_input ci, layer_norm ln): a W_ih without observation
    columns is packed from its [1024, 64 + O] slot with zeros there, an absent LayerNorm from zero gamma / beta."""
    torch.manual_seed(seed)
    lib = abi.load_library()
    m = ActorCritic(O, 2, (256, 128, 64), rnn=block(ci, ln)).to(DEV)
    m.fused_cell = False
    with torch.no_grad():
        if ln:
            m.layer_norm.weight.uniform_(0.5, 1.5)
            m.layer_norm.bias.uniform_(-0.2, 0.2)
        m.mu.weight.mul_(3.0)
        m.value.weight.mul_(3.0)
        m.sigma.uniform_(-0.3, 0.1)
        for prm in m.parameters():
            if prm.dim() == 2 and prm.shape[0] > 3:
                prm.copy_(prm.bfloat16().float())
    z = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
           m.actor_mlp[4].bias, z(2, 64), z(2), z(1, 64), z(1)]
    keep = [t.detach().contiguous() for t in mlp]
    assert lib.vine_mlp_pack(*[p(t) for t in keep], O, p(packed), None) == 0
    r = m.rnn.rnn
    wih = r.weight_ih_l0 if ci else torch.cat([r.weight_ih_l0, z(1024, O)], 1)
    lnp = [m.layer_norm.weight, m.layer_norm.bias] if ln else [z(256), z(256)]
    lp = [t.detach().contiguous() for t in (wih, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, *lnp, m.mu.weight, m.mu.bias,
                                            m.value.weight, m.value.bias)]
    lpacked = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_lstm_pack(*[p(t) for t in lp], O, p(lpacked), None) == 0
    d = dict(m=m, packed=packed, lpacked=lpacked, obs=torch.randn(L, S, O, device=DEV) * 2, mean=torch.randn(O, device=DEV) * 0.3,
             inv_std=1.0 / (0.5 + torch.rand(O, device=DEV)), nd=(torch.rand(L, S, device=DEV) > 0.15).float(),
             h0=(torch.randn(S, 256, device=DEV) * 0.5).bfloat16().float(), c0=torch.randn(S, 256, device=DEV) * 0.5,
             logstd_old=torch.tensor([-0.1, 0.05], device=DEV))
    with torch.no_grad():
        mu, _, v, _ = m(torch.clamp((d["obs"] - d["mean"]) * d["inv_std"], -5, 5), (d["h0"], d["c0"]), d["nd"])
    g = torch.Generator(device=DEV).manual_seed(seed)
    d["scal"] = loss_scalars(mu.double(), v.double().squeeze(-1), m.sigma.detach(), HYP["e_clip"], g, 0.05).view(L, S, 8)
    return d


@pytest.mark.parametrize("S", [256, 200], ids=["aligned", "ragged"])
@pytest.mark.parametrize("combo", list(COMBOS) + ["reference"])
def test_minibatch_matches_autograd(combo, S):
    """One minibatch (L = 4, O = 18; S = 256 aligned, or 200 of R = 256 rows per step) of NativeLstmPath with the block's
    switches against fp32 autograd of ppo.ActorCritic built with that block: 4e-2 relative Frobenius error per weight tensor
    and 3e-2 on a_loss / c_loss (test_ragged_minibatch_o28_matches_autograd).  The head biases and the log-std are sums over
    the rows of terms of both signs that largely cancel, so their relative error is that of the kernel's bf16 rows (1e-2, more
    through a LayerNorm) over a small net sum: measured on a B200 up to 9.6e-2 (no_concat_input, aligned) and, for the
    reference block run here as the control, 9.0e-2 (ragged); bounded by 2e-1.  The head kernel's own sums are checked to
    1e-4 on its own operands (test 1, test_gpu_lstm_update.py).  The slots the block lacks get a gradient of exactly 0:
    W_ih's observation columns without concat_input, gamma / beta without layer_norm."""
    ci, ln = COMBOS.get(combo, (True, True))
    O, L = 18, 4
    d = native_problem(O, L, S, 40 + S + 2 * ci + ln, ci, ln)
    m = d["m"]
    path = NativeLstmPath(O, L, S, DEV, HYP, layer_norm=ln, concat_input=ci)
    dbg = torch.zeros(L * path.R, 4, device=DEV)
    gm, gl = run(path, d, slice(0, S), dbg=dbg)
    dbg = dbg.view(L, path.R, 4)[:, :S].reshape(L * S, 4)
    x = torch.clamp((d["obs"] - d["mean"]) * d["inv_std"], -5, 5)
    mu, _, v, _ = m(x, (d["h0"], d["c0"]), d["nd"])
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
    wih = gl[:1024 * (64 + O)].view(1024, 64 + O)
    if not ci:
        assert bool((wih[:, 64:] == 0).all())
    errs = {"W_ih": float((wih[:, :r.weight_ih_l0.shape[1]] - r.weight_ih_l0.grad.double()).norm() / r.weight_ih_l0.grad.double().norm())}
    o = wih.numel()
    for name, prm in (("W_hh", r.weight_hh_l0), ("b_ih", r.bias_ih_l0), ("b_hh", r.bias_hh_l0),
                      ("ln_g", m.layer_norm.weight if ln else None), ("ln_b", m.layer_norm.bias if ln else None), ("W_mu", m.mu.weight),
                      ("b_mu", m.mu.bias), ("W_v", m.value.weight), ("b_v", m.value.bias), ("logstd", m.sigma)):
        if prm is None:
            assert bool((gl[o:o + 256] == 0).all()), name
            o += 256
            continue
        errs[name] = float((gl[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    assert o == gl.numel() - 4
    o = 0
    for name, prm in (("W1", m.actor_mlp[0].weight), ("b1", m.actor_mlp[0].bias), ("W2", m.actor_mlp[2].weight),
                      ("b2", m.actor_mlp[2].bias), ("W3", m.actor_mlp[4].weight), ("b3", m.actor_mlp[4].bias)):
        errs[name] = float((gm[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    print(combo, S, {k: f"{e:.2e}" for k, e in errs.items()})
    P = gl.numel() - 4
    assert abs(float(gl[P]) - float(a_loss)) < 3e-2 * abs(float(a_loss)) + 1e-4
    assert abs(float(gl[P + 1]) - float(c_loss)) < 3e-2 * float(c_loss)
    assert max(e for k, e in errs.items() if k not in SUMS) < 4e-2, errs
    assert max(errs[k] for k in SUMS) < 2e-1, errs


# --------------------------------------------------------------------------------------- 4. rollout -> training hand-off
def nontrivial(agent):
    """A non-trivial LayerNorm (when the block has one), log-std and normaliser state."""
    g = torch.Generator(device=DEV).manual_seed(7)
    m = agent.model
    with torch.no_grad():
        if agent.layer_norm:
            m.layer_norm.weight.copy_(0.5 + torch.rand(256, device=DEV, generator=g))
            m.layer_norm.bias.copy_(0.1 * torch.randn(256, device=DEV, generator=g))
        m.value.weight.mul_(4.0)
        m.sigma.copy_(torch.tensor([-0.4, 0.1], device=DEV))
        agent.obs_rms.running_mean.copy_(0.2 * torch.randn(agent.O, device=DEV, generator=g).double())
        agent.obs_rms.running_var.copy_((0.3 + torch.rand(agent.O, device=DEV, generator=g)).double())
        agent.val_rms.running_mean.fill_(0.4)
        agent.val_rms.running_var.fill_(2.5)
    agent._refresh_fused(pack=True)


@pytest.mark.parametrize("combo", list(COMBOS))
def test_first_training_pass_reproduces_the_rollout(combo):
    """1024 envs (T = 16, seq_len 4, two minibatch slots of 512 envs), the second rollout of the agent: vine_lstm_gather +
    NativeLstmPath.gradients with the rollout-time statistics and no Adam step recompute the rollout's forward on the same
    operands in the same order, so debug_out mu == b_mu and fma(clamp(debug_out v), std, mean) == b_val bit for bit for
    every row (test_gpu_lstm_rollout.test_first_training_pass_reproduces_the_rollout, for the reference block)."""
    ci, ln = COMBOS[combo]
    agent = combo_agent(1024, ci, ln, ["train.params.config.minibatch_size=8192"])
    assert agent.native_lstm and agent.layer_norm is ln and agent.model.concat_input is ci
    nontrivial(agent)
    agent._rollout()
    agent._rollout()
    torch.cuda.synchronize()
    T, n, L, E, lib, path = agent.T, agent.n, agent.seq_len, agent.mb_envs, agent._lib, agent._path
    chunks = T // L
    assert E == 512 and path.R == chunks * E
    scal = torch.cat([agent.b_act, agent.b_mu, agent.b_nlp[..., None], agent.b_val[..., None], torch.zeros(T, n, 2, device=DEV)],
                     -1).contiguous()
    sigma = agent.model.sigma.detach().clone()
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    flat_before = agent.flat_l.clone()
    for e0 in range(0, n, E):
        ga = abi.VineLstmGather(obs=agent.b_obs.data_ptr(), scalars=scal.data_ptr(), not_done=agent._nd_ext.data_ptr(),
                                c_saved=agent._C_saved.data_ptr(), hh_saved=agent._HH_saved.data_ptr(),
                                mb_obs=agent._mb_obs.data_ptr(), mb_scalars=agent._mb_scal.data_ptr(),
                                mb_not_done=agent._mb_nd.data_ptr(), c0=path.C0.data_ptr(), hm0=path.HM[0].data_ptr(),
                                seq_len=L, chunks=chunks, num_envs=n, env_begin=e0, env_count=E, num_obs=agent.O, step_rows=path.R)
        assert lib.vine_lstm_gather(C.byref(ga), None) == 0
        dbg = torch.full((L * path.R, 4), SENT_F32, device=DEV)
        path.gradients(agent._packed, agent._lpacked, agent._mb_obs, agent._mb_scal, agent._mb_nd, agent._obs_mean_f,
                       agent._obs_inv_std_f, agent._val_stats, sigma, sigma.clone(), state, debug_out=dbg)
        torch.cuda.synchronize()

        def rows(buf):   # [T, N, ...] -> the minibatch's row order [step in chunk][chunk, env]
            return buf.view(chunks, L, n, -1)[:, :, e0:e0 + E].permute(1, 0, 2, 3).reshape(L * chunks * E, -1)
        differ = (bits(dbg[:, :2]) != bits(rows(agent.b_mu))).any(-1)
        assert not bool(differ.any()), (combo, e0, int(differ.sum()))
        assert torch.equal(bits(fused_value(dbg[:, 2], agent._val_stats)), bits(rows(agent.b_val)[:, 0])), (combo, e0)
    assert torch.equal(agent.flat_l, flat_before)


# ------------------------------------------------------------------------------------------------------- 5. dummy slots
def dummy_slots(agent):
    """(W_ih's observation columns, LayerNorm gamma / beta) of a [P_lstm] vector, each None where the block has them."""
    O = agent.O
    wih = 1024 * (64 + O)
    lng = wih + 1024 * 256 + 2 * 1024
    return (None if agent.model.concat_input else (lambda v: v[:wih].view(1024, 64 + O)[:, 64:]),
            None if agent.layer_norm else (lambda v: v[lng:lng + 512]))


@pytest.mark.parametrize("truncate", [False, True], ids=["unclipped", "truncate_grads"])
def test_dummy_slots_stay_zero(truncate):
    """Both switches off, 256 envs (two minibatches of 128 envs), 4 seeded training iterations with truncate_grads off and
    on: the observation columns of W_ih and gamma / beta in the flat vector, in both Adam moments and in the last minibatch's
    gradient are exactly 0, while the rest of the recurrent half moved."""
    extra = ["train.params.config.minibatch_size=2048"] + (["train.params.config.truncate_grads=True"] if truncate else [])
    agent = combo_agent(256, False, False, extra, seed=5)
    assert agent.truncate_grads is truncate
    before = agent.flat_l.clone()
    for _ in range(4):
        agent.train_epoch()
    torch.cuda.synchronize()
    for view in dummy_slots(agent):
        for vec in (agent.flat_l, agent.adam_ml, agent.adam_vl, agent._path.flat_g_lstm):
            assert bool((view(vec) == 0).all())
    moved = float((agent.flat_l - before).abs().sum())
    assert moved > 0
    assert agent.model.rnn.rnn.weight_ih_l0.data_ptr() == agent.flat_l.data_ptr()    # the torch weight is a view of the slot


# ------------------------------------------------------------------------------------- 6. kernel update vs torch update
def params_of(agent):
    return torch.cat([t.detach().reshape(-1) for t in agent.model.parameters()]).clone()


@pytest.mark.parametrize("combo", list(COMBOS))
def test_kernel_update_moves_the_parameters_like_the_torch_update(combo):
    """FSTR, 1024 envs, minibatch_size 8192 (two minibatches), one mini-epoch, with the block's switches: the kernel-only update
    against torch autograd + torch Adam on the same rollout (cosine > 0.9 of the parameter steps, loss statistics within
    5e-2, as in test_gpu_ppo_raw_normalisers.test_kernel_update_moves_the_parameters_like_the_torch_update).  The checkpoint
    carries the keys of rl_games' network for that block."""
    ci, ln = COMBOS[combo]
    one = ["train.params.config.mini_epochs=1", "train.params.config.minibatch_size=8192"]
    a = combo_agent(1024, ci, ln, one)
    b = combo_agent(1024, ci, ln, one, fused_update=False)
    assert a.native_lstm and not b.native_lstm
    sd = a.state_dict()
    assert ("a2c_network.layer_norm.weight" in sd["model"]) is ln
    assert tuple(sd["model"]["a2c_network.rnn.rnn.weight_ih_l0"].shape) == (1024, 64 + (a.O if ci else 0))
    b.load_state_dict(sd)
    start = params_of(a)
    assert torch.equal(start, params_of(b))
    a._rollout()
    torch.cuda.synchronize()
    for name in ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "b_adv", "b_done"):
        getattr(b, name).copy_(getattr(a, name))
    for ck in range(a.T // a.seq_len):
        b.b_h[ck].copy_(from_tiles(a._HH_saved[ck], a.n))
        b.b_c[ck].copy_(a._C_saved[ck])
    a._update_any()
    b._update_any()
    torch.cuda.synchronize()
    da, db = params_of(a) - start, params_of(b) - start
    cos = float((da * db).sum() / (da.norm() * db.norm()))
    print(combo, "cos", cos)
    assert cos > 0.9, cos
    sa, sb = a.pop_stats(), b.pop_stats()
    for k in ("a_loss", "c_loss", "kl"):
        assert abs(sa[k] - sb[k]) <= 5e-2 * abs(sb[k]) + 2e-4, (k, sa[k], sb[k])


def test_graph_replay_equals_eager_launches_with_both_switches_off():
    """n = 200 (two minibatches of 100 envs), both switches off: after the same number of training iterations, graph replay
    and eager launches leave bit-identical parameters and optimiser state."""
    extra = ["train.params.config.minibatch_size=1600"]
    g, e = combo_agent(200, False, False, extra, graphs=True), combo_agent(200, False, False, extra)
    for _ in range(2):
        g.train_epoch()
    for _ in range(g.epoch):
        e.train_epoch()
    torch.cuda.synchronize()
    assert g.epoch == e.epoch == 5
    assert torch.equal(g.flat, e.flat) and torch.equal(g.flat_l, e.flat_l) and torch.equal(g.ppo_state, e.ppo_state)
    assert torch.equal(g.adam_ml, e.adam_ml) and torch.equal(g.adam_vl, e.adam_vl)


# --------------------------------------------------------------------------------------------- 7. train and play back
def test_train_and_play_back_with_both_switches_off(tmp_path, monkeypatch):
    """``train.launch`` with concat_input and layer_norm off trains a few iterations and writes a checkpoint with rl_games'
    keys for that block (no layer_norm.*, weight_ih_l0 [1024, 64]); the trainer plays it back (test=True); PolicyPlayer(rnn=
    "auto") reads the block from the file, and its deterministic actions over three calls (LSTM state carried) equal those of
    the network of an agent that loaded the file."""
    from vine_robot_isaacgymenvs_b200 import train
    from vine_robot_isaacgymenvs_b200.player import PolicyPlayer
    monkeypatch.chdir(tmp_path)
    off = ["train.params.network.rnn.concat_input=False", "train.params.network.rnn.layer_norm=False"]
    base = vcfg.FSTR_OVERRIDES + ["num_envs=128", "headless=True", "train.params.config.minibatch_size=1024"] + off
    hist = train.launch(base + ["max_iterations=4"])
    assert len(hist) >= 1 and hist[-1]["epoch"] >= 4
    ck = tmp_path / "runs" / "Vine5LinkMovingBase" / "nn" / "Vine5LinkMovingBase.pth"
    sd = torch.load(ck, map_location=DEV)
    assert not any(k.startswith("a2c_network.layer_norm.") for k in sd["model"])
    assert tuple(sd["model"]["a2c_network.rnn.rnn.weight_ih_l0"].shape) == (1024, 64)
    stats = train.launch(base + ["test=True", f"checkpoint={ck}", "play_steps=64"])
    assert stats["episodes"] > 0 and 0.0 <= stats["success_rate"] <= 1.0
    pl = PolicyPlayer(18, device=DEV).restore(str(ck))
    pl.model.fused_cell = False   # both forwards in f32 torch (the fused cell runs its GEMMs in bf16)
    assert not pl.model.concat_input and not isinstance(pl.model.layer_norm, torch.nn.LayerNorm)
    agent = combo_agent(128, False, False, ["train.params.config.minibatch_size=1024"])
    agent.load_state_dict(sd)
    m = agent.model
    m.fused_cell = False
    g = torch.Generator(device=DEV).manual_seed(3)
    states = (torch.zeros(16, 256, device=DEV), torch.zeros(16, 256, device=DEV))
    with torch.no_grad():
        for step in range(3):
            obs = torch.randn(16, 18, device=DEV, generator=g) * 2
            mu, _, _, states = m(agent.obs_rms(obs), states)
            assert torch.allclose(pl.get_action(obs, is_deterministic=True), mu.clamp(-1.0, 1.0), atol=1e-5), step
