"""GPU: the kernel-only path of the reference network (MLP -> LSTM 256 -> LayerNorm) at shapes that are not multiples of the
128-row tile.  A minibatch of S sequences keeps its [step][sequence] row order with R = NativeLstmPath.step_rows(S) (S rounded
up to whole tiles) rows per step; rows [S, R) of every step are padded sequences that must add exactly nothing.

What holds, and why each check is exact or not:
  - every kernel on the rollout path is row-independent and the env and the Philox noise are keyed by the global env id, so a
    rollout at n envs equals the first n columns of the rollout at round_up(n, 128) envs bit for bit;
  - the loss is a mean over the real rows (inv_B = 1 / (L S)), so an aligned minibatch's gradient is (S1 g1 + S2 g2) / S of two
    ragged parts up to the order of the f32 sums (2e-5 of the gradient norm, 1e-5 on the loss statistics), and every row's
    mu (the update_mu_sigma write-back) is the same bits;
  - padded rows are written as zeros (dh, dG, dh_rec, dh3) and computed from finite stand-ins, so NaN in every padded row of
    the path's buffers and of the staged inputs changes no bit of the result."""
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

pytestmark = pytest.mark.gpu
DEV = "cuda"
RNN = {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": True, "layer_norm": True}
HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.0, bounds_loss_coef=1e-4)


def round_up(n):
    return -(-n // 128) * 128


def test_the_padding_rule():
    assert [NativeLstmPath.step_rows(s) for s in (1, 56, 128, 129, 200, 8000, 8192)] == [128, 128, 128, 256, 256, 8064, 8192]


# ------------------------------------------------------------------------------------------------------------- rollout
def fstr_agent(n, extra=(), graphs=False, seed=1):
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True"] + list(extra))
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=seed, use_graphs=graphs)


def nontrivial(agent, src=None):
    """A non-trivial LayerNorm, log-std and normaliser state (the same on every agent of a test), or ``src``'s."""
    m = agent.model
    g = torch.Generator(device=DEV).manual_seed(7)
    with torch.no_grad():
        if src is not None:
            for a, b in zip(m.parameters(), src.model.parameters()):
                a.copy_(b)
            agent.obs_rms.running_mean.copy_(src.obs_rms.running_mean)
            agent.obs_rms.running_var.copy_(src.obs_rms.running_var)
        else:
            m.layer_norm.weight.copy_(0.5 + torch.rand(256, device=DEV, generator=g))
            m.layer_norm.bias.copy_(0.1 * torch.randn(256, device=DEV, generator=g))
            m.value.weight.mul_(4.0)
            m.sigma.copy_(torch.tensor([-0.4, 0.1], device=DEV))
            agent.obs_rms.running_mean.copy_(0.2 * torch.randn(agent.O, device=DEV, generator=g).double())
            agent.obs_rms.running_var.copy_((0.3 + torch.rand(agent.O, device=DEV, generator=g)).double())
        agent.val_rms.running_mean.fill_(0.4)
        agent.val_rms.running_var.fill_(2.5)
    agent._refresh_fused(pack=True)


@pytest.mark.parametrize("n", [64, 200, 1000])
def test_ragged_rollout_is_the_aligned_rollout_column_for_column(n):
    """FSTR, same seed, parameters and normaliser state: the rollout at n envs against the first n env columns of the rollout
    at round_up(n, 128) envs, bit for bit, over two consecutive rollouts: every buffer the update reads, the chunk-start LSTM
    state it restarts from and the persistent state the next rollout continues from."""
    ragged, aligned = fstr_agent(n), fstr_agent(round_up(n))
    assert ragged.native_lstm and aligned.native_lstm
    nontrivial(aligned)
    nontrivial(ragged, aligned)
    for it in range(2):
        ragged._rollout()
        aligned._rollout()
        torch.cuda.synchronize()
        for name in ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_rew", "b_done"):
            a, b = getattr(ragged, name), getattr(aligned, name)[:, :n]
            assert torch.equal(a, b), (it, name, float((a - b).abs().max()))
        assert torch.equal(ragged.last_value, aligned.last_value[:n]), it
        for ck in range(ragged.T // ragged.seq_len):
            assert torch.equal(from_tiles(ragged._HH_saved[ck], n), from_tiles(aligned._HH_saved[ck], n)), (it, ck)
            assert torch.equal(ragged._C_saved[ck], aligned._C_saved[ck][:n]), (it, ck)
        assert torch.equal(from_tiles(ragged._r_HH[0], n), from_tiles(aligned._r_HH[0], n)), it
        assert torch.equal(ragged._r_C[0], aligned._r_C[0][:n]), it
    assert float(ragged.b_done.sum()) > 0          # episodes ended inside the window: the masks were exercised


def test_gather_pads_every_step_with_neutral_sequences():
    """vine_lstm_gather at 200 envs, a 100-env minibatch slot starting at env 100 (no alignment anywhere): the real rows are
    the rollout's rows, and every padded sequence gets zero observations, scalars, not_done, c0 and hm0 -- over outputs
    that held NaN before the launch."""
    agent = fstr_agent(200, ["train.params.config.minibatch_size=1600"])
    nontrivial(agent)
    agent._rollout()
    agent._rollout()
    T, L, n, E = agent.T, agent.seq_len, agent.n, agent.mb_envs
    chunks, path = T // L, agent._path
    S, R = chunks * E, path.R
    assert (E, S, R) == (100, 400, 512)
    agent._scal.copy_(torch.randn_like(agent._scal))
    for t in (agent._mb_obs, agent._mb_scal, agent._mb_nd, path.C0, path.HM[0]):
        t.fill_(float("nan"))
    e0 = 100
    ga = abi.VineLstmGather(obs=agent.b_obs.data_ptr(), scalars=agent._scal.data_ptr(), not_done=agent._nd_ext.data_ptr(),
                            c_saved=agent._C_saved.data_ptr(), hh_saved=agent._HH_saved.data_ptr(), mb_obs=agent._mb_obs.data_ptr(),
                            mb_scalars=agent._mb_scal.data_ptr(), mb_not_done=agent._mb_nd.data_ptr(), c0=path.C0.data_ptr(),
                            hm0=path.HM[0].data_ptr(), seq_len=L, chunks=chunks, num_envs=n, env_begin=e0, env_count=E,
                            num_obs=agent.O, step_rows=R)
    assert agent._lib.vine_lstm_gather(C.byref(ga), None) == 0
    torch.cuda.synchronize()
    src = lambda x: x.view(chunks, L, n, *x.shape[2:])[:, :, e0:e0 + E].transpose(0, 1).reshape(L, S, *x.shape[2:])  # noqa: E731
    assert torch.equal(agent._mb_obs[:, :S], src(agent.b_obs)) and torch.equal(agent._mb_scal[:, :S], src(agent._scal))
    assert torch.equal(agent._mb_nd[:, :S], src(agent._nd_ext[:T]))
    assert torch.equal(path.C0[:S], agent._C_saved[:, e0:e0 + E].reshape(S, 256))
    nd0 = agent._nd_ext[:T].view(chunks, L, n)[:, 0, e0:e0 + E].reshape(S, 1)
    h0 = torch.stack([from_tiles(agent._HH_saved[ck], n)[e0:e0 + E] for ck in range(chunks)]).reshape(S, 256)
    assert torch.equal(from_tiles(path.HM[0], S), (h0 * nd0).bfloat16().float())
    for t in (agent._mb_obs[:, S:], agent._mb_scal[:, S:], agent._mb_nd[:, S:], path.C0[S:], from_tiles(path.HM[0], R)[S:]):
        assert bool((t == 0).all())


# ----------------------------------------------------------------------------------------------------------- minibatch
def native_problem(O, L, S, seed):
    """Network (bf16-representable weights), packed operands, inputs and loss scalars of one minibatch of S sequences; the
    scalars keep every row 0.05 away from a branch boundary of the loss (as in test_gpu_lstm_update.py)."""
    from test_gpu_lstm_update import loss_scalars
    torch.manual_seed(seed)
    lib = abi.load_library()
    m = ActorCritic(O, 2, (256, 128, 64), rnn=RNN).to(DEV)
    m.fused_cell = False
    with torch.no_grad():
        m.layer_norm.weight.uniform_(0.5, 1.5); m.layer_norm.bias.uniform_(-0.2, 0.2)
        m.mu.weight.mul_(3.0); m.value.weight.mul_(3.0); m.sigma.uniform_(-0.3, 0.1)
        for prm in m.parameters():
            if prm.dim() == 2 and prm.shape[0] > 3:
                prm.copy_(prm.bfloat16().float())
    z = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
           m.actor_mlp[4].bias, z(2, 64), z(2), z(1, 64), z(1)]
    keep = [t.detach().contiguous() for t in mlp]
    assert lib.vine_mlp_pack(*[C.c_void_p(t.data_ptr()) for t in keep], O, C.c_void_p(packed.data_ptr()), None) == 0
    r = m.rnn.rnn
    lp = [t.detach().contiguous() for t in (r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight,
                                            m.layer_norm.bias, m.mu.weight, m.mu.bias, m.value.weight, m.value.bias)]
    lpacked = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_lstm_pack(*[C.c_void_p(t.data_ptr()) for t in lp], O, C.c_void_p(lpacked.data_ptr()), None) == 0
    d = dict(m=m, packed=packed, lpacked=lpacked, obs=torch.randn(L, S, O, device=DEV) * 2, mean=torch.randn(O, device=DEV) * 0.3,
             inv_std=1.0 / (0.5 + torch.rand(O, device=DEV)), nd=(torch.rand(L, S, device=DEV) > 0.15).float(),
             h0=(torch.randn(S, 256, device=DEV) * 0.5).bfloat16().float(), c0=torch.randn(S, 256, device=DEV) * 0.5,
             logstd_old=torch.tensor([-0.1, 0.05], device=DEV))
    with torch.no_grad():
        mu, _, v, _ = m(torch.clamp((d["obs"] - d["mean"]) * d["inv_std"], -5, 5), (d["h0"], d["c0"]), d["nd"])
    g = torch.Generator(device=DEV).manual_seed(seed)
    d["scal"] = loss_scalars(mu.double(), v.double().squeeze(-1), m.sigma.detach(), HYP["e_clip"], g, 0.05).view(L, S, 8)
    return d


def stage(path, d, sl):
    """The inputs of envs ``sl`` in the padded layout the gather writes: [L, R, ...] with zero padded rows."""
    L, S, R = path.L, path.S, path.R
    z = lambda *s: torch.zeros(L, R, *s, device=DEV)  # noqa: E731
    obs, scal, nd = z(d["obs"].shape[-1]), z(8), z()
    obs[:, :S], scal[:, :S], nd[:, :S] = d["obs"][:, sl], d["scal"][:, sl], d["nd"][:, sl]
    hm0 = torch.zeros(R, 256, device=DEV)
    hm0[:S] = d["h0"][sl] * nd[0, :S, None]
    path.HM[0].copy_(to_tiles(hm0))
    path.C0.zero_()
    path.C0[:S] = d["c0"][sl]
    return obs, scal, nd


def run(path, d, sl, staged=None, dbg=None, wb=None):
    """gradients() of envs ``sl``; ``wb`` = the [L, N, 8] scalars the mu write-back goes to (chunks = 1, env_begin = sl.start)."""
    obs, scal, nd = staged if staged is not None else stage(path, d, sl)
    vstats, state = torch.tensor([0.0, 1.0], device=DEV), torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    writeback = None if wb is None else (wb, path.L, 1, wb.shape[1], sl.start, path.S)
    path.gradients(d["packed"], d["lpacked"], obs, scal, nd, d["mean"], d["inv_std"], vstats, d["m"].sigma.detach(),
                   d["logstd_old"].clone(), state, debug_out=dbg, writeback=writeback)
    torch.cuda.synchronize()
    return path.flat_g_mlp.double().clone(), path.flat_g_lstm.double().clone()


@pytest.mark.parametrize("S,S1", [(256, 200), (8192, 8000), (400, 200), (8000, 4000)])
def test_minibatch_is_the_weighted_sum_of_its_ragged_parts(S, S1):
    """A minibatch of S sequences (aligned: 256, 8192; ragged: 400, 8000) against its parts [0, S1) and [S1, S) (all
    ragged): the mu write-back of the two parts equals the whole's row for row, bit for bit (every row's forward is the
    same arithmetic), the loss statistics agree within 1e-5 and the gradient is (S1 g1 + S2 g2) / S.  The gradient tolerance
    depends on the split: dh leaves the head kernel as bf16 already weighted by 1 / (L S), and bf16 rounding commutes with
    that weight only when the part's and the whole's differ by a power of two.  Equal halves (S = 2 S1) therefore agree up to
    the order of the f32 sums, 2e-5 of the gradient norm per network as in
    test_native_lstm_minibatch_at_the_training_size_is_the_mean_of_its_halves; other splits round every row's dh and dG
    differently (at most 2^-9 relative each), measured on a B200 as 4.3e-3 (S = 256) and 1.1e-3 (S = 8192): 1e-2."""
    O, L, S2 = 18, 4, S - S1
    tol = 2e-5 if S == 2 * S1 else 1e-2
    d = native_problem(O, L, S, 31)
    wb_whole, wb_parts = d["scal"].clone(), d["scal"].clone()
    whole = run(NativeLstmPath(O, L, S, DEV, HYP), d, slice(0, S), wb=wb_whole)
    a = run(NativeLstmPath(O, L, S1, DEV, HYP), d, slice(0, S1), wb=wb_parts)
    b = run(NativeLstmPath(O, L, S2, DEV, HYP), d, slice(S1, S), wb=wb_parts)
    for k, (w, ga, gb) in enumerate(zip(whole, a, b)):
        Pn = w.numel() - 4
        h = (S1 * ga + S2 * gb) / S
        assert float(w[:Pn].norm()) > 1e-3
        e = float((w[:Pn] - h[:Pn]).norm() / w[:Pn].norm())
        print(("mlp", "lstm")[k], f"{e:.2e}")
        assert e < tol, (k, e)
        for j in range(4):
            assert abs(float(w[Pn + j]) - float(h[Pn + j])) <= 1e-5 * max(abs(float(w[Pn + j])), 1e-3), (k, j, float(w[Pn + j]), float(h[Pn + j]))
    assert not torch.equal(wb_whole, d["scal"])
    assert torch.equal(wb_whole.view(torch.int32), wb_parts.view(torch.int32))


def test_ragged_minibatch_o28_matches_autograd():
    """One ragged minibatch (S = 200: R = 256, 56 padded rows per step) of the 28-wide network against fp32 autograd of
    ppo.ActorCritic: 4e-2 relative Frobenius error per parameter tensor, the bound of
    test_native_lstm_minibatch_o28_matches_autograd_at_the_training_size."""
    O, L, S = 28, 4, 200
    d = native_problem(O, L, S, 32)
    m = d["m"]
    path = NativeLstmPath(O, L, S, DEV, HYP)
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
    errs, o = {}, 0
    for name, prm in (("W_ih", r.weight_ih_l0), ("W_hh", r.weight_hh_l0), ("b_ih", r.bias_ih_l0), ("b_hh", r.bias_hh_l0),
                      ("ln_g", m.layer_norm.weight), ("ln_b", m.layer_norm.bias), ("W_mu", m.mu.weight), ("b_mu", m.mu.bias),
                      ("W_v", m.value.weight), ("b_v", m.value.bias), ("logstd", m.sigma)):
        errs[name] = float((gl[o:o + prm.numel()].view_as(prm) - prm.grad.double()).norm() / prm.grad.double().norm())
        o += prm.numel()
    assert o == gl.numel() - 4
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


def poison_padded_rows(path, staged):
    """NaN in every padded row of the path's activation tiles, cell arrays, dh3 and of the staged inputs.  HM[0] is the
    gather's output (its padded rows are zero by its contract, test_gather_pads_every_step_with_neutral_sequences)."""
    S, R, nan = path.S, path.R, float("nan")

    def tiles(buf, width=128):
        for t in range(buf.shape[0]):
            b = buf[t].view(path.tiles, -1, 128 * width)
            x = from_tiles(b, R, width)
            x[S:] = nan
            b.copy_(to_tiles(x, width))
    tiles(path.U)
    tiles(path.HM[1:])
    for buf in (path.HH, path.DH, path.DHREC):
        tiles(buf)
    for buf in (path.ACT, path.DG):
        tiles(buf, 64)
    for buf in (path.Cs, path.DH3) + tuple(staged):
        buf[:, S:] = nan
    for buf in [path.C0] + path.DC:
        buf[S:] = nan


def test_padded_rows_are_neutral():
    """A ragged minibatch (S = 200 of N = 256 envs) twice: once as is, once with NaN in every padded row of the path's
    buffers and of its staged inputs.  Gradients, loss statistics and the mu write-back are bit-identical, and the
    write-back leaves the other envs' rows of the [T, N, 8] scalars untouched."""
    O, L, N, S = 18, 4, 256, 200
    d = native_problem(O, L, N, 33)
    path = NativeLstmPath(O, L, S, DEV, HYP)
    wb0, wb1 = d["scal"].clone(), d["scal"].clone()
    clean = run(path, d, slice(0, S), wb=wb0)
    staged = stage(path, d, slice(0, S))
    poison_padded_rows(path, staged)
    dirty = run(path, d, slice(0, S), staged=staged, wb=wb1)
    for k, (a, b) in enumerate(zip(clean, dirty)):
        assert torch.equal(a.float().view(torch.int32), b.float().view(torch.int32)), k
        assert bool(torch.isfinite(a).all())
    assert torch.equal(wb0.view(torch.int32), wb1.view(torch.int32))
    assert torch.equal(wb1[:, S:], d["scal"][:, S:]) and not torch.equal(wb1[:, :S], d["scal"][:, :S])


# ---------------------------------------------------------------------------------------------------------- the agent
def test_ragged_kernel_update_moves_the_parameters_like_the_torch_update():
    """num_envs = 1000, minibatch_size = 4000 (250 envs per minibatch: 4 ragged minibatches of 1000 sequences), one mini-epoch:
    the kernel-only update against torch autograd + torch Adam on the same rollout, with the criteria of
    test_native_lstm_update_moves_the_parameters_like_the_torch_update."""
    one = ["train.params.config.mini_epochs=1", "train.params.config.minibatch_size=4000"]
    a = fstr_agent(1000, one)
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + ["num_envs=1000", "headless=True"] + one)
    b = PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=1, use_graphs=False, use_fused_update=False)
    assert a.native_lstm and not b.native_lstm and a.mb_envs == 250
    b.load_state_dict(a.state_dict())
    start = torch.cat([a.flat[:a.flat.numel() - 197].clone(), a.flat_l.clone()])
    a._rollout()
    for name in ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "b_adv", "b_done"):
        getattr(b, name).copy_(getattr(a, name))
    for ck in range(a.T // a.seq_len):
        b.b_h[ck].copy_(from_tiles(a._HH_saved[ck], a.n))
        b.b_c[ck].copy_(a._C_saved[ck])
    a._update_any()
    b._update_any()
    torch.cuda.synchronize()
    mb = [b.model.actor_mlp[0].weight, b.model.actor_mlp[0].bias, b.model.actor_mlp[2].weight, b.model.actor_mlp[2].bias,
          b.model.actor_mlp[4].weight, b.model.actor_mlp[4].bias]
    rb = b.model.rnn.rnn
    lb = [rb.weight_ih_l0, rb.weight_hh_l0, rb.bias_ih_l0, rb.bias_hh_l0, b.model.layer_norm.weight, b.model.layer_norm.bias,
          b.model.mu.weight, b.model.mu.bias, b.model.value.weight, b.model.value.bias, b.model.sigma]
    after_b = torch.cat([p.detach().reshape(-1) for p in mb + lb])
    after_a = torch.cat([a.flat[:a.flat.numel() - 197], a.flat_l])
    da, db = after_a - start, after_b - start
    cos = float((da * db).sum() / (da.norm() * db.norm()))
    print("cos", cos)
    assert cos > 0.9, cos
    sa, sb = a.pop_stats(), b.pop_stats()
    for k in ("a_loss", "c_loss", "kl"):
        assert abs(sa[k] - sb[k]) <= 5e-2 * abs(sb[k]) + 2e-4, (k, sa[k], sb[k])


def test_ragged_graph_replay_equals_eager_launches():
    """n = 200 (2 minibatches of 100 envs): after the same number of training iterations, graph replay and eager launches
    leave bit-identical parameters (the graph agent's first train_epoch runs three eager warm-up iterations)."""
    extra = ["train.params.config.minibatch_size=1600"]
    g, e = fstr_agent(200, extra, graphs=True), fstr_agent(200, extra)
    for _ in range(2):
        g.train_epoch()
    for _ in range(g.epoch):
        e.train_epoch()
    torch.cuda.synchronize()
    assert g.epoch == e.epoch == 5
    assert torch.equal(g.flat, e.flat) and torch.equal(g.flat_l, e.flat_l)
    assert torch.equal(g.ppo_state, e.ppo_state)


def test_train_entry_point_at_100_envs(tmp_path, monkeypatch):
    """``train.launch`` with num_envs = 100 on the kernel-only path: trains a few iterations, saves the checkpoint and plays
    it back (test=True)."""
    from vine_robot_isaacgymenvs_b200 import train
    monkeypatch.chdir(tmp_path)
    base = vcfg.FSTR_OVERRIDES + ["num_envs=100", "headless=True", "train.params.config.minibatch_size=800"]
    hist = train.launch(base + ["max_iterations=4"])
    assert len(hist) >= 1 and hist[-1]["epoch"] >= 4 and hist[-1]["frames"] > 0
    ck = tmp_path / "runs" / "Vine5LinkMovingBase" / "nn" / "Vine5LinkMovingBase.pth"
    assert ck.exists()
    stats = train.launch(base + ["test=True", f"checkpoint={ck}", "play_steps=64"])
    assert stats["episodes"] > 0 and 0.0 <= stats["success_rate"] <= 1.0


def test_fstr_training_at_4000_envs_reaches_the_success_band():
    """Learning at a ragged size: FSTR, 4000 envs, minibatch_size 32000 (2000 envs = 8000 sequences per minibatch, two
    minibatches per mini-epoch like the default), 250 iterations, the band of test_fstr_training_reaches_the_success_band."""
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + ["num_envs=4000", "headless=True", "train.params.config.minibatch_size=32000"])
    agent = PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=42, use_graphs=True)
    assert agent.native_lstm and agent.mb_envs == 2000 and agent._path.R == 8064
    hist = agent.train(250, log_every=50, log=None)
    last = hist[-1]
    print(last)
    assert last["success_rate"] >= 0.72 and last["mean_length"] < 60 and last["mean_return"] > 600, last
    assert hist[0]["success_rate"] < last["success_rate"]
