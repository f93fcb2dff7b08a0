"""GPU: the update kernels of the recurrent network (ppo/lstm_native.py) one by one at the training minibatch shape --
L = 4 steps x S = 8192 sequences = 32768 rows, 64 row tiles per step and 256 per minibatch -- where several of them take a
different code path than at the sizes of test_gpu_lstm_net.py (<= 16 tiles): the y = 2 grid of vine_lstm_step, the clamped
grid of vine_lstm_head_train, wgrad K splits with many (or no) tiles, the MLP backward with several tiles per CTA.

The references are float64 computations that start from the kernels' own bf16 operands (the U / HM / HH / ACT / DG tiles
decoded with ppo.tiles.from_tiles, the weights rounded to bf16 as vine_lstm_pack rounds them), so that only f32 accumulation
order and tanh.approx separate kernel and reference; each test derives its tolerance from those two in its docstring.
tanh.approx.f32 has a relative error below 2^-10.987 < 5e-4 (PTX ISA); the sigmoid 0.5 tanh(x/2) + 0.5 inherits half of it
as an absolute error."""
import ctypes as C
import math

import pytest
import torch

from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic
from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles, to_tiles

pytestmark = pytest.mark.gpu
DEV = "cuda"
TB = abi.LSTM_TILE_BYTES // 2      # bf16 elements of one [128 x 128] tile
AB = 128 * 64                      # bf16 elements of one [128 x 64] gate tile
E_TANH = 5e-4                      # relative error bound of tanh.approx.f32
NAMES = ["w_ih", "w_hh", "b_ih", "b_hh", "ln_g", "ln_b", "w_mu", "b_mu", "w_v", "b_v", "logstd"]
# byte ranges of the packed block (csrc/vine_lstm_net.cu LP_*)
PACKED_REGIONS = {"W_ih": (0, 262144), "W_hh": (262144, 786432), "bias": (786432, 790528), "ln_gamma": (790528, 791552),
                  "ln_beta": (791552, 792576), "head_w": (792576, 795648), "head_b": (795648, 795664)}
RNN = {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": True, "layer_norm": True}


def p(t):
    return C.c_void_p(t.data_ptr())


def gate_perm():
    """packed gate row R -> torch gate row (piece p row g*16+k = gate g of hidden unit 16p+k)."""
    R = torch.arange(1024)
    return ((R % 64) // 16) * 256 + 16 * (R // 64) + (R % 16)


def to_torch_gates(x_packed):
    """[n, 1024] columns in packed gate order -> torch gate order (i, f, g, o blocks of 256)."""
    out = torch.empty_like(x_packed)
    out[:, gate_perm().to(x_packed.device)] = x_packed
    return out


def bf16_ulp(x):
    """one bf16 ulp at |x| (float64 tensor); 0 where x == 0."""
    e = torch.frexp(x.abs())[1]
    return torch.where(x == 0, torch.zeros_like(x), torch.ldexp(torch.ones_like(x), e - 8))


def rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def make_params(O, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    r = lambda *s, k=1.0: torch.randn(*s, device=DEV, generator=g) * k  # noqa: E731
    return dict(w_ih=r(1024, 64 + O, k=0.1), w_hh=r(1024, 256, k=0.06), b_ih=r(1024, k=0.2), b_hh=r(1024, k=0.2),
                ln_g=0.5 + torch.rand(256, device=DEV, generator=g), ln_b=r(256, k=0.1), w_mu=r(2, 256, k=0.08),
                b_mu=r(2, k=0.1), w_v=r(1, 256, k=0.08), b_v=r(1, k=0.1), logstd=r(2, k=0.2))


def flat_of(P):
    return torch.cat([P[k].reshape(-1) for k in NAMES]).contiguous()


def unflat(flat, O):
    shapes = dict(w_ih=(1024, 64 + O), w_hh=(1024, 256), b_ih=(1024,), b_hh=(1024,), ln_g=(256,), ln_b=(256,), w_mu=(2, 256),
                  b_mu=(2,), w_v=(1, 256), b_v=(1,), logstd=(2,))
    out, o = {}, 0
    for k in NAMES:
        n = math.prod(shapes[k])
        out[k] = flat[o:o + n].view(shapes[k])
        o += n
    return out


def pack(lib, P, O):
    packed = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_lstm_pack(*[p(P[k].contiguous()) for k in NAMES[:10]], O, p(packed), None) == 0
    return packed


def packed_diff(a, b):
    """region -> number of differing bytes (for assertion messages)."""
    d = (a != b)
    return {k: int(d[lo:hi].sum()) for k, (lo, hi) in PACKED_REGIONS.items() if bool(d[lo:hi].any())}


# ---------------------------------------------------------------------------------------------------------------- 1. step
def step_inputs(n, O, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    tiles = (n + 127) // 128
    u = torch.zeros(n, 128, device=DEV)
    u[:, :64 + O] = torch.randn(n, 64 + O, device=DEV, generator=g)
    u[:, 95] = 1.0
    nd = (torch.rand(n, device=DEV, generator=g) > 0.2).float()
    h = (torch.rand(n, 256, device=DEV, generator=g) * 2 - 1) * 0.9
    nd_next = (torch.rand(n, device=DEV, generator=g) > 0.2).float()
    c_prev = torch.randn(n, 256, device=DEV, generator=g) * 0.8
    return dict(U=to_tiles(u).view(tiles, TB).contiguous(), HM=to_tiles(h * nd[:, None]), c_prev=c_prev, nd=nd, nd_next=nd_next)


SENT_BF16, SENT_F32 = 7.0, -9.0


def step_outputs(n):
    tiles = (n + 127) // 128
    return dict(c=torch.full((tiles * 128, 256), SENT_F32, device=DEV),
                HH=torch.full((tiles, 2, TB), SENT_BF16, dtype=torch.bfloat16, device=DEV),
                HMn=torch.full((tiles, 2, TB), SENT_BF16, dtype=torch.bfloat16, device=DEV),
                ACT=torch.full((tiles, 16, AB), SENT_BF16, dtype=torch.bfloat16, device=DEV))


def run_step(lib, lp, x, o, n, t0=0):
    """vine_lstm_step over rows [128 t0, 128 t0 + n) of the inputs x into the outputs o."""
    r0 = 128 * t0
    a = abi.VineLstmStep(params=lp.data_ptr(), u=x["U"][t0:].data_ptr(), hm=x["HM"][t0:].data_ptr(), c_prev=x["c_prev"][r0:].data_ptr(),
                         not_done=x["nd"][r0:].data_ptr(), not_done_next=x["nd_next"][r0:].data_ptr(), c=o["c"][r0:].data_ptr(),
                         hh=o["HH"][t0:].data_ptr(), hm_next=o["HMn"][t0:].data_ptr(), act=o["ACT"][t0:].data_ptr(), n=n)
    assert lib.vine_lstm_step(C.byref(a), None) == 0


def bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def test_lstm_step_y2_grid_equals_two_y4_launches_bit_for_bit():
    """vine_lstm_step picks gridDim.y = 2 above 37 tiles (8 weight pieces per CTA, 4 mbarrier phases per ring stage and TMEM
    buffer) and gridDim.y = 4 below (4 pieces, 2 phases).  n = 8192 (64 tiles, y = 2) against its two 4096-row halves (32 tiles,
    y = 4): every piece runs the same MMA sequence on the same operands whichever CTA runs it, so c, hh, hm_next and act must
    be identical bit for bit."""
    lib = abi.load_library()
    O, n = 18, 8192
    lp = pack(lib, make_params(O, 1), O)
    x = step_inputs(n, O, 2)
    whole, halves = step_outputs(n), step_outputs(n)
    run_step(lib, lp, x, whole, n)
    run_step(lib, lp, x, halves, n // 2, 0)
    run_step(lib, lp, x, halves, n // 2, 32)
    torch.cuda.synchronize()
    for k in ("c", "HH", "HMn", "ACT"):
        assert torch.equal(bits(whole[k]), bits(halves[k])), k
    assert float((whole["ACT"].float() == SENT_BF16).float().mean()) < 1e-3   # every output was written


@pytest.mark.parametrize("n", [4864, 4837, 8192])
def test_lstm_step_y2_grid_matches_float64(n):
    """The y = 2 grid of vine_lstm_step at its first size (38 tiles), a ragged size (4837: the last tile has 27 rows past n)
    and the training size (64 tiles) against float64 gates = U W_ih^T + HM W_hh^T + (b_ih + b_hh) from the decoded tiles and
    the bf16 weights.  The f32 gate sums of exact bf16 products are good to ~1e-6; the cell update uses tanh.approx (relative
    error E < 5e-4, sigmoid absolute E/2).  Per element:
      c:   |dc| <= E (|c_prev m| / 2 + 3 |g| / 2) + 2e-5                (<= 1.4e-3 here)
      h:   |dh| <= one bf16 ulp + 3 E |tanh c| / 2 + bound(c)          (stored bf16)
      act: one bf16 ulp + E / 2 (i, f, o) or E |g| (g) + 2e-5
    hm_next equals hh where not_done_next = 1 and is 0 where it is 0; rows past n keep the sentinel in every output."""
    lib = abi.load_library()
    O = 18
    P = make_params(O, n)
    lp = pack(lib, P, O)
    x = step_inputs(n, O, n + 1)
    o = step_outputs(n)
    run_step(lib, lp, x, o, n)
    torch.cuda.synchronize()
    tiles = (n + 127) // 128
    u = from_tiles(x["U"].view(tiles, 1, TB), n).double()
    hm = from_tiles(x["HM"], n).double()
    wih, whh = P["w_ih"].bfloat16().double(), P["w_hh"].bfloat16().double()
    gates = u[:, :64 + O] @ wih.t() + hm @ whh.t() + (P["b_ih"] + P["b_hh"]).double()
    gi, gf, gg, go = gates.chunk(4, -1)
    i, f, g, og = torch.sigmoid(gi), torch.sigmoid(gf), torch.tanh(gg), torch.sigmoid(go)
    cpm = x["c_prev"].double() * x["nd"].double()[:, None]
    c = f * cpm + i * g
    tc = torch.tanh(c)
    h = og * tc
    bc = E_TANH * (0.5 * cpm.abs() + 1.5 * g.abs()) + 2e-5
    err_c = (o["c"][:n].double() - c).abs()
    assert bool((err_c <= bc).all()), float((err_c - bc).max())
    assert float(err_c.max()) < 2e-3
    hh = from_tiles(o["HH"], n).double()
    bh = bf16_ulp(h) + 1.5 * E_TANH * tc.abs() + bc
    err_h = (hh - h).abs()
    assert bool((err_h <= bh).all()), float((err_h - bh).max())
    act = from_tiles(o["ACT"], n, width=64).double()
    act_ref = torch.cat([i, f, g, og], 1)[:, gate_perm().to(DEV)]
    ba = torch.cat([torch.full_like(i, 0.5 * E_TANH), torch.full_like(f, 0.5 * E_TANH), E_TANH * g.abs(),
                    torch.full_like(og, 0.5 * E_TANH)], 1)[:, gate_perm().to(DEV)] + bf16_ulp(act_ref) + 2e-5
    err_a = (act - act_ref).abs()
    assert bool((err_a <= ba).all()), float((err_a - ba).max())
    # hm_next: hh where the next step continues the episode, 0 where it starts a new one
    hmn = from_tiles(o["HMn"], n)
    live = x["nd_next"] > 0
    assert torch.equal(bits(hmn[live].bfloat16()), bits(hh[live].float().bfloat16()))
    assert float(hmn[~live].abs().max()) == 0.0 and int((~live).sum()) > 0
    # rows of the last tile past n are not written
    full = tiles * 128
    for k, w in (("HH", 128), ("HMn", 128), ("ACT", 64)):
        assert bool((from_tiles(o[k], full, width=w)[n:] == SENT_BF16).all()), k
    assert bool((o["c"][n:] == SENT_F32).all())


# ------------------------------------------------------------------------------------------------------------ 2. head train
def head_reference(Pd, hq, scal, logstd_old, hyp):
    """float64 LayerNorm (eps 1e-5, biased variance) -> heads -> PPO loss of ppo.PPOAgent; returns outputs and gradients."""
    leaves = {k: Pd[k].clone().requires_grad_(True) for k in ("ln_g", "ln_b", "w_mu", "b_mu", "w_v", "b_v", "logstd")}
    hr = hq.clone().requires_grad_(True)
    y = torch.nn.functional.layer_norm(hr, (256,), leaves["ln_g"], leaves["ln_b"], 1e-5)
    mu = y @ leaves["w_mu"].t() + leaves["b_mu"]
    v = (y @ leaves["w_v"].t() + leaves["b_v"])[:, 0]
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
    grads = {k: t.grad for k, t in leaves.items()}
    stats = torch.stack([a_loss.detach(), c_loss.detach(), kl, b_loss.detach()])
    return mu.detach(), v.detach(), nlp.detach(), ratio.detach(), hr.grad, grads, stats


def loss_scalars(mu, v, logstd, e_clip, g, margin):
    """f32 [n, 8] per-row loss scalars (action, mu_old, neglogp_old, value_old, return, advantage) for a network whose outputs
    are mu [n, 2], v [n] (float64), built so that a real fraction of rows takes each branch of the loss -- ratio clipped below
    and above, value clipped -- and every row stays ``margin`` away from a branch boundary (ratio at 1 +- e_clip,
    |v - v_old| at e_clip, (v - ret)^2 == (v_clip - ret)^2), where a kernel and a reference that differ by rounding could take
    different branches and so different gradients."""
    n = mu.shape[0]
    rn = lambda *s: torch.randn(*s, device=DEV, generator=g).double()  # noqa: E731
    sig = torch.exp(logstd.double())
    act = mu + sig * rn(n, 2)
    nlp = 0.5 * (((act - mu) / sig) ** 2).sum(-1) + math.log(2 * math.pi) + logstd.double().sum()
    d = (torch.rand(n, device=DEV, generator=g).double() - 0.5) * 1.2          # log ratio
    for b in (math.log(1 - e_clip), math.log(1 + e_clip)):
        close = (d - b).abs() < margin
        d[close] = b + 2 * margin * torch.sign(d[close] - b + 1e-9)
    dv = (torch.rand(n, device=DEV, generator=g).double() - 0.5) * 1.2
    close = (dv.abs() - e_clip).abs() < margin
    dv[close] = torch.sign(dv[close]) * (e_clip + 2 * margin)
    vo = v + dv
    ret = v + rn(n) * 0.5
    for _ in range(8):
        vc = vo + (v - vo).clamp(-e_clip, e_clip)
        amb = (((v - ret) ** 2 - (vc - ret) ** 2).abs() < margin) & ((v - vo).abs() > e_clip)
        ret[amb] += 0.37
    assert not bool(amb.any())
    return torch.stack([act[:, 0], act[:, 1], mu[:, 0] + 0.1 * rn(n), mu[:, 1] + 0.1 * rn(n), nlp + d, vo, ret, rn(n)],
                       1).float().contiguous()


def head_problem(n, seed, hyp):
    """HH tiles, parameters and loss scalars (every row 0.01 away from a branch boundary of the loss: the f32 kernel's mu, v
    are within 1e-4 of float64)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, device=DEV, generator=g)  # noqa: E731
    P = make_params(18, seed)
    h = torch.tanh(rn(n, 256) * 0.9 + 0.3 * rn(n, 1))
    HH = to_tiles(h)
    hq = from_tiles(HH, n).double()
    Pd = {k: P[k].double() for k in P}
    y = torch.nn.functional.layer_norm(hq, (256,), Pd["ln_g"], Pd["ln_b"], 1e-5)
    mu, v = y @ Pd["w_mu"].t() + Pd["b_mu"], (y @ Pd["w_v"].t() + Pd["b_v"])[:, 0]
    scal = loss_scalars(mu, v, P["logstd"], hyp["e_clip"], g, 0.01)
    logstd_old = P["logstd"] + 0.05
    return P, HH, hq, scal, logstd_old


HEAD_HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.01, bounds_loss_coef=0.05)


@pytest.mark.parametrize("n", [32768, 32765, 640])
def test_lstm_head_train_matches_float64_above_the_block_clamp(n):
    """vine_lstm_head_train clamps its grid to 296 blocks above 2368 rows: each warp then loops over row pairs (HT_ROWS = 2,
    rows past n masked by ok[]) and its A_j sums build up over ~7 iterations.  n = 32768 (the training minibatch), the ragged
    32765 (a masked row in the last pair) and 640 (one pair per warp, no clamp) against a float64 LayerNorm -> heads -> PPO loss
    on the decoded HH, with entropy_coef != 0 and every loss branch taken by a real fraction of rows.
    Tolerances: the row math is f32 with __expf (a few ulp): mu, v within 2e-5 + 1e-5 |x|, neglogp within 2e-5 (1 + |x|); dh
    is stored bf16: one ulp + 1e-4 of the row's largest |dh| (f32 cancellation in rstd (dyh - mean1 - yh mean2)) + 1e-5 of
    the median row's largest |dh| (the f32 loss gradient: act - mu loses ~1e-5 absolute in rows where it is small); the summed
    parameter gradients and loss statistics (f32 sums of 32768 rows through warp, block and partial sums) within 1e-4
    relative per tensor.  At n = 32768 the write-back of update_mu_sigma is checked too: T = 16, N = 4096, L = 4, 4 chunks,
    envs [2048, 4096): columns 2-3 of exactly the minibatch's rows hold debug_out's mu bit for bit, every other byte stays."""
    lib = abi.load_library()
    P, HH, hq, scal, logstd_old = head_problem(n, 100 + n, HEAD_HYP)
    lp = pack(lib, P, 18)
    tiles = HH.shape[0]
    DH = torch.full_like(HH, SENT_BF16)
    gparts = torch.zeros(abi.LSTM_HEAD_GRAD_PARTS, abi.LSTM_HEAD_GRAD_FLOATS, device=DEV)
    dbg = torch.zeros(n, 4, device=DEV)
    ht = abi.VineLstmHeadTrain(params=lp.data_ptr(), hh=HH.data_ptr(), scalars=scal.data_ptr(), logstd=P["logstd"].data_ptr(),
                               logstd_old=logstd_old.data_ptr(), dh=DH.data_ptr(), grads=gparts.data_ptr(), debug_out=dbg.data_ptr(),
                               n=n, inv_B=1.0 / n, **HEAD_HYP)
    wb = None
    if n == 32768:
        T, N, L, chunks, e0, E = 16, 4096, 4, 4, 2048, 2048
        wb = torch.randn(T, N, 8, device=DEV)
        wb_before = wb.clone()
        ht.mu_writeback, ht.wb_seq_len, ht.wb_chunks, ht.wb_num_envs, ht.wb_env_begin, ht.wb_env_count = wb.data_ptr(), L, chunks, N, e0, E
    nparts = lib.vine_lstm_head_train(C.byref(ht), None)
    assert nparts == min((n + 7) // 8, 296)
    torch.cuda.synchronize()
    Pd = {k: P[k].double() for k in P}
    mu, v, nlp, ratio, dh_ref, grads, stats = head_reference(Pd, hq, scal.double(), logstd_old, HEAD_HYP)
    # every branch is exercised
    e = HEAD_HYP["e_clip"]
    fr = {"ratio_low": float((ratio < 1 - e).double().mean()), "ratio_high": float((ratio > 1 + e).double().mean()),
          "value_clipped": float(((v - scal[:, 5].double()).abs() > e).double().mean()),
          "mu_bound": float(((mu.abs() > 1.1).any(-1)).double().mean())}
    assert min(fr.values()) > 0.1, fr
    # per row
    assert bool(((dbg[:, :2].double() - mu).abs() <= 2e-5 + 1e-5 * mu.abs()).all()), float((dbg[:, :2].double() - mu).abs().max())
    assert bool(((dbg[:, 2].double() - v).abs() <= 2e-5 + 1e-5 * v.abs()).all()), float((dbg[:, 2].double() - v).abs().max())
    assert bool(((dbg[:, 3].double() - nlp).abs() <= 2e-5 * (1 + nlp.abs())).all()), float((dbg[:, 3].double() - nlp).abs().max())
    dh = from_tiles(DH, n).double()
    row_max = dh_ref.abs().amax(-1, keepdim=True)
    tol = bf16_ulp(dh_ref) + 1e-4 * row_max + 1e-5 * row_max.median()
    assert bool(((dh - dh_ref).abs() <= tol).all()), float(((dh - dh_ref).abs() - tol).max())
    assert bool((from_tiles(DH, tiles * 128)[n:] == SENT_BF16).all())
    # summed partials
    gs = gparts[:nparts].double().sum(0)
    errs = {"ln_g": rel(gs[0:256], grads["ln_g"]), "ln_b": rel(gs[256:512], grads["ln_b"]),
            "w_mu": rel(gs[512:1024], grads["w_mu"].reshape(-1)), "w_v": rel(gs[1024:1280], grads["w_v"].reshape(-1)),
            "b_mu": rel(gs[1280:1282], grads["b_mu"]), "b_v": rel(gs[1282:1283], grads["b_v"]),
            "logstd": rel(gs[1284:1286], grads["logstd"])}
    errs.update({k: abs(float(gs[1286 + j]) - float(stats[j])) / abs(float(stats[j])) for j, k in enumerate(["a_loss", "c_loss", "kl", "b_loss"])})
    print(n, nparts, fr, {k: f"{x:.1e}" for k, x in errs.items()})
    assert max(errs.values()) < 1e-4, errs
    if wb is not None:
        want = wb_before.clone()
        want.view(chunks, L, N, 8)[:, :, e0:e0 + E, 2:4] = dbg[:, :2].view(L, chunks, E, 2).permute(1, 0, 2, 3)
        assert torch.equal(wb.view(torch.int32), want.view(torch.int32))


# ------------------------------------------------------------------------------------------------------------------ 3. BPTT
def test_lstm_bptt_step_matches_float64_at_the_training_size():
    """vine_lstm_cell_bwd_tiles then vine_lstm_bwd_gemm at S = 8192 (64 tiles x 16 pieces, 64 x 2 GEMM CTAs), from the
    kernel's own ACT and C of a vine_lstm_step, with a non-trivial dh_rec and dc_next.  float64 reference on the decoded tiles.
    Tolerances: the cell backward recomputes tanh(c) with tanh.approx (relative error E), so 1 - tanh^2 c is off by up to
    2 E tanh^2 c and |d(dc)| <= |dh o| (2 E tanh^2 c + 1e-6) + 1e-6 |dc_next| (f32 rounding), which propagates linearly into dG;
    dG is stored bf16: one ulp + that term + 1e-6 relative;
    dc_prev (f32): |f m| |d(dc)| + 1e-6 relative.  The GEMM sums K = 1024 bf16 products in f32: dh3 (f32) within 1e-5 relative
    Frobenius; dh_rec is stored bf16 and masked with not_done: one ulp + 1e-6 of sum |dG| |W| per element, exactly 0 where
    not_done = 0."""
    lib = abi.load_library()
    O, n = 18, 8192
    tiles = n // 128
    P = make_params(O, 31)
    lp = pack(lib, P, O)
    x = step_inputs(n, O, 32)
    o = step_outputs(n)
    run_step(lib, lp, x, o, n)
    g = torch.Generator(device=DEV).manual_seed(33)
    DH = to_tiles(torch.randn(n, 256, device=DEV, generator=g) * 0.05)
    DHR = to_tiles(torch.randn(n, 256, device=DEV, generator=g) * 0.05)
    dc_next = torch.randn(n, 256, device=DEV, generator=g) * 0.05
    nd = x["nd"]
    DG = torch.full((tiles, 16, AB), SENT_BF16, dtype=torch.bfloat16, device=DEV)
    dc_prev = torch.full((n, 256), SENT_F32, device=DEV)
    cb = abi.VineLstmCellBwd(act=o["ACT"].data_ptr(), c_prev=x["c_prev"].data_ptr(), c=o["c"].data_ptr(), not_done=nd.data_ptr(),
                             dh=DH.data_ptr(), dh_rec=DHR.data_ptr(), dc_next=dc_next.data_ptr(), dg=DG.data_ptr(),
                             dc_prev=dc_prev.data_ptr(), n=n)
    assert lib.vine_lstm_cell_bwd_tiles(C.byref(cb), None) == 0
    dh3 = torch.full((n, 64), SENT_F32, device=DEV)
    DHR_out = torch.full_like(DH, SENT_BF16)
    bg = abi.VineLstmBwdGemm(params=lp.data_ptr(), dg=DG.data_ptr(), not_done=nd.data_ptr(), dh3=dh3.data_ptr(),
                             dh_rec=DHR_out.data_ptr(), n=n)
    assert lib.vine_lstm_bwd_gemm(C.byref(bg), None) == 0
    torch.cuda.synchronize()
    # ---- cell backward ----
    a = to_torch_gates(from_tiles(o["ACT"], n, width=64).double())
    gi, gf, gg, go = a.chunk(4, -1)
    dh = from_tiles(DH, n).double() + from_tiles(DHR, n).double()
    cc, cp, m, dcn = o["c"][:n].double(), x["c_prev"].double(), nd.double()[:, None], dc_next.double()
    t = torch.tanh(cc)
    d = dh * go * (1 - t * t) + dcn
    dg_ref = torch.cat([d * gg * gi * (1 - gi), d * cp * m * gf * (1 - gf), d * gi * (1 - gg * gg), dh * t * go * (1 - go)], 1)
    bd = (dh * go).abs() * (2 * E_TANH * t * t + 1e-6) + 1e-6 * dcn.abs()
    bdg = torch.cat([bd * (gg * gi * (1 - gi)).abs(), bd * (cp * m * gf * (1 - gf)).abs(), bd * (gi * (1 - gg * gg)).abs(),
                     (dh * go * (1 - go)).abs() * E_TANH * t.abs()], 1) + 1e-6 * dg_ref.abs()
    dg_k = to_torch_gates(from_tiles(DG, n, width=64).double())
    err = (dg_k - dg_ref).abs() - bf16_ulp(dg_ref) - bdg
    assert float(err.max()) <= 0.0, float(err.max())
    dcp_ref = d * gf * m
    err = (dc_prev.double() - dcp_ref).abs() - (gf * m).abs() * bd - 1e-6 * dcp_ref.abs() - 1e-12
    assert float(err.max()) <= 0.0, float(err.max())
    # ---- backward-data GEMM on the kernel's own dG ----
    wih, whh = P["w_ih"].bfloat16().double(), P["w_hh"].bfloat16().double()
    dh3_ref = dg_k @ wih[:, :64]
    assert rel(dh3, dh3_ref) < 1e-5, rel(dh3, dh3_ref)
    dhr_ref = (dg_k @ whh) * m
    dhr = from_tiles(DHR_out, n).double()
    tol = bf16_ulp(dhr_ref) + 1e-6 * (dg_k.abs() @ whh.abs())
    assert bool(((dhr - dhr_ref).abs() <= tol).all()), float(((dhr - dhr_ref).abs() - tol).max())
    assert float(dhr[nd == 0].abs().max()) == 0.0
    print("dh3", rel(dh3, dh3_ref), "dh_rec", rel(dhr, dhr_ref))


# ------------------------------------------------------------------------------------------------------- 4. wgrad + reduce
@pytest.mark.parametrize("ntiles,splits,O", [(256, 1, 18), (256, 12, 18), (256, 256, 18), (1024, 12, 18), (13, 12, 18),
                                             (256, 12, 28), (256, 12, 14)])
def test_lstm_wgrad_and_reduce_match_float64(ntiles, splits, O):
    """vine_lstm_wgrad + vine_lstm_reduce at the training minibatch (256 tiles; 12 splits = 22 tiles per split and 14 in the
    last), one split, one tile per split, configs[2] (1024 tiles) and 13 tiles over 12 splits (splits 7-11 get none and must
    contribute zeros), against float64 U^T dG and HM^T dG from the decoded tiles in torch gate-row order.  The U tile carries
    junk in its unused columns (64+O..94, 96..127), which the reduce must not map anywhere.  Each split accumulates
    8 x (its tiles) K = 16 MMA blocks in one f32 TMEM accumulator, then the reduce adds <= 256 split sums in f32.  On a B200
    the relative Frobenius error grows linearly with the tiles per split -- 1.9e-7 (1 tile), 2.3e-7 (2), 2.9e-6 (22),
    1.2e-5 (86), 3.8e-5 (256), i.e. ~1.5e-7 per tile, not the sqrt growth of round-to-nearest sums: the tensor core's
    accumulation is biased by a fraction of an ulp per MMA.  Bound: 2.5e-7 per tile of the longest split + 1e-6; one tile
    missed or added would be off by ~1 / ntiles (>= 1e-3 here).
    b_ih and b_hh both come from U column 95 (== 1) and must be identical bits; the LayerNorm / head / logstd / statistics
    slots are the summed head partials (the first head_parts rows only), bit for bit the summed row, 2e-6 of float64;
    every slot of the flat vector is written."""
    lib = abi.load_library()
    rows = ntiles * 128
    g = torch.Generator(device=DEV).manual_seed(ntiles * 1000 + splits + O)
    u = torch.randn(rows, 128, device=DEV, generator=g)
    u[:, 95] = 1.0
    U = to_tiles(u).view(ntiles, TB).contiguous()
    HM = to_tiles(torch.randn(rows, 256, device=DEV, generator=g) * 0.5)
    DG = (torch.randn(ntiles, 16, AB, device=DEV, generator=g) * 0.01).bfloat16()
    ws = torch.full((splits, abi.LSTM_WGRAD_BLOCK_FLOATS), float("nan"), device=DEV)
    wg = abi.VineLstmWgrad(u=U.data_ptr(), hm=HM.data_ptr(), dg=DG.data_ptr(), workspace=ws.data_ptr(), ntiles=ntiles, splits=splits)
    assert lib.vine_lstm_wgrad(C.byref(wg), None) == 0
    hparts = 296
    hg = torch.rand(abi.LSTM_HEAD_GRAD_PARTS + 1, abi.LSTM_HEAD_GRAD_FLOATS, device=DEV, generator=g) * 1e-3
    hg[hparts:] = 1e6                        # rows past head_parts must not be summed
    PL = lib.vine_lstm_num_params(O)
    flat = torch.full((PL + 4,), float("nan"), device=DEV)
    assert lib.vine_lstm_reduce(p(ws), splits, p(hg), hparts, O, p(flat), None, None) == 0
    torch.cuda.synchronize()
    assert bool(torch.isfinite(flat).all())
    Ud, Hd = from_tiles(U.view(ntiles, 1, TB), rows).double(), from_tiles(HM, rows).double()
    Gt = to_torch_gates(from_tiles(DG, rows, width=64).double())
    F = unflat(flat, O)
    errs = {"W_ih": rel(F["w_ih"], Gt.t() @ Ud[:, :64 + O]), "W_hh": rel(F["w_hh"], Gt.t() @ Hd), "b": rel(F["b_ih"], Gt.sum(0))}
    per = -(-ntiles // splits)
    print(ntiles, splits, O, {k: f"{e:.1e}" for k, e in errs.items()})
    assert max(errs.values()) < 2.5e-7 * per + 1e-6, (per, errs)
    assert torch.equal(F["b_ih"].view(torch.int32), F["b_hh"].view(torch.int32))
    hsum = hg[abi.LSTM_HEAD_GRAD_PARTS]
    want = torch.cat([hsum[0:256], hsum[256:512], hsum[512:1024], hsum[1280:1282], hsum[1024:1280], hsum[1282:1283],
                      hsum[1284:1286], hsum[1286:1290]])
    assert torch.equal(flat[F["w_hh"].numel() + F["w_ih"].numel() + 2048:], want)
    ref = hg[:hparts].double().sum(0)
    assert bool(((hsum[:1290].double() - ref[:1290]).abs() <= 2e-6 * ref[:1290].abs()).all())


# ------------------------------------------------------------------------------------------------------------------ 5. gather
@pytest.mark.parametrize("O", [18, 28, 14, 27])
@pytest.mark.parametrize("e0", [0, 2048])
def test_lstm_gather_matches_torch_indexing(O, e0):
    """vine_lstm_gather at the training layout (T = 16, N = 4096, L = 4, 4 chunks, 2048 envs per minibatch = S 8192) against
    torch indexing of the [T, N] rollout buffers: rows ordered [step][chunk, env]; c0 from the saved cell states; hm0 =
    bf16(h_saved) x not_done at the chunk start.  O even takes the float2 path, the odd 27 the scalar one.  Pure data
    movement (and a multiplication by 0 or 1): bit for bit, and nothing written past the outputs."""
    lib = abi.load_library()
    T, N, L, E = 16, 4096, 4, 2048
    chunks, S = T // L, (T // L) * E
    g = torch.Generator(device=DEV).manual_seed(O * 7 + e0)
    obs = torch.randn(T, N, O, device=DEV, generator=g)
    scal = torch.randn(T, N, 8, device=DEV, generator=g)
    nd = (torch.rand(T, N, device=DEV, generator=g) > 0.3).float()
    c_saved = torch.randn(chunks, N, 256, device=DEV, generator=g)
    hh_saved = to_tiles(torch.randn(chunks * N, 256, device=DEV, generator=g))
    mb_obs = torch.full((L * S + 1, O), float("nan"), device=DEV)
    mb_scal = torch.full((L * S + 1, 8), float("nan"), device=DEV)
    mb_nd = torch.full((L * S + 1,), float("nan"), device=DEV)
    c0 = torch.full((S + 1, 256), float("nan"), device=DEV)
    hm0 = torch.full((S // 128 + 1, 2, TB), SENT_BF16, dtype=torch.bfloat16, device=DEV)
    ga = abi.VineLstmGather(obs=obs.data_ptr(), scalars=scal.data_ptr(), not_done=nd.data_ptr(), c_saved=c_saved.data_ptr(),
                            hh_saved=hh_saved.data_ptr(), mb_obs=mb_obs.data_ptr(), mb_scalars=mb_scal.data_ptr(),
                            mb_not_done=mb_nd.data_ptr(), c0=c0.data_ptr(), hm0=hm0.data_ptr(), seq_len=L, chunks=chunks,
                            num_envs=N, env_begin=e0, env_count=E, num_obs=O)
    assert lib.vine_lstm_gather(C.byref(ga), None) == 0
    torch.cuda.synchronize()

    def rows(buf):   # [T, N, ...] -> [L * S, ...] ordered [step][chunk, env]
        return buf.view(chunks, L, N, -1)[:, :, e0:e0 + E].permute(1, 0, 2, 3).reshape(L * S, -1)
    assert torch.equal(mb_obs[:-1], rows(obs)) and bool(mb_obs[-1].isnan().all())
    assert torch.equal(mb_scal[:-1], rows(scal)) and bool(mb_scal[-1].isnan().all())
    assert torch.equal(mb_nd[:-1], rows(nd)[:, 0]) and bool(mb_nd[-1].isnan())
    assert torch.equal(c0[:-1], c_saved[:, e0:e0 + E].reshape(S, 256)) and bool(c0[-1].isnan().all())
    h = from_tiles(hh_saved, chunks * N).view(chunks, N, 256)[:, e0:e0 + E].reshape(S, 256)
    m = nd.view(chunks, L, N)[:, 0, e0:e0 + E].reshape(S, 1)
    assert torch.equal(bits(hm0[:-1]), bits(to_tiles(h * m)))
    assert bool((hm0[-1] == SENT_BF16).all())


# -------------------------------------------------------------------------------------------------------------------- 6. Adam
def adam_grads(PL, seed, k):
    g = torch.Generator(device=DEV).manual_seed(seed * 10 + k)
    grad = torch.randn(PL + 4, device=DEV, generator=g) * torch.pow(10.0, -3 * torch.rand(PL + 4, device=DEV, generator=g))
    grad[PL:] = torch.rand(4, device=DEV, generator=g) + 0.1   # loss statistics
    return grad


@pytest.mark.parametrize("O", [18, 28, 14])
@pytest.mark.parametrize("scale", [1.0, 0.5])
def test_lstm_adam_matches_torch_adam_and_repacks_exactly(O, scale):
    """vine_lstm_adam: three steps against torch.optim.Adam on the flat vector (f32 both: 1e-6 absolute on the parameters;
    exp_avg within 2e-6 of the running sum of its terms' magnitudes, beta1 |m| + (1 - beta1) |g|, since it cancels where the
    gradient changes sign; exp_avg_sq within 2e-5 relative: the kernel takes 1 - beta2 in f32, 1 - 0.999f = 0.00099998713,
    torch in double rounded once, 0.001, which is 1.29e-5 apart), the state bookkeeping (slot 2 = this step's KL, 3 = 1, 4-7 = the summed statistics,
    8 = the step count) and the packed block, which must be byte for byte what vine_lstm_pack makes of the new parameters --
    the packed bias included: fl(b_ih + b_hh), not the old sum plus the two updates."""
    lib = abi.load_library()
    P0 = make_params(O, 40 + O)
    flat = flat_of(P0)
    PL = lib.vine_lstm_num_params(O)
    assert PL == flat.numel()
    packed = pack(lib, P0, O)
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    state[0] = 3e-4
    m, v = torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV)
    ref = flat.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=3e-4, betas=(0.9, 0.999), eps=1e-8)
    stats = torch.zeros(4, dtype=torch.float64, device=DEV)
    m_mag = torch.zeros(PL, dtype=torch.float64, device=DEV)
    for k in range(3):
        grad = adam_grads(PL, O, k)
        state[1] = k + 1.0         # the step count: vine_ppo_minibatch increments it before both Adam launches
        ref.grad = grad[:PL] * scale
        opt.step()
        m_mag = 0.9 * m_mag + 0.1 * ref.grad.double().abs()
        stats += (grad[PL:] * scale).double()
        assert lib.vine_lstm_adam(p(grad), scale, p(flat), p(m), p(v), p(packed), p(state), O, 0.9, 0.999, 1e-8, None, None) == 0
        torch.cuda.synchronize()
        assert float((flat - ref.detach()).abs().max()) < 1e-6
        st = opt.state[ref]
        assert bool(((m.double() - st["exp_avg"].double()).abs() <= 2e-6 * m_mag).all())
        assert torch.allclose(v, st["exp_avg_sq"], rtol=2e-5, atol=1e-14)
        assert float(state[2]) == float(grad[PL + 2] * scale) and float(state[3]) == 1.0
    assert float(state[8]) == 3.0 and torch.allclose(state[4:8].double(), stats, rtol=1e-6)
    packed_ref = pack(lib, unflat(flat, O), O)
    torch.cuda.synchronize()
    assert torch.equal(packed, packed_ref), f"packed block differs from vine_lstm_pack of the new parameters: {packed_diff(packed, packed_ref)}"


def test_lstm_p2p_channel_on_one_rank_is_transparent():
    """world = 1: vine_lstm_reduce writes into the channel's buffer seq & 1 and vine_lstm_adam reads it back (including the
    b_hh gradient its b_ih threads fetch with p2p_sum): after five exchanges (both buffers reused) parameters, moments, packed
    block and state are bit-identical to the run without a channel, and the sequence number advanced once per exchange.
    More ranks need more GPUs (tools/p2p_check.py)."""
    from vine_robot_isaacgymenvs_b200 import distributed as vd
    lib = abi.load_library()
    O = 18
    PL = lib.vine_lstm_num_params(O)
    g = torch.Generator(device=DEV).manual_seed(5)
    wss = [torch.randn(1, abi.LSTM_WGRAD_BLOCK_FLOATS, device=DEV, generator=g) * 0.01 for _ in range(5)]
    hgs = [torch.rand(abi.LSTM_HEAD_GRAD_PARTS + 1, abi.LSTM_HEAD_GRAD_FLOATS, device=DEV, generator=g) * 1e-3 for _ in range(5)]
    results = []
    for use_channel in (False, True):
        P0 = make_params(O, 6)
        flat, packed = flat_of(P0), pack(lib, P0, O)
        m, v, fg = torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV), torch.zeros(PL + 4, device=DEV)
        state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
        state[0] = 3e-4
        ch = vd.P2PChannel(lib, PL + 4, DEV) if use_channel else None
        for k in range(5):
            state[1] = k + 1.0
            hg = hgs[k].clone()
            assert lib.vine_lstm_reduce(p(wss[k]), 1, p(hg), 8, O, p(fg), ch.ptr if ch else None, None) == 0
            assert lib.vine_lstm_adam(p(fg), 1.0, p(flat), p(m), p(v), p(packed), p(state), O, 0.9, 0.999, 1e-8,
                                      ch.ptr if ch else None, None) == 0
        torch.cuda.synchronize()
        if ch is not None:
            assert ch.status() == (5, False)
            ch.close()
        results.append((flat.clone(), m.clone(), v.clone(), packed.clone(), state.clone()))
    for name, a, b in zip(("params", "exp_avg", "exp_avg_sq", "packed", "state"), *results):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), name


# ---------------------------------------------------------------------------------------------------- 7. the whole minibatch
def native_problem(O, L, S, seed):
    torch.manual_seed(seed)
    lib = abi.load_library()
    m = ActorCritic(O, 2, (256, 128, 64), rnn=RNN).to(DEV)
    m.fused_cell = False
    with torch.no_grad():
        m.layer_norm.weight.uniform_(0.5, 1.5); m.layer_norm.bias.uniform_(-0.2, 0.2)
        m.mu.weight.mul_(3.0); m.value.weight.mul_(3.0); m.sigma.uniform_(-0.3, 0.1)
        for prm in m.parameters():     # the kernels see bf16 weights: compare against the same rounded weights
            if prm.dim() == 2 and prm.shape[0] > 3:
                prm.copy_(prm.bfloat16().float())
    z = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    mlp = [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
           m.actor_mlp[4].bias, z(2, 64), z(2), z(1, 64), z(1)]
    assert lib.vine_mlp_pack(*[p(t.detach().contiguous()) for t in mlp], O, p(packed), None) == 0
    r = m.rnn.rnn
    lp = [r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight, m.layer_norm.bias, m.mu.weight,
          m.mu.bias, m.value.weight, m.value.bias]
    lpacked = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_lstm_pack(*[p(t.detach().contiguous()) for t in lp], O, p(lpacked), None) == 0
    d = dict(m=m, packed=packed, lpacked=lpacked, obs=torch.randn(L, S, O, device=DEV) * 2, mean=torch.randn(O, device=DEV) * 0.3,
             inv_std=1.0 / (0.5 + torch.rand(O, device=DEV)), nd=(torch.rand(L, S, device=DEV) > 0.15).float(),
             h0=(torch.randn(S, 256, device=DEV) * 0.5).bfloat16().float(), c0=torch.randn(S, 256, device=DEV) * 0.5,
             logstd_old=torch.tensor([-0.1, 0.05], device=DEV))
    # loss scalars around the fp32 network's outputs, every row 0.05 away from a branch boundary of the loss (the bf16 kernels'
    # mu, v are ~1e-2 off the fp32 ones; a row that lands on the other side of a clip changes the gradient by its whole term)
    with torch.no_grad():
        mu, _, v, _ = m(torch.clamp((d["obs"] - d["mean"]) * d["inv_std"], -5, 5), (d["h0"], d["c0"]), d["nd"])
    g = torch.Generator(device=DEV).manual_seed(seed)
    d["scal"] = loss_scalars(mu.double(), v.double().squeeze(-1), m.sigma.detach(), HYP["e_clip"], g, 0.05).view(L, S, 8)
    return d


def run_path(path, d, sl, dbg=None):
    nd =d["nd"][:, sl].contiguous()
    path.HM[0].copy_(to_tiles(d["h0"][sl] * nd[0][:, None]))
    path.C0.copy_(d["c0"][sl])
    vstats, state = torch.tensor([0.0, 1.0], device=DEV), torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    path.gradients(d["packed"], d["lpacked"], d["obs"][:, sl].contiguous(), d["scal"][:, sl].contiguous(), nd, d["mean"], d["inv_std"],
                   vstats, d["m"].sigma.detach(), d["logstd_old"], state, debug_out=dbg)
    torch.cuda.synchronize()
    return path.flat_g_mlp.double().clone(), path.flat_g_lstm.double().clone()


HYP = dict(e_clip=0.2, critic_coef=2.0, entropy_coef=0.0, bounds_loss_coef=1e-4)


def test_native_lstm_minibatch_at_the_training_size_is_the_mean_of_its_halves():
    """NativeLstmPath(18, 4, 8192).gradients -- the default training minibatch: y = 2 step grids, the clamped head grid, the
    MLP backward with 256 tiles on 148 CTAs (several tiles per CTA in persistent TMEM accumulators), 22-tile wgrad splits --
    against the mean of the same minibatch's two 4096-sequence halves (y = 4 step grids, other splits and CTA loads).  The loss
    is a mean over rows: halving n doubles inv_B exactly, so every per-row quantity of a half is exactly twice the whole's and
    only the order of the f32 sums differs: 2e-5 of the gradient norm per network and 1e-5 on the loss statistics."""
    from vine_robot_isaacgymenvs_b200.ppo.lstm_native import NativeLstmPath
    O, L, S = 18, 4, 8192
    d = native_problem(O, L, S, 21)
    whole = run_path(NativeLstmPath(O, L, S, DEV, HYP), d, slice(0, S))
    half = NativeLstmPath(O, L, S // 2, DEV, HYP)
    a = run_path(half, d, slice(0, S // 2))
    b = run_path(half, d, slice(S // 2, S))
    for k, (w, ga, gb) in enumerate(zip(whole, a, b)):
        Pn = w.numel() - 4
        h = 0.5 * (ga + gb)
        assert float(w[:Pn].norm()) > 1e-3
        e = float((w[:Pn] - h[:Pn]).norm() / w[:Pn].norm())
        print(("mlp", "lstm")[k], f"{e:.2e}")
        assert e < 2e-5, (k, e)
        for j in range(4):
            assert abs(float(w[Pn + j]) - float(h[Pn + j])) <= 1e-5 * max(abs(float(w[Pn + j])), 1e-3), (k, j, float(w[Pn + j]), float(h[Pn + j]))


def test_native_lstm_minibatch_o28_matches_autograd_at_the_training_size():
    """The 28-wide network (the default pipe task) through the whole kernel-only minibatch at S = 8192 against fp32 torch
    autograd of ppo.ActorCritic: 4e-2 relative Frobenius error per parameter tensor, as in test_gpu_lstm_net.py (bf16
    operands through a 4-step recurrence).  The loss scalars keep every row 0.05 away from a clip boundary: with the
    boundary-blind scalars of test_gpu_lstm_net.py, the rows whose ratio or value the bf16 forward moves across a clip put
    the head bias gradient (a sum of terms of both signs) 5.8e-2 off at this size."""
    from vine_robot_isaacgymenvs_b200.ppo.lstm_native import NativeLstmPath
    O, L, S = 28, 4, 8192
    d = native_problem(O, L, S, 22)
    m = d["m"]
    dbg = torch.zeros(L * S, 4, device=DEV)
    gm, gl = run_path(NativeLstmPath(O, L, S, DEV, HYP), d, slice(0, S), dbg)
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
        errs[name] = rel(gl[o:o + prm.numel()].view_as(prm), prm.grad)
        o += prm.numel()
    assert o == gl.numel() - 4
    o = 0
    for name, prm in (("W1", m.actor_mlp[0].weight), ("b1", m.actor_mlp[0].bias), ("W2", m.actor_mlp[2].weight),
                      ("b2", m.actor_mlp[2].bias), ("W3", m.actor_mlp[4].weight), ("b3", m.actor_mlp[4].bias)):
        errs[name] = rel(gm[o:o + prm.numel()].view_as(prm), prm.grad)
        o += prm.numel()
    print({k: f"{e:.2e}" for k, e in errs.items()})
    P = gl.numel() - 4
    assert abs(float(gl[P]) - float(a_loss)) < 3e-2 * abs(float(a_loss)) + 1e-4
    assert abs(float(gl[P + 1]) - float(c_loss)) < 3e-2 * float(c_loss)
    assert max(errs.values()) < 4e-2, errs
