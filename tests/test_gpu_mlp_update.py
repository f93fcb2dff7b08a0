"""GPU: the actor-critic MLP kernels -- vine_ppo_minibatch (both epilogue variants) + vine_ppo_reduce, vine_policy_act and
the update prologue (vine_ppo_moments / vine_ppo_finalize) -- against float64 references that round where the kernels round.

The forward reference restates the kernel's data path on its own bf16 operands:
  x  = bf16(clamp((obs - mean) * inv_std, +-5))   (f32 arithmetic, as build_x_tile; column 31 = 1 carries db1 through dW1)
  hi = bf16(ELU(h_{i-1} Wi^T + bi))                (weights rounded to bf16 as vine_mlp_pack rounds them)
  mu, v = h3 Wh^T + bh
and the backward its roundings: the head gradients (dmu, dv, already scaled by 1/B) are rounded to bf16 before the
backward GEMMs, and dz_i = bf16(dh_i ELU'(h_i)) with ELU'(h) = 1 if h > 0 else h + 1 evaluated on the bf16-stored h.
The loss follows torch's rules: torch.max splits its gradient on a tie, clamp passes it at its bounds.

What then separates kernel and reference: f32 accumulation order (tensor-core MMA, warp sums, CTA partials), ex2.approx in
ELU (a few f32 ulp), __expf in the ratio, and -- the largest -- the rare activation whose f32 pre-image sits within that
noise of a bf16 rounding boundary and so rounds to the neighbouring bf16 value (one bf16 ulp, 2^-8 relative).  The loss
scalars keep every row 0.02 away from a branch boundary of the loss (the kernel's mu, v are within ~1e-3 of float64 even
on a row with such a flip), so kernel and reference take the same branch on every row except where a test plants rows
exactly on a boundary.  Each test states the tolerance it derives from these sources."""
import ctypes as C
import math

import pytest
import torch

from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200.ppo.ppo import RunningMeanStd
from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles
from test_gpu_lstm_update import HEAD_HYP, bf16_ulp, loss_scalars, rel
from test_gpu_ppo_fused import NAMES, _act, make_problem, p, run_kernel, split

pytestmark = pytest.mark.gpu
DEV = "cuda"
MARGIN = 0.02      # distance of every row from a loss-branch boundary (log ratio, |v - v_old|, c1 - c2)
# T, N, e0, E of a minibatch: rows s = t * E + (env - e0) of the [T, N] rollout buffers
SHAPES = {"train": (16, 4096, 2048, 2048),   # the training minibatch: 256 tiles on 148 CTAs
          "ragged": (8, 600, 100, 333),      # B = 2664 (20 tiles + 104 rows), unaligned slice
          "tiny": (1, 200, 37, 77),          # one partial tile
          "many": (16, 4096, 0, 4096)}       # 512 tiles > 2 x 148: three or four tiles per CTA


def bf(t):
    """round to bf16 the way the kernels do (f32 value, round to nearest even), back to float64."""
    return t.float().bfloat16().double()


def elu(z):
    return torch.where(z > 0, z, torch.expm1(z))


def elu_grad(h):
    """ELU' as a function of the (bf16-stored) output."""
    return torch.where(h > 0, torch.ones_like(h), h + 1)


def x_tile(obs, mean, inv_std, ones_column):
    """[n, 32] float64 of the bf16 x tile build_x_tile writes."""
    n, O = obs.shape
    x = torch.zeros(n, 32, dtype=torch.float64, device=obs.device)
    x[:, :O] = bf(torch.clamp((obs - mean) * inv_std, -5.0, 5.0))   # f32, no FMA contraction possible: (a - b) * c
    if ones_column:
        x[:, 31] = 1.0
    return x


def forward_ref(W, obs, mean, inv_std):
    """float64 forward on the kernel's bf16 operands; W = make_problem's list (torch layouts, f32)."""
    w1, b1, w2, b2, w3, b3, wmu, bmu, wv, bv = [w.double() for w in W[:10]]
    O = obs.shape[1]
    x = x_tile(obs, mean, inv_std, True)
    h1 = bf(elu(x[:, :O] @ bf(w1).t() + b1))
    h2 = bf(elu(h1 @ bf(w2).t() + b2))
    h3 = bf(elu(h2 @ bf(w3).t() + b3))
    wh, bh = torch.cat([bf(wmu), bf(wv)]), torch.cat([bmu, bv])
    head = h3 @ wh.t() + bh
    return dict(x=x, h1=h1, h2=h2, h3=h3, wh=wh, bh=bh, mu=head[:, :2], v=head[:, 2])


def value_branches(v, vo, ret, e_clip):
    """(c1 > c2, c2 > c1, |v - vo| <= e_clip) in the dtype of v -- the kernel's f32 expression order when v is f32."""
    e = torch.tensor(e_clip, dtype=v.dtype, device=v.device)
    dvo = v - vo
    vclip = vo + torch.clamp(dvo, -e, e)
    c1, c2 = (v - ret) ** 2, (vclip - ret) ** 2
    return c1 > c2, c2 > c1, dvo.abs() <= e


def loss_ref(mu, v, scal, logstd, logstd_old, hyp, clip_value, v_branch=None):
    """float64 per-row loss gradients (d/dmu, d/dv, d/dlogstd, all before the 1/B of the mean) and the four loss statistics
    of ppo.PPOAgent's loss on the network outputs mu [n, 2], v [n].  ``v_branch`` overrides the branch masks of the value
    loss (rows planted exactly on the clip boundary are decided by the kernel's f32 arithmetic)."""
    s = scal.double()
    act, muo, nlpo, vo, ret, adv = s[:, :2], s[:, 2:4], s[:, 4], s[:, 5], s[:, 6], s[:, 7]
    ls, lso = logstd.double(), logstd_old.double()
    sig, e = torch.exp(ls), hyp["e_clip"]
    d = (act - mu) / sig
    nlp = 0.5 * (d * d).sum(-1) + math.log(2 * math.pi) + ls.sum()
    ratio = torch.exp(nlpo - nlp)
    t1, t2 = -adv * ratio, -adv * torch.clamp(ratio, 1 - e, 1 + e)
    # torch.max: the larger term takes the gradient, a tie (ratio inside the clip, both terms equal) splits it half and
    # half between -adv ratio and -adv clamp(ratio) -- whose gradients are equal there (clamp passes it at its bounds)
    inside = (ratio >= 1 - e) & (ratio <= 1 + e)
    g_nlp = torch.where(inside | (t1 > t2), adv * ratio, torch.zeros_like(adv))
    dmu = g_nlp[:, None] * (-d / sig)
    dls = g_nlp[:, None] * (1 - d * d) - hyp["entropy_coef"]
    e1, vclip = v - ret, vo + torch.clamp(v - vo, -e, e)
    e2 = vclip - ret
    gt, lt, pass2 = v_branch if v_branch is not None else value_branches(v, vo, ret, e)
    pass2 = pass2.double()
    if clip_value:
        dvc = torch.where(gt, 2 * e1, torch.where(lt, 2 * e2 * pass2, e1 + e2 * pass2))
        c_row = torch.maximum(e1 * e1, e2 * e2)
    else:
        dvc, c_row = 2 * e1, e1 * e1
    dv = 0.5 * hyp["critic_coef"] * dvc
    bhi, blo = torch.clamp_min(mu - 1.1, 0), torch.clamp_max(mu + 1.1, 0)
    dmu = dmu + hyp["bounds_loss_coef"] * 2 * (bhi + blo)
    so = torch.exp(lso)
    kl = (torch.log(so / sig + 1e-5) + (sig ** 2 + (mu - muo) ** 2) / (2 * (so ** 2 + 1e-5)) - 0.5).sum(-1)
    rows = dict(a_loss=torch.maximum(t1, t2), c_loss=c_row, kl=kl, b_loss=(bhi ** 2 + blo ** 2).sum(-1))
    fr = {"ratio_low": ratio < 1 - e, "ratio_in": inside, "ratio_high": ratio > 1 + e}
    branches = {f"{k}_adv{sg}": m & (adv > 0 if sg == "+" else adv < 0) for k, m in fr.items() for sg in "+-"}
    branches.update(value_clipped=(v - vo).abs() > e, value_inside=(v - vo).abs() <= e, mu_above=(mu > 1.1).any(-1),
                    mu_below=(mu < -1.1).any(-1))
    return dict(dmu=dmu, dv=dv, dls=dls, nlp=nlp, rows=rows, branches=branches)


def gradients_ref(fwd, W, loss, inv_B):
    """float64 backward of the kernel's chain from the bf16-rounded head gradients; -> list in NAMES order."""
    O = W[0].shape[1]
    dzh = bf(torch.cat([loss["dmu"], loss["dv"][:, None]], 1) * inv_B)     # [n, 3]: dmu0, dmu1, dv
    h1, h2, h3, x = fwd["h1"], fwd["h2"], fwd["h3"], fwd["x"]
    gwh, gbh = dzh.t() @ h3, dzh.sum(0)
    dz3 = bf((dzh @ fwd["wh"]) * elu_grad(h3))
    gw3, gb3 = dz3.t() @ h2, dz3.sum(0)
    dz2 = bf((dz3 @ bf(W[4].double())) * elu_grad(h2))
    gw2, gb2 = dz2.t() @ h1, dz2.sum(0)
    dz1 = bf((dz2 @ bf(W[2].double())) * elu_grad(h1))
    gw1 = dz1.t() @ x                                                       # column 31 (== 1) is db1
    gls = loss["dls"].sum(0) * inv_B
    return [gw1[:, :O], gw1[:, 31], gw2, gb2, gw3, gb3, gwh[:2], gbh[:2], gwh[2:], gbh[2:], gls]


def rows_of(buf, key, e0, E):
    t = buf[key][:, e0:e0 + E]
    return t.reshape(-1, *t.shape[2:])


def mlp_problem(shape, O, seed):
    """make_problem's network and observations (its head puts |mu| > 1.1 on a good share of rows in both directions) and
    loss scalars built around the float64 forward so that every branch of the loss is taken (loss_scalars)."""
    T, N, e0, E = SHAPES[shape]
    W, buf, mean, inv_std, logstd_old = make_problem(T, N, O, seed=seed)
    obs = rows_of(buf, "obs", e0, E).contiguous()
    fwd = forward_ref(W, obs, mean, inv_std)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    scal = loss_scalars(fwd["mu"], fwd["v"], W[10], HEAD_HYP["e_clip"], g, MARGIN)
    set_scalars(buf, scal, e0, E)
    return W, buf, mean, inv_std, logstd_old, obs, fwd, scal


def set_scalars(buf, scal, e0, E):
    T = buf["act"].shape[0]
    s = scal.view(T, E, 8)
    buf["act"][:, e0:e0 + E] = s[..., 0:2]
    buf["mu_old"][:, e0:e0 + E] = s[..., 2:4]
    for j, k in ((4, "nlp_old"), (5, "val_old"), (6, "ret"), (7, "adv")):
        buf[k][:, e0:e0 + E] = s[..., j]


def u_tile(lib, packed, obs, mean, inv_std):
    """vine_policy_act in u_out mode: -> [n, 128] float64 of the U tile [h3 | x | 0] (the kernel's own h3 and x)."""
    n, O = obs.shape
    tiles = (n + 127) // 128
    U = torch.full((tiles, 1, 128 * 128), 7.0, dtype=torch.bfloat16, device=DEV)
    vstats = torch.tensor([0.0, 1.0], device=DEV)
    a = abi.VinePolicyAct(packed=packed.data_ptr(), obs=obs.data_ptr(), obs_mean=mean.data_ptr(), obs_inv_std=inv_std.data_ptr(),
                          value_stats=vstats.data_ptr(), n=n, num_obs=O, u_out=U.data_ptr())
    assert lib.vine_policy_act(C.byref(a), None) == 0
    torch.cuda.synchronize()
    return U, from_tiles(U, n).double()


def check_h3(h3_k, fwd, w3):
    """The kernel's h3 against the float64 forward.  Each layer's f32 accumulator is exact up to the rounding of its sum
    (~1e-6 relative) and ELU's ex2.approx - 1 (a few f32 ulp, more relative to tiny negative pre-activations), so an
    activation rounds to the reference's bf16 value unless its pre-image lies within that noise of a rounding boundary;
    such a flip moves it by one bf16 ulp and the next layer's pre-image by |w| times that.  So nearly every element is
    identical and the others are off by a flip of their own or one inherited from an h2 element: at most 1 % of elements
    may differ, none by more than 2 ulp(h3) + 2 max_k |W3_jk| max_k ulp(h2_k) (a wrong bias, column or layer would move
    most elements by many ulps)."""
    h3_ref = fwd["h3"]
    d = (h3_k - h3_ref).abs()
    ulp = bf16_ulp(h3_ref)
    inherited = bf16_ulp(fwd["h2"]).amax(-1, keepdim=True) * bf(w3.double()).abs().amax(-1)[None, :]
    tol = 2 * ulp + 2 * inherited
    frac = float((d > 0).double().mean())
    worst = float((d / (ulp + 1e-30)).max())
    assert frac < 1e-2, frac
    assert bool((d <= tol).all()), float((d - tol).max())
    return frac, worst


def check_heads(mu_k, v_k, h3_k, wh, bh):
    """mu, v against float64 heads on the kernel's own h3: 64 exact bf16 products summed in f32, then + the f32 bias:
    within 1e-5 of sum |w h| + |b| (f32 accumulation, with room for the tensor core's truncating adds)."""
    ref = h3_k @ wh.t() + bh
    tol = 1e-5 * (h3_k.abs() @ wh.abs().t() + bh.abs()) + 1e-7
    got = torch.cat([mu_k.double(), v_k.double()[:, None]], 1)
    err = (got - ref).abs()
    assert bool((err <= tol).all()), float((err - tol).max())


def check_nlp(nlp_k, mu_k, act, logstd):
    """neglogp of the kernel against float64 from the kernel's own mu: f32 arithmetic on O(1) terms with __expf in sigma:
    within 2e-5 (1 + |nlp|)."""
    sig = torch.exp(logstd.double())
    d = (act.double() - mu_k.double()) / sig
    ref = 0.5 * (d * d).sum(-1) + math.log(2 * math.pi) + logstd.double().sum()
    err = (nlp_k.double() - ref).abs()
    assert bool((err <= 2e-5 * (1 + ref.abs())).all()), float((err / (1 + ref.abs())).max())


# -------------------------------------------------------------------------------------------- 1. minibatch gradients vs float64
# Relative Frobenius error of each summed gradient tensor: the f32 sums over B rows (tensor-core accumulation across a
# CTA's tiles, warp butterflies, the f32 sum of <= 148 partials) contribute ~1e-6; a bf16 flip of one activation or dz
# element (probability ~1e-4 each, see check_h3) moves one product by 2^-8 of itself, and such flips add up like a random
# walk over the rows: ~1e-4 of a tensor whose rows mostly agree in sign, more for tensors that are small sums of
# terms of both signs (logstd: the actor term and the entropy term nearly cancel; on a B200 the worst measured error,
# 7.2e-4, is logstd at O = 31).  Bound: 2e-3 per tensor, 15x below the 3e-2 of the fp32 autograd comparison.
# The loss statistics are compared with float64 rows evaluated on the kernel's own mu, v (debug_out, which check_heads
# ties to the kernel's h3): a row whose mu moved by a bf16 flip would otherwise count fully in a small minibatch.  What is
# left is the f32 row arithmetic (__expf of the log ratio: ~1e-6 of a term) and the f32 sums of the rows: 1e-5 of the
# mean |row term| (a statistic can be a mean of terms of both signs).  The KL adds a bias that does not average out:
# its constants klc = __logf(sigma_old / sigma + 1e-5) - 1/2 carry lg2.approx's absolute error (~2^-22) into every row
# alike, 1e-6 absolute for the two of them (measured on a B200: 8.7e-6 of the mean |row|, 0.09, at the training size).
TOL_GRAD = 2e-3
TOL_STAT = 1e-5
KL_LOG_BIAS = 1e-6
STATS = ["a_loss", "c_loss", "kl", "b_loss"]


def compare_to_reference(tag, W, out, dbg, fwd, loss, stat_rows, B):
    P = out.numel() - 4
    grads = gradients_ref(fwd, W, loss, 1.0 / B)
    got = split(out[:P].double(), W)
    errs = {k: rel(g, r) for k, g, r in zip(NAMES, got, grads)}
    for j, k in enumerate(STATS):
        rows = stat_rows[k]
        errs[k] = abs(float(out[P + j]) - float(rows.mean())) / (float(rows.abs().mean()) + 1e-30)
    print(tag, {k: f"{e:.1e}" for k, e in errs.items()})
    tol = {k: TOL_STAT for k in STATS}
    tol["kl"] += KL_LOG_BIAS / (float(stat_rows["kl"].abs().mean()) + 1e-30)
    bad = {k: e for k, e in errs.items() if e > tol.get(k, TOL_GRAD)}
    assert not bad, (tag, bad)
    assert bool(torch.isfinite(out).all()) and bool(torch.isfinite(dbg).all())
    return errs


CASES = [("train", 14, 1), ("train", 18, 1), ("train", 26, 1), ("train", 28, 1), ("train", 31, 1),
         ("ragged", 14, 1), ("ragged", 31, 1), ("tiny", 18, 1), ("tiny", 31, 1), ("many", 26, 1),
         ("train", 18, 0), ("ragged", 31, 0)]


@pytest.mark.parametrize("shape,O,clip_value", CASES)
def test_minibatch_matches_float64_with_both_epilogues(shape, O, clip_value):
    """vine_ppo_minibatch + vine_ppo_reduce against the float64 restatement: all 11 gradient tensors, the four loss
    statistics (TOL_GRAD, TOL_STAT above), debug_out's mu, v (check_heads on the kernel's own h3, which vine_policy_act's
    u_out mode emits from the same x tile; check_h3 ties that h3 to float64) and nlp (check_nlp), and the mu_old
    write-back (run_kernel), with entropy_coef = 0.01, bounds_loss_coef = 0.05 and every branch of the loss taken by a
    real fraction of rows.

    Q = 4 (default) and Q = 2 (reserved = 2): the variants differ only in which thread applies the element-wise epilogues
    (bias + ELU, dh ELU') to which columns -- the same f32 operation on the same inputs -- while every sum is formed in the
    same order: the MMAs are issued by thread 0 over the same tiles, the loss and its statistics by the 128 threads of
    part 0 (warps 0-3 in both), the head gradient and the db2 / db3 column sums by warps 0-7 (present in both), and the
    workspace partials go through the same reduce.  So all 11 gradient tensors, a_loss, c_loss, b_loss, debug_out and
    the mu_old write-back must be identical bit for bit.  The KL statistic is the exception: its per-row expression
    klc0 + (sig0^2 + m0^2) klq0 + klc1 + (sig1^2 + m1^2) klq1 is the same source in both instantiations, but each is
    compiled on its own and the compiler may fuse a different product of it into an FMA (IEEE f32 semantics allow either
    contraction).  On a B200 the summed KL of the two differs in its last bits (<= 8 ulp is allowed) while every other
    slot agrees.  The KL only feeds the adaptive learning rate's comparison with kl_threshold."""
    T, N, e0, E = SHAPES[shape]
    B = T * E
    lib = abi.load_library()
    W, buf, mean, inv_std, logstd_old, obs, fwd, scal = mlp_problem(shape, O, seed=1000 * O + B + clip_value)
    hyp = dict(HEAD_HYP, value_loss_unclipped=1 - clip_value)
    runs = {}
    for q in (4, 2):
        flat, packed, _, out, dbg, n_part = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, dict(hyp, reserved=q), O, T, N)
        assert n_part == min((B + 127) // 128, lib.vine_ppo_max_ctas())
        runs[q] = (out.clone(), dbg.clone(), buf["mu_after"].clone())
    P = lib.vine_ppo_num_params(O)
    kl4, kl2 = runs[4][0][P + 2].clone(), runs[2][0][P + 2].clone()
    for q in (4, 2):
        runs[q][0][P + 2] = 0.0
    for name, a, b in zip(("gradients and statistics", "debug_out", "mu_old write-back"), runs[4], runs[2]):
        differ = (a.view(torch.int32) != b.view(torch.int32)).nonzero().flatten().tolist()
        assert not differ, f"Q = 2 and Q = 4 differ in {name} at {differ[:20]} (P = {P})"
    kl_ulps = abs(int(kl4.view(torch.int32)) - int(kl2.view(torch.int32)))
    print(f"Q = 2 vs Q = 4: identical except the KL statistic, {kl_ulps} ulp apart")
    assert kl_ulps <= 8, (float(kl4), float(kl2))
    out, dbg, _ = runs[4]
    out[P + 2] = kl4
    logstd = flat[-2:]
    loss = loss_ref(fwd["mu"], fwd["v"], scal, logstd, logstd_old, HEAD_HYP, clip_value)
    # every branch of the loss is taken (a real fraction of rows at the larger shapes)
    fr = {k: float(m.double().mean()) for k, m in loss["branches"].items()}
    print(shape, O, "clip_value", clip_value, "partials", n_part, "branch fractions", {k: f"{f:.3f}" for k, f in fr.items()})
    if B >= 2000:
        assert min(fr.values()) > 0.02, fr
    # per row: the kernel's x and h3 (u_out of vine_policy_act), then debug_out's heads on that h3 and nlp
    U, u = u_tile(lib, packed, obs, mean, inv_std)
    ref_x = fwd["x"].float().bfloat16()
    assert torch.equal(u[:, 64:96].float().bfloat16().view(torch.int16), ref_x.view(torch.int16))
    frac, worst = check_h3(u[:, :64], fwd, W[4])
    check_heads(dbg[:, :2], dbg[:, 2], u[:, :64], fwd["wh"], fwd["bh"])
    check_nlp(dbg[:, 3], dbg[:, :2], scal[:, :2], logstd)
    print(f"h3: {frac:.2e} of elements differ from float64, by <= {worst:.1f} bf16 ulp")
    stat_rows = loss_ref(dbg[:, :2].double(), dbg[:, 2].double(), scal, logstd, logstd_old, HEAD_HYP, clip_value)["rows"]
    compare_to_reference(f"{shape} O={O} clip_value={clip_value}", W, out, dbg, fwd, loss, stat_rows, B)


@pytest.mark.parametrize("q", [4, 2])
def test_minibatch_value_clip_boundary_follows_torch(q):
    """Rows planted exactly on the value clip: from a first pass's debug_out v, values_old is chosen per row so that the
    kernel's f32 v - v_old is +e_clip or -e_clip exactly (checked in f32 on the host, adjusted by ulps).  torch's clamp
    passes the gradient at its bounds, so v_clip = v_old + clamp(v - v_old) moves with v there, and (v - ret)^2 and
    (v_clip - ret)^2 (equal up to the rounding of v_old + e_clip) tie or nearly tie: the branch is decided in f32 on the
    kernel's v, with the tie split half and half as torch.max does.  Every second row of the training minibatch is
    planted; it lands exactly on the boundary where an f32 v_old with v - v_old == +-e_clip exists (|v| up to ~0.4: beyond,
    v - v_old is a multiple of a coarser ulp than e_clip's), at least 1/32 of the minibatch.  The second pass must
    reproduce the first pass's v bit for bit, and every tensor must match float64 as in
    test_minibatch_matches_float64_with_both_epilogues."""
    T, N, e0, E = SHAPES["train"]
    B, O = T * E, 18
    lib = abi.load_library()
    W, buf, mean, inv_std, logstd_old, obs, fwd, scal = mlp_problem("train", O, seed=77)
    hyp = dict(HEAD_HYP, reserved=q)
    _, _, _, _, dbg0, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, hyp, O, T, N)
    v = dbg0[:, 2].clone()
    e = torch.tensor(HEAD_HYP["e_clip"], dtype=torch.float32, device=DEV)
    on = torch.zeros(B, dtype=torch.bool, device=DEV)
    on[::2] = True
    sign = torch.where(torch.arange(B, device=DEV) % 4 == 0, 1.0, -1.0)
    vo = scal[:, 5].clone()
    cand = v - sign * e
    for _ in range(16):   # v - cand == sign * e in f32, moving cand by one ulp at a time towards it
        diff = (v - cand) - sign * e
        cand = torch.where(diff > 0, torch.nextafter(cand, torch.full_like(cand, math.inf)),
                           torch.where(diff < 0, torch.nextafter(cand, torch.full_like(cand, -math.inf)), cand))
    exact = on & ((v - cand) == sign * e)
    assert int(exact.sum()) >= B // 32, int(exact.sum())
    vo = torch.where(exact, cand, vo)
    scal = scal.clone()
    scal[:, 5] = vo
    set_scalars(buf, scal, e0, E)
    _, _, _, out, dbg, _ = run_kernel(lib, W, buf, mean, inv_std, logstd_old, e0, E, hyp, O, T, N)
    assert torch.equal(dbg[:, 2].view(torch.int32), v.view(torch.int32))
    gt, lt, pass2 = value_branches(v, vo, scal[:, 6], HEAD_HYP["e_clip"])
    assert bool(pass2[exact].all())
    ties = exact & ~gt & ~lt
    print(f"q={q}: {int(exact.sum())} rows on the clip boundary, {int(ties.sum())} of them exact ties")
    logstd = W[10]
    loss = loss_ref(fwd["mu"], fwd["v"], scal, logstd, logstd_old, HEAD_HYP, True, v_branch=(gt, lt, pass2))
    stat_rows = loss_ref(dbg[:, :2].double(), dbg[:, 2].double(), scal, logstd, logstd_old, HEAD_HYP, True,
                         v_branch=(gt, lt, pass2))["rows"]
    compare_to_reference(f"boundary q={q}", W, out, dbg, fwd, loss, stat_rows, B)


# ------------------------------------------------------------------------------------------------------- 2. vine_policy_act
VSTATS = (0.3, 1.7)   # value_stats test_gpu_ppo_fused._act passes


def act_problem(n, O, seed):
    lib = abi.load_library()
    W, buf, mean, inv_std, _ = make_problem(1, n, O, seed=seed)
    W[8].mul_(12.0)    # |v| > 5 on a real fraction of rows: the value clamp
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_mlp_pack(*[p(w.contiguous()) for w in W[:10]], O, p(packed), None) == 0
    return lib, W, buf["obs"][0].contiguous(), mean, inv_std, packed


@pytest.mark.parametrize("O", [14, 26, 31])
def test_policy_act_matches_float64(O):
    """vine_policy_act in sampling mode at n = 300 tiles + 45 rows (grid clamped to the SMs, ragged last tile) against the
    float64 forward: h3 from the u_out mode of the same launch configuration (check_h3), mu and the raw value on that h3
    (check_heads), value = clamp(v, +-5) * std + mean in f32 (the clamp is taken by a real fraction of rows), neglogp
    against float64 from the kernel's own noise z = (a - mu) / sigma (a = fma(sigma, z, mu) in f32, so z comes back
    within 1e-6 of |z| + one ulp of a / sigma: 2e-5 (1 + nlp) covers it), env_actions = clamp(actions, +-1) exactly."""
    n = 300 * 128 + 45
    lib, W, obs, mean, inv_std, packed = act_problem(n, O, seed=500 + O)
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    counter = torch.zeros(1, dtype=torch.int32, device=DEV)
    o = _act(lib, packed, obs, mean, inv_std, logstd, counter, n, O)
    fwd = forward_ref(W, obs, mean, inv_std)
    _, u = u_tile(lib, packed, obs, mean, inv_std)
    frac, worst = check_h3(u[:, :64], fwd, W[4])
    # the raw head output v is not an output here: invert the value affine where the clamp is not active
    vm, vs = VSTATS
    v_ref = u[:, :64] @ fwd["wh"][2] + fwd["bh"][2]
    clamped = v_ref.abs() > 5.0 + 1e-3
    inside = v_ref.abs() < 5.0 - 1e-3
    assert 0.02 < float(clamped.double().mean()) < 0.98
    v_k = (o["value"].double() - vm) / vs
    check_heads(o["mu"][inside], v_k[inside].float(), u[inside, :64], fwd["wh"], fwd["bh"])
    want = torch.clamp(v_ref[clamped], -5, 5) * vs + vm
    assert bool(((o["value"][clamped].double() - want).abs() <= 1e-6 * want.abs()).all())
    check_nlp(o["neglogp"], o["mu"], o["actions"], logstd)
    assert torch.equal(o["env_actions"], o["actions"].clamp(-1, 1))
    assert 0.02 < float((o["actions"].abs() > 1).double().mean())
    print(f"O={O}: h3 {frac:.2e} of elements differ from float64, by <= {worst:.1f} bf16 ulp; value clamped on "
          f"{float(clamped.double().mean()):.3f} of rows")


@pytest.mark.parametrize("O", [14, 26, 31])
def test_policy_act_u_tile_carries_x_and_h3(O):
    """u_out mode: the U tile is [h3 (64) | x (32) | 0 (32)] per row.  Columns 64..95 are the bf16 x tile bit for bit --
    clamp((obs - mean) inv_std, +-5) in f32 rounded to bf16, zeros from column 64 + O, the constant 1 at column 95 (O = 31:
    right beside the last observation) -- columns 96..127 are zero, h3 matches float64 (check_h3), and the rows of the
    last tile past n are written with x = 0 (no 1) and zeros after it."""
    n = 160 * 128 + 77
    lib, W, obs, mean, inv_std, packed = act_problem(n, O, seed=600 + O)
    U, u = u_tile(lib, packed, obs, mean, inv_std)
    bits = lambda t: t.float().bfloat16().view(torch.int16)  # noqa: E731
    assert torch.equal(bits(u[:, 64:96]), bits(x_tile(obs, mean, inv_std, True)))
    assert float(u[:, 95].min()) == 1.0 and float(u[:, 96:].abs().max()) == 0.0
    assert float(u[:, 64 + O:95].abs().sum()) == 0.0                       # (empty at O = 31)
    assert float((u[:, 64:64 + O].abs() == 5.0).double().mean()) > 0.0     # the clamp is exercised
    frac, worst = check_h3(u[:, :64], forward_ref(W, obs, mean, inv_std), W[4])
    tail = from_tiles(U, U.shape[0] * 128)[n:].double()
    assert float(tail[:, 64:].abs().max()) == 0.0
    print(f"O={O}: h3 {frac:.2e} of elements differ from float64, by <= {worst:.1f} bf16 ulp")


# --------------------------------------------------------------------------------------------------- 3. the update prologue
@pytest.mark.parametrize("count", [65536, 16 * 65536])
@pytest.mark.parametrize("normalize_advantage", [1, 0])
def test_update_prologue_matches_float64_at_the_training_size(count, normalize_advantage):
    """vine_ppo_moments -> vine_ppo_finalize (+ normalize) at the training rollout (16 x 4096 rows) and 16x that: both
    grids are clamped to 148 blocks, so every block runs the grid-stride row loop.  Three iterations against a float64
    RunningMeanStd fed float64 data, with observations, values and returns far from zero (mean 1000, std 1..3), where an
    f32 sum of squares minus n mean^2 would keep about one digit of the variance.
    Tolerances: the moments are f64 sums of f32 inputs (atomics: the order varies), and the variance comes out of
    sumsq - n mean^2, which loses log10(mean^2 / var) = 6 of f64's 16 digits: running mean and var within 1e-9 relative;
    the f32 copies are the f32 rounding of the float64 mean exactly, rsqrtf / sqrtf of the rounded variance within 2e-6;
    in the normalised values and returns x - mean is exact in f32 (Sterbenz: both near 1000), so they carry the f32
    rounding of the mean, 2^-24 |mean| / std, and a few f32 roundings of the result: 6e-8 |mean| / std + 1e-6 (1 + |x_n|);
    returns - values is exact in f32 for the same reason, so the normalised advantage is within 1e-6 (1 + |a_n|), and
    with normalize_advantage = 0 it is returns - values bit for bit.  The moments scratch is zero after every finalize."""
    lib = abi.load_library()
    O = 18
    g = torch.Generator(device=DEV).manual_seed(count + normalize_advantage)
    f = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    obs_rms, val_rms = RunningMeanStd((O,)).to(DEV), RunningMeanStd(()).to(DEV)
    ref_obs, ref_val = RunningMeanStd((O,)).to(DEV), RunningMeanStd(()).to(DEV)
    moments = torch.zeros(2 * O + 4, dtype=torch.float64, device=DEV)
    mean_f, inv_f, vstats, astats, vn, rn, an = f(O), f(O), f(2), f(2), f(count), f(count), f(count)
    for it in range(3):
        obs = torch.randn(count, O, device=DEV, generator=g) * (1 + it) + 1000.0 + 10 * it
        val = torch.randn(count, device=DEV, generator=g) * 3 + 1000.0
        ret = val + torch.randn(count, device=DEV, generator=g) * 2 + 0.5
        a = abi.VinePpoPrologue(
            obs=obs.data_ptr(), values=val.data_ptr(), returns=ret.data_ptr(), moments=moments.data_ptr(),
            obs_mean=obs_rms.running_mean.data_ptr(), obs_var=obs_rms.running_var.data_ptr(), obs_count=obs_rms.count.data_ptr(),
            val_mean=val_rms.running_mean.data_ptr(), val_var=val_rms.running_var.data_ptr(), val_count=val_rms.count.data_ptr(),
            obs_mean_f=mean_f.data_ptr(), obs_inv_std_f=inv_f.data_ptr(), value_stats=vstats.data_ptr(), adv_stats=astats.data_ptr(),
            values_n=vn.data_ptr(), returns_n=rn.data_ptr(), advantages_n=an.data_ptr(), count=count, num_obs=O, world=1,
            normalize_advantage=normalize_advantage)
        assert lib.vine_ppo_moments(C.byref(a), None) == 0 and lib.vine_ppo_finalize(C.byref(a), None) == 0
        torch.cuda.synchronize()
        assert float(moments.abs().max()) == 0.0
        ref_obs.update(obs.double())
        ref_val.update(torch.cat([val, ret]).double())
        for got, want in ((obs_rms.running_mean, ref_obs.running_mean), (obs_rms.running_var, ref_obs.running_var),
                          (val_rms.running_mean, ref_val.running_mean), (val_rms.running_var, ref_val.running_var)):
            assert bool(((got - want).abs() <= 1e-9 * want.abs()).all()), float(((got - want).abs() / want.abs()).max())
        assert float(obs_rms.count) == float(ref_obs.count) and float(val_rms.count) == float(ref_val.count)
        assert torch.equal(mean_f, ref_obs.running_mean.float())
        assert torch.allclose(inv_f.double(), torch.rsqrt(ref_obs.running_var.float().double() + 1e-5), rtol=2e-6, atol=0)
        vm, vsd = float(ref_val.running_mean), math.sqrt(float(ref_val.running_var) + 1e-5)
        assert float(vstats[0]) == float(ref_val.running_mean.float()) and abs(float(vstats[1]) - vsd) <= 2e-6 * vsd
        for x, xn in ((val, vn), (ret, rn)):
            xd = x.double()
            want = torch.clamp((xd - vm) / vsd, -5, 5)
            tol = 6e-8 * abs(vm) / vsd + 1e-6 * (1 + want.abs())
            assert bool(((xn.double() - want).abs() <= tol).all()), float(((xn.double() - want).abs() - tol).max())
        adv = ret.double() - val.double()
        if normalize_advantage:
            want = (adv - adv.mean()) / (adv.std() + 1e-8)
            tol = 1e-6 * (1 + want.abs())
            assert bool(((an.double() - want).abs() <= tol).all()), float(((an.double() - want).abs() - tol).max())
        else:
            assert float(astats[0]) == 0.0 and float(astats[1]) == 1.0
            assert torch.equal(an, ret - val)
