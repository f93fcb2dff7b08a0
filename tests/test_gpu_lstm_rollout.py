"""GPU: the rollout of the recurrent (reference) network -- vine_policy_act (u_out) -> vine_lstm_mask -> vine_lstm_step ->
vine_lstm_head (sampling) -> env step -> vine_rollout_post, PPOAgent._rollout_native_lstm -- against float64 references on
the kernels' own bf16 operands, launch by launch, together with the rollout's bookkeeping (chunk-start snapshots, done
masks, bootstrap value, persistent state) and its hand-off to the first training pass.

As in test_gpu_lstm_update.py, the references start from the decoded tiles (ppo.tiles.from_tiles) and the weights rounded
to bf16 as vine_lstm_pack rounds them, so that only f32 accumulation order, tanh.approx (relative error E < 5e-4), rsqrtf
and the Box-Muller functions separate kernel and reference; each check derives its tolerance from those in its docstring.

The LayerNorm + heads bound (check_head_outputs), per output j of (mu0, mu1, v):
  the f32 row mean and variance are tree sums of 256 terms (8 in-lane + 5 butterfly levels): the mean is off by at most
  8 eps mean|h| (eps = 2^-24), which moves every y_k by that times rstd g_k, coherently; rstd = rsqrtf (2 ulp) of a sum
  with the same relative error; y = fma(h rstd, g, b) and the head dot product (8 FMAs in-lane, 5 butterfly adds, + bias)
  add ~13 eps of sum |y w| + |b|.  So |d_j| <= 1e-5 (sum_k |y_k W_jk| + |b_j|) + 1e-6 mean|h| rstd sum_k |g_k W_jk|,
  the bound check_heads of test_gpu_mlp_update.py uses plus the mean term.  A LayerNorm eps of 1e-6 instead of 1e-5 moves
  the rows of small variance (var ~ 1e-5 below) by percents.

The noise: vine_lstm_head draws z = normal4(philox(key = seed, counter = (global_env_offset + s, 16, rng_counter, 0)))[:2]
exactly as oracle.normal4 does; the kernel's logf / sqrtf / Cephes sin-cos and the oracle's libm logf / sqrtf / sinf / cosf
agree to a few f32 ulp of the radius r = |z| <= 5.8: |dz| <= 2e-6 (1 + r).  A wrong key half, site or counter moves z by
O(1) on every row."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import vine_robot_isaacgymenvs_b200 as vine
from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200 import config as vcfg
from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles, to_tiles
from test_gpu_lstm_update import (E_TANH, SENT_BF16, SENT_F32, TB, bf16_ulp, bits, make_params, pack, step_inputs,
                                  step_outputs)
from test_gpu_mlp_update import forward_ref, x_tile
from test_gpu_ppo_fused import _act_problem, _act

pytestmark = pytest.mark.gpu
DEV = "cuda"
SITE_POLICY = 16
WORST = {}     # quantity -> worst measured error (in the unit named by the key), printed by every test


def note(key, x):
    WORST[key] = max(WORST.get(key, 0.0), float(x))


def report(tag):
    print(tag, {k: f"{v:.2e}" for k, v in sorted(WORST.items())})


def f32_ulp(x):
    """one f32 ulp at |x| (float64 tensor)."""
    e = torch.frexp(x.abs().clamp_min(2.0 ** -126))[1]
    return torch.ldexp(torch.ones_like(x), e - 24)


def fused_value(v, vstats):
    """The rollout's value, fma(clamp(v, +-5), std, mean) in f32 (vine_lstm_head compiles it to one FFMA): the product of
    two f32 numbers is exact in float64, so float64 sum then one rounding to f32 is the fused result (a double-rounding
    tie would need the float64 sum to land within 2^-53 of an f32 midpoint)."""
    vm, vs = float(vstats[0]), float(vstats[1])
    return (v.double().clamp(-5.0, 5.0) * vs + vm).float()


# ------------------------------------------------------------------------------------------------------------ references
def oracle_z(seed, goff, n, ctr):
    """[n, 2] f32: the first two normals of oracle.normal4(seed, goff + s, 16, ctr, 0) for every row s."""
    from oracle import oracle
    f = oracle.lib().oracle_normal4
    buf = (C.c_float * 4)()
    out = np.empty((n, 2), dtype=np.float32)
    for s in range(n):
        f(seed, (goff + s) & 0xFFFFFFFF, SITE_POLICY, ctr, 0, buf)
        out[s, 0], out[s, 1] = buf[0], buf[1]
    return torch.from_numpy(out).to(DEV)


def head_ref(Pd, hq):
    """float64 LayerNorm (biased variance, eps 1e-5) -> heads on the decoded h; -> ([n, 3] mu0 mu1 v, [n, 3] bound)."""
    mean = hq.mean(-1, keepdim=True)
    var = ((hq - mean) ** 2).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + 1e-5)
    y = (hq - mean) * rstd * Pd["ln_g"] + Pd["ln_b"]
    W = torch.cat([Pd["w_mu"], Pd["w_v"]])                       # [3, 256]
    bh = torch.cat([Pd["b_mu"], Pd["b_v"]])
    out = y @ W.t() + bh
    tol = 1e-5 * (y.abs() @ W.abs().t() + bh.abs()) + 1e-6 * hq.abs().mean(-1, keepdim=True) * rstd * (Pd["ln_g"].abs() @ W.abs().t())
    return out, tol


def check_head_outputs(o, hq, Pd, vstats, logstd, z=None, tag=""):
    """Rollout-mode vine_lstm_head outputs o (mu, value, and with z: actions, neglogp, env_actions, all [n] rows) against
    float64 on the kernel's own h (see the module docstring for the LayerNorm / heads bound and |dz|).
      mu: the head bound.
      value: fma(clamp(v), std, mean) -- rows whose float64 v is beyond +-5 by more than the bound must hold exactly the
        f32 fma of +-5; the others give back v = (value - mean) / std within the bound + one ulp(value) / std.
      actions = fma(__expf(logstd), z, mu): within sigma (4e-7 |z| (__expf: <= 3 ulp at |logstd| < 1) + |dz|) + one
        ulp(action) of the kernel's mu + exp(logstd) z_oracle.
      neglogp = 0.5 |z|^2 + log(2 pi) + sum logstd in f32: within |z| |dz| + 1e-6 (1 + |nlp|) (a few f32 roundings and the
        f32 constant) of float64 on z_oracle: 4e-6 (1 + r)^2 + 1e-6 (1 + |nlp|).
      env_actions = clamp(actions, +-1) bit for bit."""
    ref, tol = head_ref(Pd, hq)
    mu = o["mu"].double()
    err = (mu - ref[:, :2]).abs()
    assert bool((err <= tol[:, :2]).all()), (tag, "mu", float((err - tol[:, :2]).max()))
    note("mu / bound", float((err / tol[:, :2]).max()))
    note("mu abs", float(err.max()))
    vm, vs = float(vstats[0]), float(vstats[1])
    v_ref, tv = ref[:, 2], tol[:, 2]
    value = o["value"]
    hi, lo = v_ref > 5.0 + tv, v_ref < -5.0 - tv
    inside = v_ref.abs() < 5.0 - tv
    five = fused_value(torch.tensor([5.0, -5.0], device=DEV), vstats)
    assert bool((value[hi] == five[0]).all()) and bool((value[lo] == five[1]).all()), (tag, "clamped value")
    v_k = (value.double() - vm) / vs
    ev = (v_k - v_ref).abs()[inside]
    bv = tv[inside] + f32_ulp(value.double())[inside] / vs
    assert bool((ev <= bv).all()), (tag, "value", float((ev - bv).max()))
    note("v / bound", float((ev / bv).max()))
    frac = {"v>5": float(hi.double().mean()), "v<-5": float(lo.double().mean())}
    if z is None:
        return frac
    ls = logstd.double()
    sig = torch.exp(ls)
    zd = z.double()
    r = zd.norm(dim=-1, keepdim=True)
    act_ref = mu + sig * zd
    act = o["actions"].double()
    dz = 2e-6 * (1 + r)
    ba = sig * (4e-7 * zd.abs() + dz) + f32_ulp(act)
    ea = (act - act_ref).abs()
    assert bool((ea <= ba).all()), (tag, "actions", float((ea - ba).max()), float(ea.max()))
    note("actions / bound", float((ea / ba).max()))
    nlp_ref = 0.5 * (zd * zd).sum(-1) + math.log(2 * math.pi) + ls.sum()
    bn = 4e-6 * (1 + r[:, 0]) ** 2 + 1e-6 * (1 + nlp_ref.abs())
    en = (o["neglogp"].double() - nlp_ref).abs()
    assert bool((en <= bn).all()), (tag, "neglogp", float((en - bn).max()))
    note("neglogp / bound", float((en / bn).max()))
    assert torch.equal(o["env_actions"], o["actions"].clamp(-1.0, 1.0)), tag
    frac.update({"act>1": float((o["actions"] > 1).double().mean()), "act<-1": float((o["actions"] < -1).double().mean())})
    return frac


def step_ref(P, u, hm, c_prev, nd, O):
    """float64 LSTM cell on the decoded U / HM tiles and the bf16 weights; -> c, h, and the per-element bounds of
    test_gpu_lstm_update.test_lstm_step_y2_grid_matches_float64 (c: E (|c_prev m| / 2 + 3 |g| / 2) + 2e-5; h: one bf16 ulp
    + 3 E |tanh c| / 2 + bound(c))."""
    wih, whh = P["w_ih"].bfloat16().double(), P["w_hh"].bfloat16().double()
    gates = u[:, :64 + O] @ wih.t() + hm @ whh.t() + (P["b_ih"] + P["b_hh"]).double()
    gi, gf, gg, go = gates.chunk(4, -1)
    i, f, g, og = torch.sigmoid(gi), torch.sigmoid(gf), torch.tanh(gg), torch.sigmoid(go)
    cpm = c_prev.double() * nd.double()[:, None]
    c = f * cpm + i * g
    tc = torch.tanh(c)
    h = og * tc
    bc = E_TANH * (0.5 * cpm.abs() + 1.5 * g.abs()) + 2e-5
    return c, h, bc, bf16_ulp(h) + 1.5 * E_TANH * tc.abs() + bc


def check_step(P, u, hm, c_prev, nd, c_k, hh_k, O, tag=""):
    """vine_lstm_step's c (f32) and h (bf16 tile) against step_ref; -> fraction of rows whose h differs from bf16(float64 h)
    (a bf16 rounding flip: the f32 h within tanh.approx noise of a rounding boundary)."""
    n = c_prev.shape[0]
    c, h, bc, bh = step_ref(P, u, hm, c_prev, nd, O)
    err_c = (c_k[:n].double() - c).abs()
    assert bool((err_c <= bc).all()), (tag, "c", float((err_c - bc).max()))
    note("c abs", float(err_c.max()))
    hh = from_tiles(hh_k, n).double()
    err_h = (hh - h).abs()
    assert bool((err_h <= bh).all()), (tag, "h", float((err_h - bh).max()))
    note("h / bound", float((err_h / bh).max()))
    flips = (hh != h.float().bfloat16().double()).any(-1)
    frac = float(flips.double().mean())
    note("rows with an h flip", frac)
    return frac


# ------------------------------------------------------------------------------------------------------ 1. vine_lstm_head
def head_case(n, seed):
    """h rows tanh(a (x + s)) with a log-uniform in [3e-3, 1] (row variance from ~1e-5, where the LayerNorm eps
    matters, to ~0.3) and a row offset s ~ 0.3 N(0, 1); non-trivial LayerNorm and heads, the value weights scaled so that
    |v| > 5 on a real fraction of rows of both signs."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    P = make_params(18, seed)
    P["w_v"] = P["w_v"] * 6.0
    P["b_mu"] = torch.tensor([0.3, -0.2], device=DEV)
    a = torch.exp(torch.rand(n, 1, device=DEV, generator=g) * math.log(1 / 3e-3)) * 3e-3
    h = torch.tanh(a * (torch.randn(n, 256, device=DEV, generator=g) + 0.3 * torch.randn(n, 1, device=DEV, generator=g)))
    HH = to_tiles(h)
    return P, HH, from_tiles(HH, n).double()


def head_outputs(n, sample=True):
    z = lambda *s: torch.full((n + 1, *s), SENT_F32, device=DEV)  # noqa: E731  (row n: must keep the sentinel)
    return dict(mu=z(2), value=z(), actions=z(2), neglogp=z(), env_actions=z(2))


def run_head(lib, lp, HH, n, vstats, o, logstd=None, counter=None, seed=0, goff=0):
    hd = abi.VineLstmHead(params=lp.data_ptr(), hh=HH.data_ptr(), value_stats=vstats.data_ptr(), value=o["value"].data_ptr(), n=n)
    if logstd is not None:
        hd.mu, hd.logstd, hd.rng_counter = o["mu"].data_ptr(), logstd.data_ptr(), counter.data_ptr()
        hd.actions, hd.neglogp, hd.env_actions = o["actions"].data_ptr(), o["neglogp"].data_ptr(), o["env_actions"].data_ptr()
        hd.seed, hd.global_env_offset = seed, goff
    assert lib.vine_lstm_head(C.byref(hd), None) == 0
    torch.cuda.synchronize()


HEAD_CASES = [(4096, 0x5DEECE66D ^ 42, 0, 0), (9472, 0x5DEECE66D ^ 7, 0, 3),
              (9600, 0x9E3779B97F4A7C15, 123456, 0x10000 + 5), (65536, 0x5DEECE66D ^ 42, 0, 1)]


@pytest.mark.parametrize("n,seed,goff,ctr", HEAD_CASES, ids=["4096", "9472", "9600_seed64_offset_counter", "65536"])
def test_lstm_head_rollout_matches_float64_and_the_oracle_noise(n, seed, goff, ctr):
    """vine_lstm_head in rollout mode at 4096 rows, 9472 (the last size without a grid stride: 148 x 8 warps), 9600 (the
    first with one: the first 128 warps take a second row) and 65,536 (7 rows per warp), against float64 on its own bf16 h
    (check_head_outputs): mu, value (clamped on a real fraction of rows of both signs), the noise against oracle.normal4
    at site 16 -- the 9600 case with a seed whose high half is non-zero, global_env_offset != 0 and a counter above 2^16 --,
    neglogp, env_actions.  Row n of every output keeps its sentinel.  Then the bootstrap-value mode (only value passed):
    the same value bits, and nothing else written."""
    lib = abi.load_library()
    P, HH, hq = head_case(n, n + 11)
    lp = pack(lib, P, 18)
    Pd = {k: v.double() for k, v in P.items()}
    vstats = torch.tensor([0.3, 1.7], device=DEV)
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    counter = torch.tensor([ctr], dtype=torch.int32, device=DEV)
    o = head_outputs(n)
    run_head(lib, lp, HH, n, vstats, o, logstd, counter, seed, goff)
    for k, t in o.items():
        assert bool((t[n] == SENT_F32).all()), f"{k}: row n written"
        assert not bool((t[:n] == SENT_F32).any()), f"{k}: a row below n not written"
    z = oracle_z(seed, goff, n, ctr)
    frac = check_head_outputs({k: t[:n] for k, t in o.items()}, hq, Pd, vstats, logstd, z, tag=f"n={n}")
    assert min(frac.values()) > 0.02, frac
    boot = head_outputs(n)
    run_head(lib, lp, HH, n, vstats, boot)
    assert torch.equal(bits(boot["value"]), bits(o["value"]))
    for k in ("mu", "actions", "neglogp", "env_actions"):
        assert bool((boot[k] == SENT_F32).all()), k
    print(f"n={n}: fractions {frac}")
    report(f"head n={n}")


def test_policy_act_noise_is_the_oracle_stream():
    """vine_policy_act (the MLP network's rollout) draws its noise from the same key layout as vine_lstm_head: z =
    oracle.normal4(seed, global_env_offset + e, 16, rng_counter, 0)[:2], checked through actions = fma(__expf(logstd), z,
    mu) with the bound of check_head_outputs, for a 64-bit seed, an env offset and a counter."""
    n, O = 3000, 18
    lib, W, obs, mean, inv_std, packed = _act_problem(n, O, seed=9)
    logstd = torch.tensor([-0.3, 0.2], device=DEV)
    counter = torch.tensor([77], dtype=torch.int32, device=DEV)
    seed, goff = 0x9E3779B97F4A7C15, 5000
    o = _act(lib, packed, obs, mean, inv_std, logstd, counter, n, O, offset=goff, seed=seed)
    z = oracle_z(seed, goff, n, 77).double()
    sig = torch.exp(logstd.double())
    ref = o["mu"].double() + sig * z
    act = o["actions"].double()
    bound = sig * (4e-7 * z.abs() + 2e-6 * (1 + z.norm(dim=-1, keepdim=True))) + f32_ulp(act)
    err = (act - ref).abs()
    assert bool((err <= bound).all()), float((err - bound).max())
    print(f"policy_act noise: worst |a - a_ref| / bound {float((err / bound).max()):.2e}")


# ------------------------------------------------------------------------------------- 2. vine_lstm_mask, rollout-form step
@pytest.mark.parametrize("n", [4096, 4837])
def test_lstm_mask_is_bf16_h_times_not_done(n):
    """vine_lstm_mask: HM = bf16(HH nd) bit for bit over every tile, the sign included (h nd with nd = 0 is -0 for a
    negative h), and the rows of the last tile past n multiplied by 0 (4837: 27 such rows, holding junk in HH)."""
    lib = abi.load_library()
    g = torch.Generator(device=DEV).manual_seed(n)
    tiles = (n + 127) // 128
    h = torch.randn(tiles * 128, 256, device=DEV, generator=g)
    HH = to_tiles(h)
    nd = (torch.rand(n, device=DEV, generator=g) > 0.3).float()
    HM = torch.full_like(HH, SENT_BF16)
    assert lib.vine_lstm_mask(C.c_void_p(HH.data_ptr()), C.c_void_p(nd.data_ptr()), n, C.c_void_p(HM.data_ptr()), None) == 0
    torch.cuda.synchronize()
    m = torch.zeros(tiles * 128, device=DEV)
    m[:n] = nd
    want = to_tiles(from_tiles(HH, tiles * 128) * m[:, None])
    assert torch.equal(bits(HM), bits(want))
    hm = from_tiles(HM, tiles * 128)
    assert bool((torch.signbit(hm[:n][nd == 0]) == (from_tiles(HH, n)[nd == 0] < 0)).all())   # -0 for negative h
    assert float(hm[n:].abs().max() if n % 128 else 0.0) == 0.0


@pytest.mark.parametrize("n", [4096, 16384])
def test_lstm_step_rollout_form_matches_float64(n):
    """vine_lstm_step as the rollout calls it -- act, hm_next and not_done_next null -- at 4096 envs (32 tiles, the y = 4
    grid) and 16,384 (128 tiles, y = 2), against float64 with the per-element bounds of
    test_lstm_step_y2_grid_matches_float64 (step_ref).  The omitted buffers keep their sentinels, and c / hh equal the
    training form's (all pointers given) bit for bit."""
    lib = abi.load_library()
    O = 18
    P = make_params(O, n + 3)
    lp = pack(lib, P, O)
    x = step_inputs(n, O, n + 4)
    o, full = step_outputs(n), step_outputs(n)
    a = abi.VineLstmStep(params=lp.data_ptr(), u=x["U"].data_ptr(), hm=x["HM"].data_ptr(), c_prev=x["c_prev"].data_ptr(),
                         not_done=x["nd"].data_ptr(), c=o["c"].data_ptr(), hh=o["HH"].data_ptr(), n=n)
    assert lib.vine_lstm_step(C.byref(a), None) == 0
    b = abi.VineLstmStep(params=lp.data_ptr(), u=x["U"].data_ptr(), hm=x["HM"].data_ptr(), c_prev=x["c_prev"].data_ptr(),
                         not_done=x["nd"].data_ptr(), not_done_next=x["nd_next"].data_ptr(), c=full["c"].data_ptr(),
                         hh=full["HH"].data_ptr(), hm_next=full["HMn"].data_ptr(), act=full["ACT"].data_ptr(), n=n)
    assert lib.vine_lstm_step(C.byref(b), None) == 0
    torch.cuda.synchronize()
    assert bool((o["HMn"] == SENT_BF16).all()) and bool((o["ACT"] == SENT_BF16).all())
    assert torch.equal(bits(o["c"]), bits(full["c"])) and torch.equal(bits(o["HH"]), bits(full["HH"]))
    tiles = n // 128
    u = from_tiles(x["U"].view(tiles, 1, TB), n).double()
    frac = check_step(P, u, from_tiles(x["HM"], n).double(), x["c_prev"], x["nd"], o["c"], o["HH"], O, tag=f"n={n}")
    print(f"n={n}: {frac:.2e} of rows have an h element one bf16 flip off float64")
    report(f"step n={n}")


# ------------------------------------------------------------------------------------------- 3. the agent's rollout, recorded
class RecordingLib:
    """The agent's library with the rollout's launches recorded: after each vine_policy_act (u_out), vine_lstm_mask,
    vine_lstm_step, vine_lstm_head and vine_rollout_post it clones, on the current stream, what the launch read and wrote.
    Every other symbol passes through."""

    def __init__(self, agent):
        self._lib, self._a = agent._lib, agent
        self.events = []

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def _which(self, bufs, ptr):
        for i, t in enumerate(bufs):
            if t.data_ptr() == ptr:
                return i
        raise AssertionError(f"unexpected pointer {ptr:#x}")

    def vine_policy_act(self, ref, stream):
        rc = self._lib.vine_policy_act(ref, stream)
        a = self._a
        if ref._obj.u_out:
            self.events.append(("act", dict(U=a._r_U.clone(), obs=a.env._obs_clamped.clone(),
                                             obs_copy=ref._obj.obs_copy)))
        return rc

    def vine_lstm_mask(self, hh, nd, n, hm, stream):
        rc = self._lib.vine_lstm_mask(hh, nd, n, hm, stream)
        a = self._a
        i = self._which(a._r_HH, hh.value)
        self.events.append(("mask", dict(HH_in=a._r_HH[i].clone(), HM=a._r_HM.clone(),
                                         nd_row=(nd.value - a._nd_ext.data_ptr()) // (4 * a.n))))
        return rc

    def vine_lstm_step(self, ref, stream):
        rc = self._lib.vine_lstm_step(ref, stream)
        a, s = self._a, ref._obj
        assert not s.act and not s.hm_next and not s.not_done_next
        ip, io = self._which(a._r_C, s.c_prev), self._which(a._r_C, s.c)
        assert self._which(a._r_HH, s.hh) == io != ip
        self.events.append(("step", dict(c_prev=a._r_C[ip].clone(), c=a._r_C[io].clone(), HH=a._r_HH[io].clone())))
        return rc

    def vine_lstm_head(self, ref, stream):
        a, s = self._a, ref._obj
        ctr = a._rng_counter.clone()
        rc = self._lib.vine_lstm_head(ref, stream)
        boot = not s.actions
        if boot:
            assert s.value == a.last_value.data_ptr() and not s.mu and not s.neglogp and not s.env_actions
            self.events.append(("head", dict(boot=True, value=a.last_value.clone())))
        else:
            t = (s.mu - a.b_mu.data_ptr()) // (8 * a.n)
            for name, buf, w in (("value", a.b_val, 4), ("actions", a.b_act, 8), ("neglogp", a.b_nlp, 4)):
                assert getattr(s, name) == buf.data_ptr() + t * w * a.n, name
            assert s.env_actions == a.env.actions.data_ptr()
            self.events.append(("head", dict(boot=False, t=t, ctr=ctr, seed=s.seed, goff=s.global_env_offset,
                                             mu=a.b_mu[t].clone(), value=a.b_val[t].clone(), actions=a.b_act[t].clone(),
                                             neglogp=a.b_nlp[t].clone(), env_actions=a.env.actions.clone())))
        return rc

    def vine_rollout_post(self, ref, stream):
        rc = self._lib.vine_rollout_post(ref, stream)
        a = self._a
        self.events.append(("post", dict(resets=a.env.reset_buf.clone(), nd=a._nd_ext.clone())))
        return rc

    def steps(self):
        """events grouped into one dict per rollout step (act, mask, step, head[, post])."""
        out, cur = [], None
        for kind, d in self.events:
            if kind == "act":
                cur = {}
                out.append(cur)
            assert kind not in cur, kind
            cur[kind] = d
        return out


def check_u_h3(h3_k, fwd, W):
    """The rollout's h3 (U columns 0..63) against the float64 forward.  As check_h3 of test_gpu_mlp_update.py: fewer than
    1 % of the elements may differ from float64 (a wrong weight, bias or column moves nearly all of them).  The bound per
    element follows a bf16 flip (one ulp) of any element through the layers above it: h1 flips move h2 by |W2| ulp(h1),
    h2 flips and those moves reach h3 through |W3|, so |dh3| <= 2 ulp(h3) + |W3| (2 ulp(h2) + |W2| 2 ulp(h1)).  On the
    env's observations several elements of one row can sit near a rounding boundary at once, which the single-flip bound
    of check_h3 does not cover."""
    bfd = lambda t: t.detach().float().bfloat16().double()  # noqa: E731
    w2, w3 = bfd(W[2]).abs(), bfd(W[4]).abs()
    d = (h3_k - fwd["h3"]).abs()
    tol = 2 * bf16_ulp(fwd["h3"]) + (2 * bf16_ulp(fwd["h2"]) + (2 * bf16_ulp(fwd["h1"])) @ w2.t()) @ w3.t()
    frac = float((d > 0).double().mean())
    assert frac < 1e-2, frac
    assert bool((d <= tol).all()), float((d - tol).max())
    note("h3 elements off float64", frac)


def rollout_agent(n, extra=()):
    """FSTR with the reference network on the kernel path, a non-trivial LayerNorm, log-std and observation normaliser."""
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True"] + list(extra))
    agent = PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=1, use_graphs=False)
    assert agent.native_lstm
    g = torch.Generator(device=DEV).manual_seed(n)
    m = agent.model
    with torch.no_grad():
        m.layer_norm.weight.copy_(0.5 + torch.rand(256, device=DEV, generator=g))
        m.layer_norm.bias.copy_(0.1 * torch.randn(256, device=DEV, generator=g))
        m.value.weight.mul_(4.0)
        m.sigma.copy_(torch.tensor([-0.4, 0.1], device=DEV))
        agent.obs_rms.running_mean.copy_(0.2 * torch.randn(agent.O, device=DEV, generator=g).double())
        agent.obs_rms.running_var.copy_((0.3 + torch.rand(agent.O, device=DEV, generator=g)).double())
        agent.val_rms.running_mean.fill_(0.4)
        agent.val_rms.running_var.fill_(2.5)
    agent._refresh_fused(pack=True)
    agent._rollout()       # the first step resets every env (reset_buf starts at 1): from here on progress can be set
    torch.cuda.synchronize()
    return agent


def set_timeouts(agent):
    """progress so that the k-th env not already flagged for a reset times out at step k mod T of the next rollout (~1/T
    of the envs at every step, including the last step of every seq_len chunk): the step increments progress first and
    resets at progress >= maxEpisodeLength - 1; an env flagged in reset_buf restarts from progress 0 instead."""
    env, T = agent.env, agent.T
    free = env.reset_buf == 0
    k = torch.cumsum(free.long(), 0) - 1
    env.progress_buf.copy_(torch.where(free, int(env.max_episode_length) - 2 - (k % T), env.progress_buf))


def lstm_params(agent):
    m, r = agent.model, agent.model.rnn.rnn
    P = dict(w_ih=r.weight_ih_l0, w_hh=r.weight_hh_l0, b_ih=r.bias_ih_l0, b_hh=r.bias_hh_l0, ln_g=m.layer_norm.weight,
             ln_b=m.layer_norm.bias, w_mu=m.mu.weight, b_mu=m.mu.bias, w_v=m.value.weight, b_v=m.value.bias)
    return {k: v.detach().clone() for k, v in P.items()}


def mlp_weights(agent):
    m = agent.model
    z = lambda *s: torch.zeros(*s, device=DEV)  # noqa: E731
    return [t.detach() for t in (m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias,
                                 m.actor_mlp[4].weight, m.actor_mlp[4].bias)] + [z(2, 64), z(2), z(1, 64), z(1)]


def recorded_rollout(agent):
    rec = RecordingLib(agent)
    lib, agent._lib = agent._lib, rec
    try:
        agent._rollout()
    finally:
        agent._lib = lib
    torch.cuda.synchronize()
    return rec.steps()


def check_rollout(agent, steps, state0, tag):
    """Every launch of one recorded rollout against float64 and the bookkeeping bit for bit.  ``state0`` = (HH, C, nd_T)
    the persistent state and the done row the previous rollout ended with (None for the first)."""
    n, T, L, O = agent.n, agent.T, agent.seq_len, agent.O
    assert len(steps) == T + 1
    P = lstm_params(agent)
    Pd = {k: v.double() for k, v in P.items()}
    W = mlp_weights(agent)
    mean, inv_std, vstats, logstd = agent._obs_mean_f, agent._obs_inv_std_f, agent._val_stats, agent.model.sigma.detach()
    nd_ext = agent._nd_ext
    tiles = n // 128
    seed, goff = int(agent.env._seed) ^ 0x5DEECE66D, int(agent.env._global_env_offset)
    if state0 is not None:
        assert torch.equal(bits(steps[0]["mask"]["HH_in"]), bits(state0[0]))
        assert torch.equal(bits(steps[0]["step"]["c_prev"]), bits(state0[1]))
        assert torch.equal(nd_ext[0], 1.0 - state0[2])          # row 0 carries the previous iteration's last dones
    flips = []
    for t, s in enumerate(steps):
        last = t == T
        # U: x bit for bit, h3 as check_h3
        obs = s["act"]["obs"]
        if not last:
            assert torch.equal(agent.b_obs[t], obs), (tag, t)
        u = from_tiles(s["act"]["U"].view(tiles, 1, TB), n).double()
        assert torch.equal(u[:, 64:96].float().bfloat16().view(torch.int16),
                           x_tile(obs, mean, inv_std, True).float().bfloat16().view(torch.int16)), (tag, t)
        check_u_h3(u[:, :64], forward_ref(W, obs, mean, inv_std), W)
        # HM = bf16(HH_{t-1} nd_ext[t]); the state entering step t is the one step t - 1 left
        mk = s["mask"]
        assert mk["nd_row"] == t, (tag, t, mk["nd_row"])
        hh_in = mk["HH_in"]
        if t > 0:
            assert torch.equal(bits(hh_in), bits(steps[t - 1]["step"]["HH"])), (tag, t)
            assert torch.equal(bits(s["step"]["c_prev"]), bits(steps[t - 1]["step"]["c"])), (tag, t)
        want = to_tiles(from_tiles(hh_in, n) * nd_ext[t][:, None])
        assert torch.equal(bits(mk["HM"]), bits(want)), (tag, t, "HM")
        # c, h against float64
        flips.append(check_step(P, u, from_tiles(mk["HM"], n).double(), s["step"]["c_prev"], nd_ext[t], s["step"]["c"],
                                s["step"]["HH"], O, tag=f"{tag} t={t}"))
        hq = from_tiles(s["step"]["HH"], n).double()
        hd = s["head"]
        if last:
            assert hd["boot"]
            assert torch.equal(bits(agent.last_value), bits(hd["value"]))
            check_head_outputs(dict(value=agent.last_value, mu=torch.zeros(n, 2, device=DEV)), hq,
                               dict(Pd, w_mu=torch.zeros_like(Pd["w_mu"]), b_mu=torch.zeros_like(Pd["b_mu"])), vstats, logstd)
            break
        assert not hd["boot"] and hd["t"] == t and hd["seed"] == seed and hd["goff"] == goff
        z = oracle_z(seed, goff, n, int(hd["ctr"]))
        check_head_outputs(hd, hq, Pd, vstats, logstd, z, tag=f"{tag} t={t}")
        # the buffers hold what the head wrote
        for k, buf in (("mu", agent.b_mu), ("value", agent.b_val), ("actions", agent.b_act), ("neglogp", agent.b_nlp)):
            assert torch.equal(bits(buf[t]), bits(hd[k])), (tag, t, k)
        # the done mask of the next step is 1 - this step's resets, ~1/T of them timeouts
        resets = s["post"]["resets"]
        assert torch.equal(nd_ext[t + 1], 1.0 - resets.float()), (tag, t)
        assert float(resets.float().mean()) >= 0.8 / T, (tag, t, float(resets.float().mean()))
        if t > 0:
            assert int(hd["ctr"]) == int(steps[t - 1]["head"]["ctr"]) + 1
    # chunk-start snapshots: the unmasked state entering step k L
    for k in range(T // L):
        assert torch.equal(bits(agent._HH_saved[k]), bits(steps[k * L]["mask"]["HH_in"])), (tag, "HH_saved", k)
        assert torch.equal(bits(agent._C_saved[k]), bits(steps[k * L]["step"]["c_prev"])), (tag, "C_saved", k)
    # the persistent state is the one after step T - 1, in buffer 0; the bootstrap step does not advance it
    assert agent._r_cur == 0
    assert torch.equal(bits(agent._r_HH[0]), bits(steps[T - 1]["step"]["HH"])), (tag, "persistent h")
    assert torch.equal(bits(agent._r_C[0]), bits(steps[T - 1]["step"]["c"])), (tag, "persistent c")
    return max(flips)


ROLLOUT_CASES = {"4096": (4096, []), "16384": (16384, []),
                 "odd_T15_L5": (4096, ["train.params.config.horizon_length=15", "train.params.config.seq_len=5",
                                       "train.params.config.minibatch_size=30720"])}


@pytest.mark.parametrize("case", list(ROLLOUT_CASES))
def test_native_lstm_rollout_launch_by_launch(case):
    """PPOAgent._rollout_native_lstm on the real env (FSTR, reference network) at 4096 envs (programmatic dependent
    launch, y = 4 step grid), 16,384 (plain launches, y = 2, the head's grid stride) and an odd horizon (T = 15, seq_len
    5: the persistent state comes back into buffer 0 by the final copy), two consecutive rollouts each, with ~1/T of the
    envs timing out at every step.  Per step, on the operands the launches actually read (recorded by RecordingLib): U's x
    columns bit for bit and its h3 (check_u_h3, rollout-time observation statistics), HM = bf16(HH_{t-1} _nd_ext[t]) bit for
    bit, c and h (check_step), mu / value / actions / neglogp / env_actions (check_head_outputs, noise from
    oracle.normal4 at the counter of the launch), _nd_ext[t + 1] = 1 - resets_t, and b_mu / b_val / b_act / b_nlp[t] =
    what the head wrote.  Bookkeeping bit for bit: _HH_saved[k] / _C_saved[k] = the unmasked state entering step k L,
    last_value = the head on the extra step T, _r_HH[0] / _r_C[0] = the state after step T - 1; the second rollout starts
    from that state, and its _nd_ext[0] is the first one's last done row."""
    n, extra = ROLLOUT_CASES[case]
    agent = rollout_agent(n, extra)
    assert (n <= agent.PDL_MAX_ENVS) == (n == 4096)
    if case.startswith("odd"):
        assert agent.T % 2 == 1 and agent.seq_len == 5
    state0 = (agent._r_HH[0].clone(), agent._r_C[0].clone(), agent._done_ext[agent.T].clone())   # after rollout_agent's
    for it in range(2):
        set_timeouts(agent)
        steps = recorded_rollout(agent)
        worst_flip = check_rollout(agent, steps, state0, tag=f"{case} it={it}")
        if it == 1:
            assert float(agent._nd_ext[0].min()) == 0.0        # the first rollout's timeouts at its last step
        state0 = (agent._r_HH[0].clone(), agent._r_C[0].clone(), agent._done_ext[agent.T].clone())
        print(f"{case} iteration {it}: at most {worst_flip:.2e} of the rows of a step have an h element one bf16 flip off float64")
    report(case)


# ------------------------------------------------------------------------------------------- 4. rollout -> update hand-off
def test_first_training_pass_reproduces_the_rollout():
    """After a rollout at 4096 envs (T = 16, seq_len 4, minibatch 2 x 2048 envs), vine_lstm_gather + NativeLstmPath.
    gradients for both minibatch slots of the first mini-epoch, with the rollout-time observation and value statistics
    and no Adam step in between, recompute the rollout's forward: the MLP, the LSTM steps from the chunk-start snapshots
    and the head run on the same operands in the same order (vine_lstm_head and vine_lstm_head_train sum the LayerNorm
    and the heads identically), so
      debug_out mu == b_mu bit for bit for every row;
      fma(clamp(debug_out v), std, mean) == b_val bit for bit (vine_lstm_head evaluates the value affine as one FFMA;
        fused_value rounds once like it);
      debug_out nlp = 0.5 |(a - mu) / sigma|^2 + ... vs b_nlp = 0.5 |z|^2 + ...: a = fma(sigma, z, mu) rounds once,
        (a - mu) and the multiplication by 1 / sigma once each, so each e_j = z_j (1 + 3 eps) + ulp(a_j) / (2 sigma_j)
        and |d nlp| <= sum_j |z_j| (ulp(a_j) / sigma_j + 4 eps |z_j|) + 8 ulp(nlp) (four roundings of each side's sum),
        z from b_act;
      the KL statistic (mu_old = mu, sigma_old = sigma) is the identical-policy value sum_j log(1 + 1e-5) +
        sigma_j^2 / (2 (sigma_j^2 + 1e-5)) - 1/2 of every row: within 1e-6 absolute (__logf's lg2.approx, ~1e-7 per
        dimension, and a few ulp of the O(1/2) terms that cancel to O(1e-5))."""
    from vine_robot_isaacgymenvs_b200.ppo.lstm_native import NativeLstmPath  # noqa: F401
    agent = rollout_agent(4096, ["train.params.config.minibatch_size=32768"])
    set_timeouts(agent)
    agent._rollout()
    torch.cuda.synchronize()
    T, n, L, E, lib = agent.T, agent.n, agent.seq_len, agent.mb_envs, agent._lib
    chunks = T // L
    assert E == 2048 and n // E == 2
    path = agent._path
    scal = torch.cat([agent.b_act, agent.b_mu, agent.b_nlp[..., None], agent.b_val[..., None],
                      torch.zeros(T, n, 2, device=DEV)], -1).contiguous()
    sigma = agent.model.sigma.detach().clone()
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    state[0] = 3e-4
    flat_before = agent.flat_l.clone()
    worst = {"nlp / bound": 0.0, "kl abs": 0.0}
    for e0 in range(0, n, E):
        ga = abi.VineLstmGather(obs=agent.b_obs.data_ptr(), scalars=scal.data_ptr(), not_done=agent._nd_ext.data_ptr(),
                                c_saved=agent._C_saved.data_ptr(), hh_saved=agent._HH_saved.data_ptr(),
                                mb_obs=agent._mb_obs.data_ptr(), mb_scalars=agent._mb_scal.data_ptr(),
                                mb_not_done=agent._mb_nd.data_ptr(), c0=path.C0.data_ptr(), hm0=path.HM[0].data_ptr(),
                                seq_len=L, chunks=chunks, num_envs=n, env_begin=e0, env_count=E, num_obs=agent.O)
        assert lib.vine_lstm_gather(C.byref(ga), None) == 0
        dbg = torch.full((L * chunks * E, 4), SENT_F32, device=DEV)
        path.gradients(agent._packed, agent._lpacked, agent._mb_obs, agent._mb_scal, agent._mb_nd, agent._obs_mean_f,
                       agent._obs_inv_std_f, agent._val_stats, sigma, sigma.clone(), state, debug_out=dbg)
        torch.cuda.synchronize()

        def rows(buf):   # [T, N, ...] -> the minibatch's row order [step in chunk][chunk, env]
            return buf.view(chunks, L, n, -1)[:, :, e0:e0 + E].permute(1, 0, 2, 3).reshape(L * chunks * E, -1)
        mu, val, act, nlp = rows(agent.b_mu), rows(agent.b_val)[:, 0], rows(agent.b_act), rows(agent.b_nlp)[:, 0]
        differ = (bits(dbg[:, :2]) != bits(mu)).any(-1)
        assert not bool(differ.any()), (f"e0={e0}: {int(differ.sum())} rows of debug_out mu differ from b_mu, worst "
                                        f"{float((dbg[:, :2] - mu).abs().max()):.2e}")
        assert torch.equal(bits(fused_value(dbg[:, 2], agent._val_stats)), bits(val)), e0
        sig = torch.exp(sigma.double())
        z = (act.double() - mu.double()) / sig
        bn = (z.abs() * (f32_ulp(act.double()) / sig + 4 * 2.0 ** -24 * z.abs())).sum(-1) + 8 * f32_ulp(nlp.double())
        en = (dbg[:, 3].double() - nlp.double()).abs()
        assert bool((en <= bn).all()), (e0, float((en - bn).max()))
        worst["nlp / bound"] = max(worst["nlp / bound"], float((en / bn).max()))
        kl_ref = float((torch.log(torch.tensor(1 + 1e-5, dtype=torch.float64)) + sig ** 2 / (2 * (sig ** 2 + 1e-5)) - 0.5).sum())
        kl = float(path.flat_g_lstm[path.P_lstm + 2])
        assert abs(kl - kl_ref) <= 1e-6, (kl, kl_ref)
        worst["kl abs"] = max(worst["kl abs"], abs(kl - kl_ref))
    assert torch.equal(agent.flat_l, flat_before)
    print("hand-off: mu and value bit for bit;", {k: f"{v:.2e}" for k, v in worst.items()})


# ------------------------------------------------------------------------------------------------------ 5. launch modes
ROLLOUT_BUFFERS = ["b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_rew", "b_adv", "b_ret", "_done_ext", "_nd_ext",
                   "_HH_saved", "_C_saved", "last_value", "ep_ret", "ep_len", "ep_stats", "_rng_counter"]


def test_rollout_launch_modes_are_bit_identical():
    """At 4096 envs the rollout runs with programmatic dependent launch.  Three agents from identical state: PDL (the
    default), PDL forced off, and the second rollout replayed from a captured CUDA graph.  After two rollouts every buffer
    the rollout writes, the persistent LSTM state and the env's observations are bit-identical: PDL only lets a kernel's
    prologue overlap its predecessor's tail (each kernel waits on its predecessor before touching memory), and a graph
    replays the same launches."""
    agents = [rollout_agent(4096) for _ in range(3)]
    agents[1].PDL_MAX_ENVS = 0
    assert agents[0].n <= agents[0].PDL_MAX_ENVS
    for it in range(2):
        for k, a in enumerate(agents):
            set_timeouts(a)
            if k == 2 and it == 1:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    a._rollout()
                set_timeouts(a)
                g.replay()
            else:
                a._rollout()
        torch.cuda.synchronize()
    ref = agents[0]
    for k, a in enumerate(agents[1:], 1):
        for name in ROLLOUT_BUFFERS:
            x, y = getattr(ref, name), getattr(a, name)
            assert torch.equal(x.view(torch.uint8), y.view(torch.uint8)), (k, name)
        for name in ("_r_HH", "_r_C"):
            assert torch.equal(getattr(ref, name)[0].view(torch.uint8), getattr(a, name)[0].view(torch.uint8)), (k, name)
        assert torch.equal(ref.env._obs_clamped, a.env._obs_clamped), k
    assert float(ref._done_ext[1:].mean()) > 0.5 / ref.T
