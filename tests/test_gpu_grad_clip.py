"""GPU: gradient-norm clipping in the kernel-only PPO update (rl_games truncate_grads / grad_norm): vine_grad_clip writes the
norm of the mean gradient and the clamped coefficient into the state block, vine_ppo_adam_clipped / vine_lstm_adam_clipped
multiply the coefficient in, and PPOAgent(truncate_grads=True) runs them between the reduction and Adam.

Adam's first step is lr * sign(g) whatever the scale of g, so one clipped step says nothing about clipping: these tests check
the coefficient itself against torch.nn.utils.clip_grad_norm_, and Adam over several steps whose coefficients differ."""
import ctypes as C
import math

import pytest
import torch

from vine_robot_isaacgymenvs_b200 import abi
from vine_robot_isaacgymenvs_b200.ppo.ppo import ActorCritic

pytestmark = pytest.mark.gpu
DEV = "cuda"
RNN = {"name": "lstm", "units": 256, "layers": 1, "before_mlp": False, "concat_input": True, "layer_norm": True}
DUMMY = 2 * 64 + 2 + 64 + 1 + 2          # unused head slots of the MLP half of the reference network
COEF, NORM = abi.PPO_STATE_CLIP_COEF, abi.PPO_STATE_GRAD_NORM


def p(t):
    return C.c_void_p(t.data_ptr())


def coef_ptr(state):
    return C.c_void_p(state.data_ptr() + COEF * 4)


def mlp_params(m):
    return [m.actor_mlp[0].weight, m.actor_mlp[0].bias, m.actor_mlp[2].weight, m.actor_mlp[2].bias, m.actor_mlp[4].weight,
            m.actor_mlp[4].bias]


def lstm_params(m):
    r = m.rnn.rnn
    return [r.weight_ih_l0, r.weight_hh_l0, r.bias_ih_l0, r.bias_hh_l0, m.layer_norm.weight, m.layer_norm.bias, m.mu.weight,
            m.mu.bias, m.value.weight, m.value.bias, m.sigma]


def head_params(m):
    return [m.mu.weight, m.mu.bias, m.value.weight, m.value.bias, m.sigma]


def random_grad(n, seed, norm):
    """n floats of mixed magnitudes scaled to the given Euclidean norm."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(n, device=DEV, generator=g) * torch.pow(10.0, -3 * torch.rand(n, device=DEV, generator=g))
    return x * (norm / float(x.double().norm())) if norm > 0 else torch.zeros(n, device=DEV)


def clip(lib, vecs, scale, max_norm, state, ws, channels=(None, None)):
    """vecs: [(flat, count)] (one or two); length = the whole vector."""
    (f1, c1), (f2, c2) = vecs[0], (vecs[1] if len(vecs) > 1 else (None, 0))
    rc = lib.vine_grad_clip(p(f1), c1, f1.numel(), p(f2) if f2 is not None else None, c2, f2.numel() if f2 is not None else 0,
                            scale, max_norm, p(state), p(ws), channels[0], channels[1], None)
    assert rc == 0, rc


def torch_norm_and_coef(model, groups, scale, max_norm):
    """clip_grad_norm_ over ActorCritic's parameters with .grad = the given flat pieces * scale (groups: [(flat piece, params)]).
    Returns (total norm, clamped coefficient) as torch computes them."""
    for flat, params in groups:
        o = 0
        for q in params:
            q.grad = (flat[o:o + q.numel()] * scale).view_as(q).clone()
            o += q.numel()
        assert o == flat.numel()
    total = torch.nn.utils.clip_grad_norm_(list(model.parameters()), max_norm)
    return float(total), float(torch.clamp(max_norm / (total + 1e-6), max=1.0))


# ------------------------------------------------------------------------------------------------- 1. norm and coefficient
CASES = {"above": 7.5, "below": 0.2, "zero": 0.0}


@pytest.mark.parametrize("net,O", [("mlp", 18), ("mlp", 28), ("lstm", 18)])
@pytest.mark.parametrize("case", list(CASES))
def test_norm_and_coefficient_match_clip_grad_norm(net, O, case):
    """state[10] = the norm clip_grad_norm_ returns over ActorCritic's parameters (relative 1e-5: f32 in another summation
    order), state[9] = torch's clamped coefficient; exactly 1.0 below the threshold and for a zero gradient.  The loss
    statistics behind each vector and (reference network) the 197 unused head slots of the MLP half carry 1e4 and do not count:
    zeroing them gives the same bits."""
    lib = abi.load_library()
    torch.manual_seed(O)
    max_norm, scale = 1.5, 0.5
    target = CASES[case] / scale
    P = lib.vine_ppo_num_params(O)
    if net == "mlp":
        model = ActorCritic(O, 2, (256, 128, 64)).to(DEV)
        g1 = torch.cat([random_grad(P, 3 + O, target), torch.full((4,), 1e4, device=DEV)])
        vecs, groups = [(g1, P)], [(g1[:P], mlp_params(model) + head_params(model))]
        junk = [(g1, slice(P, P + 4))]
    else:
        model = ActorCritic(O, 2, (256, 128, 64), rnn=RNN).to(DEV)
        PL = lib.vine_lstm_num_params(O)
        g1 = torch.cat([random_grad(P - DUMMY, 5, target * 0.3), torch.full((DUMMY + 4,), 1e4, device=DEV)])
        g2 = torch.cat([random_grad(PL, 6, target * math.sqrt(1 - 0.09)), torch.full((4,), 1e4, device=DEV)])
        vecs, groups = [(g1, P - DUMMY), (g2, PL)], [(g1[:P - DUMMY], mlp_params(model)), (g2[:PL], lstm_params(model))]
        junk = [(g1, slice(P - DUMMY, P + 4)), (g2, slice(PL, PL + 4))]
    ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
    state = torch.full((abi.PPO_STATE_FLOATS,), -3.0, device=DEV)
    clip(lib, vecs, scale, max_norm, state, ws)
    torch.cuda.synchronize()
    total, coef = torch_norm_and_coef(model, groups, scale, max_norm)
    got_total, got_coef = float(state[NORM]), float(state[COEF])
    assert abs(got_total - total) <= 1e-5 * total, (got_total, total)
    assert abs(got_coef - coef) <= 1e-5 * coef, (got_coef, coef)
    if case == "above":
        assert got_coef < 1.0 and abs(total - CASES[case]) < 1e-3 * CASES[case]
    else:
        assert got_coef == 1.0
    if case == "zero":
        assert got_total == 0.0
    assert torch.equal(state[:COEF], torch.full((COEF,), -3.0, device=DEV)) and bool((state[NORM + 1:] == -3.0).all())
    assert int(ws[:1].view(torch.int32)) == 0                       # the ticket is ready for the next call
    # the statistics and dummy slots are excluded, not merely small: zero them, same bits
    for vec, sl in junk:
        vec[sl] = 0.0
    state2 = state.clone()
    clip(lib, vecs, scale, max_norm, state2, ws)
    torch.cuda.synchronize()
    assert torch.equal(state2, state)


# ------------------------------------------------------------------------------- 2. clipped Adam against torch, several steps
NORMS = [3.0, 0.4, 5.0, 2.0]     # against max_norm 1: above, below, above again, above


def test_clipped_adam_matches_clip_grad_norm_and_torch_adam_mlp():
    """MLP network, four steps whose coefficients differ (< 1, exactly 1, < 1, < 1): clip + vine_ppo_adam_clipped against
    clip_grad_norm_ + torch.optim.Adam with the tolerances of test_adam_kernel_matches_torch_adam_and_repacks_the_weights
    (1e-6 absolute on the parameters); the packed block is byte for byte vine_mlp_pack of the new parameters."""
    lib = abi.load_library()
    O = 18
    torch.manual_seed(1)
    model = ActorCritic(O, 2, (256, 128, 64)).to(DEV)
    order = mlp_params(model) + head_params(model)
    flat = torch.cat([q.detach().reshape(-1) for q in order]).contiguous()
    P = flat.numel()
    packed = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_mlp_pack(*[p(q.detach().contiguous()) for q in order[:10]], O, p(packed), None) == 0
    ref = flat.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=3e-4, eps=1e-8)
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    state[0] = 3e-4
    m, v = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV)
    ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
    for k, nrm in enumerate(NORMS):
        grad = torch.cat([random_grad(P, 100 + k, nrm), torch.rand(4, device=DEV) + 0.1])
        state[1] = k + 1.0
        ref.grad = grad[:P].clone()
        total = float(torch.nn.utils.clip_grad_norm_([ref], 1.0))
        opt.step()
        clip(lib, [(grad, P)], 1.0, 1.0, state, ws)
        assert lib.vine_ppo_adam_clipped(p(grad), 1.0, p(flat), p(m), p(v), p(packed), p(state), O, 0.9, 0.999, 1e-8, 1,
                                         coef_ptr(state), None, None) == 0
        torch.cuda.synchronize()
        assert abs(float(state[NORM]) - total) <= 1e-5 * total
        assert (float(state[COEF]) == 1.0) == (nrm < 1.0)
        assert float((flat - ref.detach()).abs().max()) < 1e-6, k
        assert abs(float(state[2]) - float(grad[P + 2])) < 1e-7 and float(state[3]) == 1.0
    assert float(state[8]) == 4.0
    packed_ref = torch.zeros_like(packed)
    o, Wn = 0, []
    for q in order:
        Wn.append(flat[o:o + q.numel()].view_as(q))
        o += q.numel()
    assert lib.vine_mlp_pack(*[p(w.contiguous()) for w in Wn[:10]], O, p(packed_ref), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(packed, packed_ref)


def reference_problem(lib, O, seed):
    torch.manual_seed(seed)
    model = ActorCritic(O, 2, (256, 128, 64), rnn=RNN).to(DEV)
    P, PL = lib.vine_ppo_num_params(O), lib.vine_lstm_num_params(O)
    flat = torch.cat([q.detach().reshape(-1) for q in mlp_params(model)] + [torch.zeros(DUMMY, device=DEV)]).contiguous()
    for q in lstm_params(model)[4:10]:   # non-trivial LayerNorm and heads
        q.data.add_(0.05 * torch.randn_like(q))
    flat_l = torch.cat([q.detach().reshape(-1) for q in lstm_params(model)]).contiguous()
    assert flat.numel() == P and flat_l.numel() == PL
    return model, flat, flat_l


def pack_both(lib, flat, flat_l, O):
    shapes_m = [(256, O), (256,), (128, 256), (128,), (64, 128), (64,), (2, 64), (2,), (1, 64), (1,)]
    shapes_l = [(1024, 64 + O), (1024, 256), (1024,), (1024,), (256,), (256,), (2, 256), (2,), (1, 256), (1,)]

    def pieces(f, shapes):
        out, o = [], 0
        for s in shapes:
            n = math.prod(s)
            out.append(f[o:o + n].view(s).contiguous())
            o += n
        return out
    pm = torch.zeros(abi.MLP_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    pl = torch.zeros(abi.LSTM_PACKED_BYTES, dtype=torch.uint8, device=DEV)
    assert lib.vine_mlp_pack(*[p(t) for t in pieces(flat, shapes_m)], O, p(pm), None) == 0
    assert lib.vine_lstm_pack(*[p(t) for t in pieces(flat_l, shapes_l)], O, p(pl), None) == 0
    return pm, pl


def reference_grads(P, PL, seed, nrm):
    g1 = torch.zeros(P + 4, device=DEV)
    g1[:P - DUMMY] = random_grad(P - DUMMY, seed, 0.4 * nrm)
    g2 = torch.cat([random_grad(PL, seed + 1, math.sqrt(1 - 0.16) * nrm), torch.rand(4, device=DEV) + 0.1])
    return g1, g2


def test_clipped_adam_matches_clip_grad_norm_and_torch_adam_reference_network():
    """Reference network, both halves in one norm, four steps with differing coefficients: vine_grad_clip over the two vectors
    + vine_ppo_adam_clipped (MLP half) + vine_lstm_adam_clipped against clip_grad_norm_ + torch.optim.Adam on the two parameter
    groups, with the tolerances of test_lstm_adam_matches_torch_adam_and_repacks_exactly; both packed blocks are byte for byte
    the packing of the new parameters."""
    lib = abi.load_library()
    O = 18
    model, flat, flat_l = reference_problem(lib, O, 2)
    P, PL = flat.numel(), flat_l.numel()
    pm, pl = pack_both(lib, flat, flat_l, O)
    ref_m, ref_l = flat[:P - DUMMY].clone().requires_grad_(True), flat_l.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref_m, ref_l], lr=3e-4, betas=(0.9, 0.999), eps=1e-8)
    state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
    state[0] = 3e-4
    m, v = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV)
    ml, vl = torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV)
    m_mag = torch.zeros(P - DUMMY + PL, dtype=torch.float64, device=DEV)
    ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
    for k, nrm in enumerate(NORMS):
        g1, g2 = reference_grads(P, PL, 200 + 2 * k, nrm)
        state[1] = k + 1.0
        ref_m.grad, ref_l.grad = g1[:P - DUMMY].clone(), g2[:PL].clone()
        total = float(torch.nn.utils.clip_grad_norm_([ref_m, ref_l], 1.0))
        opt.step()
        m_mag = 0.9 * m_mag + 0.1 * torch.cat([ref_m.grad, ref_l.grad]).double().abs()
        clip(lib, [(g1, P - DUMMY), (g2, PL)], 1.0, 1.0, state, ws)
        assert lib.vine_ppo_adam_clipped(p(g1), 1.0, p(flat), p(m), p(v), p(pm), p(state), O, 0.9, 0.999, 1e-8, 0,
                                         coef_ptr(state), None, None) == 0
        assert lib.vine_lstm_adam_clipped(p(g2), 1.0, p(flat_l), p(ml), p(vl), p(pl), p(state), O, 0.9, 0.999, 1e-8,
                                          coef_ptr(state), None, None) == 0
        torch.cuda.synchronize()
        assert abs(float(state[NORM]) - total) <= 1e-5 * total
        assert (float(state[COEF]) == 1.0) == (nrm < 1.0)
        got = torch.cat([flat[:P - DUMMY], flat_l])
        want = torch.cat([ref_m.detach(), ref_l.detach()])
        assert float((got - want).abs().max()) < 1e-6, k
        st_m, st_l = opt.state[ref_m], opt.state[ref_l]
        m_ref = torch.cat([st_m["exp_avg"], st_l["exp_avg"]]).double()
        assert bool(((torch.cat([m[:P - DUMMY], ml]).double() - m_ref).abs() <= 2e-6 * m_mag).all())
        assert torch.allclose(torch.cat([v[:P - DUMMY], vl]), torch.cat([st_m["exp_avg_sq"], st_l["exp_avg_sq"]]), rtol=2e-5,
                              atol=1e-14)
        assert float(state[2]) == float(g2[PL + 2]) and float(state[3]) == 1.0
    assert float(state[8]) == 4.0
    assert torch.equal(flat[P - DUMMY:], torch.zeros(DUMMY, device=DEV))    # zero gradient: the dummy heads stay zero
    pm_ref, pl_ref = pack_both(lib, flat, flat_l, O)
    torch.cuda.synchronize()
    assert torch.equal(pm, pm_ref) and torch.equal(pl, pl_ref)


# ------------------------------------------------------------------------------------------- 3. below the threshold: exact
@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_clipping_below_the_threshold_is_bit_identical_to_no_clipping(net):
    """grad_norm above the gradient's norm: the coefficient is exactly 1.0 and g * 1.0 == g, so three steps give the same
    parameters, moments, packed blocks and state slots 0-8, bit for bit, as the launches without clipping."""
    lib = abi.load_library()
    O = 18
    results = []
    for clipped in (False, True):
        model, flat, flat_l = reference_problem(lib, O, 4)
        P, PL = flat.numel(), flat_l.numel()
        pm, pl = pack_both(lib, flat, flat_l, O)
        state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
        state[0] = 3e-4
        m, v, ml, vl = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV), torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV)
        ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
        for k in range(3):
            state[1] = k + 1.0
            g1, g2 = reference_grads(P, PL, 300 + 2 * k, 2.0)
            if net == "mlp":
                g1 = torch.cat([random_grad(P, 310 + k, 2.0), torch.rand(4, device=DEV) + 0.1])
            if clipped:
                vecs = [(g1, P)] if net == "mlp" else [(g1, P - DUMMY), (g2, PL)]
                clip(lib, vecs, 0.5, 50.0, state, ws)
                cf = coef_ptr(state)
                assert lib.vine_ppo_adam_clipped(p(g1), 0.5, p(flat), p(m), p(v), p(pm), p(state), O, 0.9, 0.999, 1e-8,
                                                 int(net == "mlp"), cf, None, None) == 0
                if net == "lstm":
                    assert lib.vine_lstm_adam_clipped(p(g2), 0.5, p(flat_l), p(ml), p(vl), p(pl), p(state), O, 0.9, 0.999, 1e-8,
                                                      cf, None, None) == 0
            else:
                assert lib.vine_ppo_adam(p(g1), 0.5, p(flat), p(m), p(v), p(pm), p(state), O, 0.9, 0.999, 1e-8,
                                         int(net == "mlp"), None, None) == 0
                if net == "lstm":
                    assert lib.vine_lstm_adam(p(g2), 0.5, p(flat_l), p(ml), p(vl), p(pl), p(state), O, 0.9, 0.999, 1e-8,
                                              None, None) == 0
        torch.cuda.synchronize()
        if clipped:
            assert float(state[COEF]) == 1.0 and 0.0 < float(state[NORM]) < 50.0
        results.append([flat, m, v, pm] + ([flat_l, ml, vl, pl] if net == "lstm" else []) + [state[:COEF].clone()])
    for i, (a, b) in enumerate(zip(*results)):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), i


# ---------------------------------------------------------------------------------- 4. peer-memory channels on one rank
def test_clip_as_the_p2p_consumer_on_one_rank_is_transparent():
    """world = 1, reference network: vine_ppo_reduce and vine_lstm_reduce write into their channels' buffers, vine_grad_clip
    consumes both channels (the rank sums land in the local vectors) and the Adam launches run without a channel.  After five
    exchanges (both buffers of each region reused) everything is bit-identical to the same launches without channels, with a
    coefficient below 1, and each channel advanced once per exchange without a timeout."""
    from vine_robot_isaacgymenvs_b200 import distributed as vd
    lib = abi.load_library()
    O = 18
    P, PL = lib.vine_ppo_num_params(O), lib.vine_lstm_num_params(O)
    g = torch.Generator(device=DEV).manual_seed(8)
    mws = [torch.randn(3, abi.PPO_WS_FLOATS, device=DEV, generator=g) * 1e-2 for _ in range(5)]
    lws = [torch.randn(1, abi.LSTM_WGRAD_BLOCK_FLOATS, device=DEV, generator=g) * 0.01 for _ in range(5)]
    hgs = [torch.rand(abi.LSTM_HEAD_GRAD_PARTS + 1, abi.LSTM_HEAD_GRAD_FLOATS, device=DEV, generator=g) * 1e-3 for _ in range(5)]
    results = []
    for use_channel in (False, True):
        model, flat, flat_l = reference_problem(lib, O, 9)
        pm, pl = pack_both(lib, flat, flat_l, O)
        state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
        state[0] = 3e-4
        m, v, ml, vl = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV), torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV)
        f1, f2 = torch.zeros(P + 4, device=DEV), torch.zeros(PL + 4, device=DEV)
        ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
        ch1 = vd.P2PChannel(lib, P + 4, DEV) if use_channel else None
        ch2 = vd.P2PChannel(lib, PL + 4, DEV) if use_channel else None
        coefs = []
        for k in range(5):
            state[1] = k + 1.0
            assert lib.vine_ppo_reduce(p(mws[k]), 3, O, p(f1), None, None, ch1.ptr if ch1 else None, None) == 0
            hg = hgs[k].clone()
            assert lib.vine_lstm_reduce(p(lws[k]), 1, p(hg), 8, O, p(f2), ch2.ptr if ch2 else None, None) == 0
            clip(lib, [(f1, P - DUMMY), (f2, PL)], 1.0, 0.05, state, ws,
                 channels=(ch1.ptr if ch1 else None, ch2.ptr if ch2 else None))
            assert lib.vine_ppo_adam_clipped(p(f1), 1.0, p(flat), p(m), p(v), p(pm), p(state), O, 0.9, 0.999, 1e-8, 0,
                                             coef_ptr(state), None, None) == 0
            assert lib.vine_lstm_adam_clipped(p(f2), 1.0, p(flat_l), p(ml), p(vl), p(pl), p(state), O, 0.9, 0.999, 1e-8,
                                              coef_ptr(state), None, None) == 0
            coefs.append(state[COEF:COEF + 1].clone())
        torch.cuda.synchronize()
        assert all(float(c) < 1.0 for c in coefs)
        if use_channel:
            assert ch1.status() == (5, False) and ch2.status() == (5, False)
            ch1.close()
            ch2.close()
        results.append((flat.clone(), m.clone(), v.clone(), pm.clone(), flat_l.clone(), ml.clone(), vl.clone(), pl.clone(),
                        state.clone(), f1.clone(), f2.clone()))
    for i, (a, b) in enumerate(zip(*results)):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), i


# ------------------------------------------------------------------------------------------------------- 5. graph replay
def test_graph_replay_of_clip_and_adam_is_bit_identical_to_eager_calls():
    """Clip + both Adam launches captured once and replayed five times on fresh gradients give the same bits as five eager
    calls: the ticket of the block-partial sum resets itself inside the kernel."""
    lib = abi.load_library()
    O = 18
    P, PL = lib.vine_ppo_num_params(O), lib.vine_lstm_num_params(O)
    grads = [reference_grads(P, PL, 400 + 2 * k, [3.0, 0.5, 2.0, 4.0, 1.5][k]) for k in range(5)]
    results = []
    for graphed in (False, True):
        model, flat, flat_l = reference_problem(lib, O, 11)
        pm, pl = pack_both(lib, flat, flat_l, O)
        state = torch.zeros(abi.PPO_STATE_FLOATS, device=DEV)
        state[0] = 3e-4
        m, v, ml, vl = torch.zeros(P, device=DEV), torch.zeros(P, device=DEV), torch.zeros(PL, device=DEV), torch.zeros(PL, device=DEV)
        g1, g2 = torch.zeros(P + 4, device=DEV), torch.zeros(PL + 4, device=DEV)
        ws = torch.zeros(abi.GRAD_CLIP_WS_FLOATS, device=DEV)
        norms = []

        def step():
            state[1:2].add_(1.0)
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert lib.vine_grad_clip(p(g1), P - DUMMY, P + 4, p(g2), PL, PL + 4, 1.0, 1.0, p(state), p(ws), None, None, st) == 0
            assert lib.vine_ppo_adam_clipped(p(g1), 1.0, p(flat), p(m), p(v), p(pm), p(state), O, 0.9, 0.999, 1e-8, 0,
                                             coef_ptr(state), None, st) == 0
            assert lib.vine_lstm_adam_clipped(p(g2), 1.0, p(flat_l), p(ml), p(vl), p(pl), p(state), O, 0.9, 0.999, 1e-8,
                                              coef_ptr(state), None, st) == 0
        graph = None
        if graphed:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
        for a, b in grads:
            g1.copy_(a)
            g2.copy_(b)
            if graph is not None:
                graph.replay()
            else:
                step()
            norms.append(state[COEF:NORM + 1].clone())
        torch.cuda.synchronize()
        assert float(state[1]) == 5.0 and int(ws[:1].view(torch.int32)) == 0
        results.append((flat, m, v, pm, flat_l, ml, vl, pl, state, torch.stack(norms)))
    assert float(results[1][-1][1, 0]) == 1.0 and float(results[1][-1][0, 0]) < 1.0   # the coefficients really differ
    for i, (a, b) in enumerate(zip(*results)):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), i


# ------------------------------------------------------------------------------------------------------------ 6. trainer
def make_agent(extra, graphs, n=512, **kw):
    import vine_robot_isaacgymenvs_b200 as vine
    from vine_robot_isaacgymenvs_b200 import config as vcfg
    from vine_robot_isaacgymenvs_b200.ppo.ppo import PPOAgent
    cfg = vcfg.compose(vcfg.FSTR_OVERRIDES + [f"num_envs={n}", "headless=True", "train.params.config.minibatch_size=4096"]
                       + extra)
    return PPOAgent(vine.make(cfg=cfg), cfg["train"], seed=1, use_graphs=graphs, **kw)


MLP = ["train.params.network.rnn=null"]
CLIP = ["train.params.config.truncate_grads=True", "train.params.config.grad_norm=0.01"]


@pytest.mark.parametrize("net", ["mlp", "lstm"])
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
def test_agent_with_truncate_grads_trains_on_the_kernel_path(net, graphs):
    agent = make_agent((MLP if net == "mlp" else []) + CLIP, graphs)
    assert agent.truncate_grads and agent.fused_update and agent.native_lstm == (net == "lstm")
    before = [q.detach().clone() for q in agent.model.parameters()]
    for _ in range(3):
        agent.train_epoch()
    torch.cuda.synchronize()
    st = agent.pop_stats()
    assert all(x == x and abs(x) < 1e6 for x in (st["a_loss"], st["c_loss"], st["kl"]))
    assert all(torch.isfinite(q).all() for q in agent.model.parameters())
    assert any(not torch.equal(a, b) for a, b in zip(before, agent.model.parameters()))
    coef, norm = float(agent.ppo_state[COEF]), float(agent.ppo_state[NORM])
    assert 0.0 < coef < 1.0 and norm > 0.01 and abs(coef - 0.01 / (norm + 1e-6)) <= 1e-6


@pytest.mark.parametrize("net", ["mlp", "lstm"])
def test_agent_gradient_norm_matches_the_torch_update(net, monkeypatch):
    """Same rollout, one minibatch: the norm vine_grad_clip records (state[10]) is the norm clip_grad_norm_ returns in the torch
    baseline's update, within the bf16 tolerance of the parity tests (5e-2), and grad_norm below it clips (state[9] < 1)."""
    one = ["train.params.config.mini_epochs=1", "train.params.config.minibatch_size=8192", "train.params.config.truncate_grads=True"]
    extra = (MLP if net == "mlp" else []) + one
    seen = []
    real = torch.nn.utils.clip_grad_norm_

    def recording(params, max_norm, *args, **kw):
        total = real(params, max_norm, *args, **kw)
        seen.append((float(total), float(max_norm)))
        return total
    monkeypatch.setattr(torch.nn.utils, "clip_grad_norm_", recording)
    a = make_agent(extra, False, use_fused_update=True)
    agents = [make_agent(extra, False, use_fused_update=False) for _ in range(2)]
    for b in agents:
        b.load_state_dict(a.state_dict())
    a._rollout()
    for b in agents:
        for name in ("b_obs", "b_act", "b_mu", "b_nlp", "b_val", "b_ret", "b_adv", "b_done"):
            getattr(b, name).copy_(getattr(a, name))
        if net == "lstm":
            from vine_robot_isaacgymenvs_b200.ppo.tiles import from_tiles
            for ck in range(a.T // a.seq_len):
                b.b_h[ck].copy_(from_tiles(a._HH_saved[ck], a.n))
                b.b_c[ck].copy_(a._C_saved[ck])
    agents[0].grad_norm = 1e9
    agents[0]._update_any()                  # first update: the unclipped norm of this rollout
    torch.cuda.synchronize()
    unclipped = seen[-1][0]
    a.grad_norm = agents[1].grad_norm = 0.25 * unclipped
    a._update_any()
    agents[1]._update_any()
    torch.cuda.synchronize()
    total, max_norm = seen[-1]
    assert len(seen) == 2 and max_norm == a.grad_norm and abs(total - unclipped) <= 1e-3 * unclipped
    got = float(a.ppo_state[NORM])
    assert abs(got - total) <= 5e-2 * total, (got, total)
    assert float(a.ppo_state[COEF]) < 1.0 and abs(float(a.ppo_state[COEF]) - max_norm / total) <= 5e-2 * max_norm / total
    sa, sb = a.pop_stats(), agents[1].pop_stats()
    for k in ("a_loss", "c_loss", "kl"):
        assert abs(sa[k] - sb[k]) <= 5e-2 * abs(sb[k]) + 2e-4, (k, sa[k], sb[k])


# -------------------------------------------------------------------------------------------------------- 7. two GPUs
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs with peer access")
def test_clipped_training_keeps_ranks_bit_identical_on_two_gpus():
    import json
    import os
    import subprocess
    import sys
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(repo, "tools", "grad_clip_multi_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=repo, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    assert d["world"] == 2
    for net in ("mlp", "lstm"):
        p2p, nccl = d[net]["p2p"], d[net]["nccl"]
        for res in (p2p, nccl):
            assert res["params_bit_identical_across_ranks"] and res["coef_bit_identical_across_ranks"] and res["finite"]
            assert 0.0 < res["coef"] < 1.0
        assert not p2p["timed_out"] and p2p["exchanges"] > 0
        assert abs(p2p["c_loss"] - nccl["c_loss"]) <= 0.1 * abs(nccl["c_loss"]) + 1e-3
