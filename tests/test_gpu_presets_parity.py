"""GPU parity of the LITERAL benchmarked presets (``config.FSTR_OVERRIDES`` — what bench.py and the
scaling run time — ``SHELF_OVERRIDES`` and ``PIPE_DR_OVERRIDES``), kernel vs the CPU oracle.

The reference-made fixtures in tests/golden strip ACCEL_TARGET_SCALING_* (this snapshot of the
reference has no code for that README.md:63 knob, SURVEY 0.1), so these presets are pinned
oracle-vs-kernel here:
  * fused ``vine_step`` from identical states, one control step at a time (same loop and the same
    stated tolerances as test_gpu_parity.test_fused_step_single_step_parity);
  * with ``controlFrequencyInv=1`` the reported rail force is the first sim step's, computed from
    identical inputs, so it must be BIT-EXACT — that pins the acceleration-target draw
    (which 16-bit Philox half, which range) of the fused kernel to the oracle's;
  * function-level ``vine_actuation`` with ``accel_scaling`` bit-exact vs ``oracle_actuation``;
  * the oracle's 24 dynamics uniforms of a sim step are exactly the 16-bit halves of Philox blocks
    8 i .. 8 i + 2 (low half first), read back raw from the device generator.
Measured error distributions are printed (pytest -s / captured in the junit log) so drift between
rounds is visible.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_parity import _dev, call_abi, make_handle, sync_env_to_oracle
from vine_robot_isaacgymenvs_b200 import abi, config as vcfg

pytestmark = pytest.mark.gpu

PRESETS = {
    "fstr": (vcfg.FSTR_OVERRIDES, "uniform"),
    "shelf": (vcfg.SHELF_OVERRIDES + ["task.env.maxEpisodeLength=60"], "reach"),
    "pipe_dr": (vcfg.PIPE_DR_OVERRIDES + ["task.env.maxEpisodeLength=50"], "reach"),
}


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available()
    return abi.load_library()


def _actions(mode, rng, T, n):
    a = rng.uniform(-1.3, 1.3, (T, n, 2)).astype(np.float32)
    if mode == "reach":
        a[:, : n // 2, 0] = rng.uniform(-1.0, -0.2, (T, n // 2)).astype(np.float32)
        a[:, : n // 2, 1] = rng.uniform(0.3, 1.0, (T, n // 2)).astype(np.float32)
    return a


def _make(overrides, n, seed):
    from vine_robot_isaacgymenvs_b200.tasks import isaacgym_task_map
    task_cfg = vcfg.task_config(["num_envs=%d" % n] + list(overrides))
    vc = vcfg.task_cfg_to_vine_config(task_cfg)
    env = isaacgym_task_map["Vine5LinkMovingBase"](
        cfg={**task_cfg, "seed": seed}, rl_device="cuda:0", sim_device="cuda:0", graphics_device_id=-1,
        headless=True, virtual_screen_capture=False, force_render=False)
    env.enable_debug_outputs(True)
    return env, vc


@pytest.mark.parametrize("name", sorted(PRESETS))
def test_benchmarked_presets_fused_step_vs_oracle(name, oracle_lib):
    overrides, mode = PRESETS[name]
    n, T, seed = 256, 48, 42
    env, vc = _make(overrides, n, seed)
    assert vc.accel_target_scaling_max > vc.accel_target_scaling_min or name == "shelf"   # the knob under test is ON
    ora = oracle_lib.OracleEnv(vc, n, seed=seed, use_f64=True)
    ora32 = oracle_lib.OracleEnv(vc, n, seed=seed, use_f64=False)
    actions = _actions(mode, np.random.default_rng(sum(map(ord, name))), T, n)
    contact_cfg = bool(vc.create_shelf or vc.create_pipe)
    n_checked = n_flip = n_ill = 0
    errs_obs, errs_rew, errs_q = [], [], []
    for t in range(T):
        for k in ora.a:
            ora32.a[k][...] = ora.a[k]
        od, rew, reset, extras = env.step(torch.from_numpy(actions[t]).cuda())
        ora.step(actions[t]); ora32.step(actions[t])
        well = (np.abs(ora32.dof_pos - ora.dof_pos).max(1) < 2e-5) & (np.abs(ora32.dof_vel - ora.dof_vel).max(1) < 2e-3) \
            & (ora32.reset == ora.reset)
        n_ill += int((~well).sum())
        st = env.get_state_dict(debug=True)
        for k, ok in (("u_rail_velocity", "u_rail"), ("u_fpam", "u_fpam"), ("smoothed_u_fpam", "smoothed"),
                      ("prev_u_rail_velocity", "prev_u_rail"), ("target_positions", "target"), ("object_info", "object_info")):
            assert np.array_equal(st[k].cpu().numpy(), getattr(ora, ok)), f"{k} step {t}"
        assert np.array_equal(env.progress_buf.cpu().numpy(), ora.progress), f"progress_buf step {t}"
        flip = (reset.cpu().numpy() != ora.reset) & well
        n_flip += int(flip.sum()); n_checked += n
        same = well & ~flip
        assert np.array_equal(extras["time_outs"].cpu().numpy()[same], ora.timeout[same].astype(bool))
        np.testing.assert_allclose(st["dof_pos"].cpu().numpy()[well], ora.dof_pos[well], rtol=1e-3, atol=2e-5)
        np.testing.assert_allclose(st["dof_vel"].cpu().numpy()[well], ora.dof_vel[well], rtol=1e-2,
                                   atol=5e-3 if contact_cfg else 2e-4)
        obs_gpu = env.obs_buf.cpu().numpy()
        e_obs = (np.abs(obs_gpu - ora.obs) / (1.0 + np.abs(ora.obs)))[well]
        assert e_obs.max() < (1e-3 if contact_cfg else 1e-4), f"obs step {t}: {e_obs.max()}"
        assert np.array_equal(od["obs"].cpu().numpy(), np.clip(obs_gpu, -5.0, 5.0))
        np.testing.assert_allclose(rew.cpu().numpy()[same], ora.rew[same], rtol=1e-3 if contact_cfg else 1e-5,
                                   atol=5e-4 if contact_cfg else 1e-5)
        errs_obs.append(e_obs.ravel()); errs_rew.append(np.abs(rew.cpu().numpy()[same] - ora.rew[same]))
        errs_q.append(np.abs(st["dof_pos"].cpu().numpy()[well] - ora.dof_pos[well]).ravel())
        sync_env_to_oracle(env, ora)
    eo, er, eq = np.concatenate(errs_obs), np.concatenate(errs_rew), np.concatenate(errs_q)
    print(f"\n[parity {name}] {n_checked} env-steps: obs rel err max {eo.max():.2e} p99 {np.quantile(eo, 0.99):.2e} | "
          f"reward abs err max {er.max():.2e} p99 {np.quantile(er, 0.99):.2e} | dof_pos abs err max {eq.max():.2e} | "
          f"mask flips {n_flip} | ill-conditioned {n_ill}")
    assert n_flip <= max(1, n_checked // 2000), f"{n_flip} reset flips in {n_checked} env-steps"
    assert n_ill <= max(2, n_checked // (50 if contact_cfg else 500)), f"{n_ill} ill-conditioned of {n_checked}"


@pytest.mark.parametrize("name", ["fstr", "pipe_dr"])
def test_accel_target_scaling_draw_of_the_fused_kernel_is_the_oracles(name, oracle_lib):
    """controlFrequencyInv=1: the rail force in the debug plane is the first (only) sim step's, a pure-f32
    function of identical inputs and of the acceleration-target multiplier -> bit-exact or the draw differs."""
    overrides = list(PRESETS[name][0]) + ["task.env.controlFrequencyInv=1"]
    n, T, seed = 512, 12, 7
    env, vc = _make(overrides, n, seed)
    ora = oracle_lib.OracleEnv(vc, n, seed=seed, use_f64=True)
    rng = np.random.default_rng(3)
    n_bang = 0
    for t in range(T):
        a = rng.uniform(-1.2, 1.2, (n, 2)).astype(np.float32)
        env.step(torch.from_numpy(a).cuda())
        ora.step(a)
        st = env.get_state_dict(debug=True)
        assert np.array_equal(st["rail_force"].cpu().numpy(), ora.rail_force), f"rail force step {t}"
        assert np.array_equal(st["prev_cart_vel_error"].cpu().numpy(), ora.prev_cart_vel_error)
        # the multiplier only enters the bang-bang branch |u_rail - v| > 0.1 (V5:1094): make sure it was exercised
        n_bang += int((np.abs(ora.prev_cart_vel_error) > 0.1).sum())
        sync_env_to_oracle(env, ora)
    assert n_bang > n, "bang-bang branch (where ACCEL_TARGET_SCALING acts) hardly exercised"


def test_actuation_with_accel_scaling_is_bit_exact(lib, oracle_lib):
    vc = vcfg.task_cfg_to_vine_config(vcfg.task_config(["num_envs=1024"] + list(vcfg.FSTR_OVERRIDES)))
    n = 1024
    rng = np.random.default_rng(17)
    f = np.float32
    inp = {"dof_pos": rng.normal(0, 0.3, (n, 6)).astype(f), "dof_vel": rng.normal(0, 2.0, (n, 6)).astype(f),
           "cart_vel_y": rng.normal(0, 0.5, n).astype(f), "u_rail_velocity": rng.uniform(-1, 1, n).astype(f),
           "u_fpam_to_use": rng.uniform(-0.1, 3, n).astype(f), "prev_cart_vel": rng.normal(0, 0.5, n).astype(f),
           "prev_cart_vel_error": rng.normal(0, 0.5, n).astype(f),
           "dynamics_scaling": rng.uniform(0.9, 1.1, (n, 5, 4)).astype(f),
           "accel_scaling": rng.uniform(0.9, 1.1, n).astype(f)}
    inp["cart_vel_y"][:8] = (inp["u_rail_velocity"][:8] - np.array([0.1, -0.1, 0.1000001, -0.1000001, 0.0999999, -0.0999999, 0, 1e-9], f))
    ref = {k: v.copy() for k, v in inp.items()}
    ref.update({"dof_efforts": np.zeros((n, 6), f), "prev_cart_vel_out": np.zeros(n, f), "prev_cart_vel_error_out": np.zeros(n, f)})
    oracle_lib.call_io("oracle_actuation", vc, n, abi.VineActuationIO, ref)
    out = {"dof_efforts": torch.zeros(n, 6, device="cuda"), "prev_cart_vel_out": torch.zeros(n, device="cuda"),
           "prev_cart_vel_error_out": torch.zeros(n, device="cuda")}
    t = {k: _dev(v) for k, v in inp.items()}
    t.update(out)
    h = make_handle(lib, vc, n)
    call_abi(lib, "vine_actuation", h, abi.VineActuationIO, t)
    lib.vine_destroy(h)
    assert np.array_equal(out["dof_efforts"].cpu().numpy(), ref["dof_efforts"])      # incl. the 4-term joint torques
    assert np.array_equal(out["prev_cart_vel_out"].cpu().numpy(), ref["prev_cart_vel_out"])
    assert np.array_equal(out["prev_cart_vel_error_out"].cpu().numpy(), ref["prev_cart_vel_error_out"])
    # and the multiplier matters: without it the bang-bang lanes differ
    t2 = dict(t); t2["accel_scaling"] = None
    t2["dof_efforts"] = torch.zeros(n, 6, device="cuda")
    h = make_handle(lib, vc, n)
    call_abi(lib, "vine_actuation", h, abi.VineActuationIO, t2)
    lib.vine_destroy(h)
    assert (t2["dof_efforts"].cpu().numpy()[:, 0] != ref["dof_efforts"][:, 0]).mean() > 0.3


def test_dynamics_uniform_halves_are_the_raw_philox_words(lib, oracle_lib):
    """oracle_dynamics_uniforms (what oracle/vine_oracle.c:509-511 draws from; entry 20 is the acceleration-target
    multiplier) == half k of blocks 8 i .. 8 i + 2 of the DEVICE generator, low half first, times 2^-16."""
    out = torch.zeros(3 * 4, dtype=torch.int32, device="cuda")
    for (seed, gid, step, sim_i) in [(42, 0, 0, 0), (42, 1000003, 77, 3), (2 ** 40 + 9, 2 ** 31 + 5, 12345, 2)]:
        assert lib.vine_philox_debug(seed, gid, oracle_lib.SITE_DYNAMICS, step, 8 * sim_i, 3, C.c_void_p(out.data_ptr()), None) == 0
        torch.cuda.synchronize()
        w = out.cpu().numpy().view(np.uint32)
        halves = np.stack([w & 0xFFFF, w >> 16], 1).reshape(-1).astype(np.float32) * np.float32(2.0 ** -16)
        assert np.array_equal(halves, oracle_lib.dynamics_uniforms(seed, gid, step, sim_i))
        assert halves[20] == np.float32(w[10] & 0xFFFF) * np.float32(2.0 ** -16)   # vine_b200.cu: u[10] & 0xffff


@pytest.mark.parametrize("name", ["c2_fstr", "c3_shelf"])
def test_wandb_dict_matches_the_reference_key_by_key(name, oracle_lib):
    """tests/golden/metrics_<name>.npz holds what the reference's own compute_reward put into ``self.wandb_dict`` at every
    step of the step_<name> rollout (V5:1250-1322: 19 aggregate scalars, 3 aggregated-reward entries, 54 reward-term
    statistics and the per-view-env traces).  ``env.wandb_dict()`` (one reduction launch + one state read) must have exactly
    those keys and, stepping from the reference's state, those values (means of f32 per-env quantities that match to ~1e-5)."""
    import json
    import os
    from conftest import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, f"metrics_{name}.npz"))
    keys, values, actions = json.loads(str(z["keys"])), z["values"], z["actions"]
    overrides = json.loads(str(z["overrides"]))
    T, n = actions.shape[:2]
    task_cfg = vcfg.task_config(overrides)
    vc = vcfg.task_cfg_to_vine_config(task_cfg)
    from vine_robot_isaacgymenvs_b200.tasks import isaacgym_task_map
    env = isaacgym_task_map["Vine5LinkMovingBase"](
        cfg={**task_cfg, "seed": int(z["seed"])}, rl_device="cuda:0", sim_device="cuda:0", graphics_device_id=-1,
        headless=True, virtual_screen_capture=False, force_render=False)
    env.enable_debug_outputs(True)
    assert env.index_to_view == int(z["index_to_view"])
    ora = oracle_lib.OracleEnv(vc, n, seed=int(z["seed"]), use_f64=True)
    worst = {}
    for t in range(T):
        env.step(torch.from_numpy(actions[t]).cuda())
        ora.step(actions[t])
        got = env.wandb_dict()
        assert sorted(got) == keys, (sorted(set(got) ^ set(keys)))
        for k, ref in zip(keys, values[t]):
            g = got[k]
            loose = "qd" in k or "vel" in k.lower() or "Velocity" in k        # velocities: the stated 1e-2 dynamics tolerance
            tol = (2e-2 * abs(ref) + 5e-3) if loose else (2e-3 * abs(ref) + 2e-4)
            if "nonzero_contact" in k or k in ("target_reached", "limit_hit", "tip_limit_hit"):
                tol = 1.0 / n + 1e-6                                          # a mask mean: at most one env at a threshold tie
            assert abs(g - ref) <= tol, (t, k, g, ref)
            worst[k] = max(worst.get(k, 0.0), abs(g - ref))
        sync_env_to_oracle(env, ora)
    top = sorted(worst.items(), key=lambda kv: -kv[1])[:3]
    print(f"\n[wandb_dict {name}] {len(keys)} keys x {T} steps; largest |difference|: " + ", ".join(f"{k}: {v:.2e}" for k, v in top))
