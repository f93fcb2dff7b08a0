"""Generate the golden fixtures in tests/golden/ by EXECUTING THE REFERENCE.

Run in the build container only (needs /root/reference):
    python tests/golden/generate_golden.py

Fixtures:
  reference_cfg.json    the reference's cfg/ YAML files, composed and resolved (compose(cfg_dir=...))
  step_<scenario>.npz   whole ``VecTask.step`` rollouts of the reference's unmodified task under
                        ref_harness.FakeGym (dynamics = oracle f64, RNG = product Philox streams)
  fn_<name>.npz         single calls of the reference's own functions on synthetic inputs:
                        compute_observations + compute_reward(+_jit) + compute_reset_jit,
                        pre_physics_step's action path, compute_and_set_dof_actuation_force_tensor,
                        reset_idx.
Each file stores the Hydra-style overrides it was made with, so tests rebuild the exact config.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import ref_harness as H  # noqa: E402
from vine_robot_isaacgymenvs_b200 import config as vcfg  # noqa: E402

FULL_DR = [
    "task.task.randomization_parameters.DYNAMICS_SCALING_MIN=0.9",
    "task.task.randomization_parameters.DYNAMICS_SCALING_MAX=1.1",
    "task.task.randomization_parameters.ACTION_NOISE_STD=0.01",
    "task.task.randomization_parameters.OBSERVATION_NOISE_STD=0.01",
]
NO_OBST = ["task.env.CREATE_PIPE=False", "task.env.CREATE_SHELF=False"]
# ACCEL_TARGET_SCALING_* appears only on the README.md:63 command line; this snapshot of the
# reference has no code for it (SURVEY 0.1), so the reference-made fixtures leave it out.
FSTR_SNAPSHOT = [o for o in vcfg.FSTR_OVERRIDES if "ACCEL_TARGET_SCALING" not in o]

# name -> (overrides, num_envs, steps, action mode)
STEP_SCENARIOS = {
    # BASELINE configs[0]: free space, defaults
    "c1_free": (NO_OBST, 64, 24, "uniform"),
    # BASELINE configs[1]: the README.md:63 FSTR command line
    "c2_fstr": (FSTR_SNAPSHOT, 32, 130, "uniform"),
    # BASELINE configs[2]: shelf with contact-force resets
    "c3_shelf": (["task.env.CREATE_SHELF=True", "task.env.CREATE_PIPE=False",
                  "task.env.USE_NONZERO_CONTACT_FORCE_RESET=True",
                  "task.task.randomization_parameters.ACTION_NOISE_STD=0.01",
                  "task.env.maxEpisodeLength=60"], 48, 90, "reach"),
    # BASELINE configs[3]: pipe + full DR (default obs type, 28 wide)
    "c4_pipe_dr": (["task.env.CREATE_PIPE=True", "task.env.maxEpisodeLength=50"] + FULL_DR, 32, 70, "reach"),
    # literal zero-order-hold efforts (VT:346-356): numerically unstable with the URDF inertias
    # (SURVEY R1; diverges to NaN within 3 control steps), so only 2 steps are pinned
    "zoh": (NO_OBST + ["+task.env.TORQUE_LAW_INTEGRATION=zoh"], 16, 2, "uniform"),
    "delay0": (NO_OBST + ["task.env.ACTION_DELAY=0", "task.env.maxEpisodeLength=12"], 16, 20, "uniform"),
    "delay3": (NO_OBST + ["task.env.ACTION_DELAY=3", "task.env.maxEpisodeLength=12"] + FULL_DR, 16, 20, "uniform"),
    "obs_pos_only": (NO_OBST + ["OBSERVATION_TYPE=POS_ONLY", "task.env.SCALE_OBSERVATIONS=False",
                                "task.env.maxEpisodeLength=6"], 8, 10, "uniform"),
    "obs_pos_and_vel": (NO_OBST + ["OBSERVATION_TYPE=POS_AND_VEL", "task.env.SCALE_OBSERVATIONS=False",
                                   "task.env.maxEpisodeLength=6"], 8, 10, "uniform"),
    "obs_pos_and_fd_vel": (NO_OBST + ["OBSERVATION_TYPE=POS_AND_FD_VEL", "task.env.SCALE_OBSERVATIONS=False",
                                      "task.env.maxEpisodeLength=6"], 8, 10, "uniform"),
    "obs_pos_and_prev_pos": (NO_OBST + ["OBSERVATION_TYPE=POS_AND_PREV_POS", "task.env.SCALE_OBSERVATIONS=False",
                                        "task.env.maxEpisodeLength=6"], 8, 10, "uniform"),
    "flags": (NO_OBST + ["task.env.USE_SMOOTHED_FPAM=False", "task.env.FORCE_U_RAIL_VELOCITY=True",
                         "task.env.USE_TIP_LIMIT_HIT_RESET=True", "task.env.USE_TARGET_REACHED_RESET=False",
                         "task.env.RANDOMIZE_TARGETS=False", "task.env.RANDOMIZE_DOF_INIT=False",
                         "task.env.RAIL_D_GAIN=0.5", "vine_randomize=False", "task.env.maxEpisodeLength=8",
                         "task.env.POSITION_REWARD_WEIGHT=1.5", "task.env.CONST_NEGATIVE_REWARD_WEIGHT=0.25",
                         "task.env.VELOCITY_SUCCESS_REWARD_WEIGHT=0.5", "task.env.U_FPAM_CONTROL_REWARD_WEIGHT=0.125",
                         "task.env.U_RAIL_VELOCITY_CONTROL_REWARD_WEIGHT=0.3", "task.env.RAIL_VELOCITY_CHANGE_REWARD_WEIGHT=0.7",
                         "task.env.U_FPAM_CHANGE_REWARD_WEIGHT=0.2", "task.env.CART_Y_REWARD_WEIGHT=0.4",
                         "task.env.TIP_Y_REWARD_WEIGHT=0.01"], 16, 14, "uniform"),
}


# scenarios whose rollout also freezes the reference's wandb_dict of every step (metrics_<name>.npz)
METRIC_SCENARIOS = ("c2_fstr", "c3_shelf")


def make_actions(mode, rng, T, n):
    a = rng.uniform(-1.3, 1.3, (T, n, 2)).astype(np.float32)   # beyond +-1: exercises clipActions
    if mode == "reach":  # half the envs drive toward -y with high pressure so obstacles get touched
        a[:, : n // 2, 0] = rng.uniform(-1.0, -0.2, (T, n // 2)).astype(np.float32)
        a[:, : n // 2, 1] = rng.uniform(0.3, 1.0, (T, n // 2)).astype(np.float32)
    return a


def gen_step(name, overrides, n, T, mode, seed=42):
    cfg = vcfg.task_config(["num_envs=%d" % n] + list(overrides))
    rt = H.ReferenceTask(cfg, seed=seed)
    rng = np.random.default_rng(sum(map(ord, name)))
    actions = make_actions(mode, rng, T, n)
    keys = ["obs_buf", "obs_clamped", "rew_buf", "reset_buf", "progress_buf", "timeout_buf", "dof_pos",
            "dof_vel", "tip_positions", "target_positions", "object_info", "smoothed_u_fpam", "u_fpam",
            "u_rail_velocity", "prev_u_rail_velocity", "rail_force", "prev_cart_vel", "prev_cart_vel_error",
            "aggregated_rew_buf"]
    rec = {k: [] for k in keys}
    contact = []
    wandb_rows, wandb_keys = [], None
    for t in range(T):
        rt.step(actions[t])
        s = rt.snapshot()
        for k in keys:
            rec[k].append(s[k])
        contact.append(rt.gym.c_lip.copy())
        if name in METRIC_SCENARIOS:   # the reference's own per-step wandb dict (compute_reward, V5:1250-1322)
            wd = {k: float(v) for k, v in rt.task.wandb_dict.items()}
            wandb_keys = wandb_keys or sorted(wd)
            assert sorted(wd) == wandb_keys
            wandb_rows.append([wd[k] for k in wandb_keys])
        if name == "delay0" and t == 9:   # VT:412-427 reset_done path: reset_idx outside step
            rt.reset_done_ids(np.arange(0, n, 3))
    out = {k: np.stack(v) for k, v in rec.items()}
    out["contact"] = np.stack(contact)
    out["actions"] = actions
    out["overrides"] = np.array(json.dumps(["num_envs=%d" % n] + list(overrides)))
    out["seed"] = np.array(seed)
    out["reset_done_at"] = np.array(9 if name == "delay0" else -1)
    path = os.path.join(HERE, "step_%s.npz" % name)
    np.savez_compressed(path, **out)
    if wandb_rows:
        np.savez_compressed(os.path.join(HERE, "metrics_%s.npz" % name), keys=np.array(json.dumps(wandb_keys)),
                            values=np.array(wandb_rows, np.float64), index_to_view=np.array(int(rt.task.index_to_view)),
                            overrides=out["overrides"], seed=out["seed"], actions=actions)
    print("%-22s n=%3d T=%3d  resets=%5d  timeouts=%4d  max|contact|=%.3g  %d KB" % (
        name, n, T, int(out["reset_buf"].sum()), int(out["timeout_buf"].sum()), float(out["contact"].max()),
        os.path.getsize(path) // 1024))


# ------------------------------------------------------------------------------------------------
# function-level goldens
# ------------------------------------------------------------------------------------------------
def gen_fn_post_physics(name, overrides, n=512, seed=7):
    """compute_observations (V5:1339) + compute_reward (V5:1218) on synthetic state."""
    cfg = vcfg.task_config(["num_envs=%d" % n] + list(overrides))
    rt = H.ReferenceTask(cfg, seed=seed)
    t, g = rt.task, rt.gym
    rng = np.random.default_rng(seed)
    f = np.float32
    C = int(cfg["env"]["controlFrequencyInv"])
    inp = {
        "dof_pos": rng.normal(0, 0.3, (n, 6)).astype(f), "dof_vel": rng.normal(0, 2.0, (n, 6)).astype(f),
        "prev_dof_pos": rng.normal(0, 0.3, (n, 6)).astype(f),
        "tip_positions": (rng.normal(0, 0.2, (n, 3)) + [0, -0.2, 0.6]).astype(f),
        "prev_tip_positions": (rng.normal(0, 0.2, (n, 3)) + [0, -0.2, 0.6]).astype(f),
        "tip_velocities": rng.normal(0, 1.0, (n, 3)).astype(f),
        "cart_positions_y": rng.uniform(-0.4, 0.4, n).astype(f),
        "target_positions": (rng.normal(0, 0.1, (n, 3)) + [0, -0.3, 0.6]).astype(f),
        "target_velocities": rng.normal(0, 0.3, (n, 3)).astype(f),
        "smoothed_u_fpam": rng.uniform(-0.1, 3, n).astype(f), "u_fpam": rng.uniform(-0.1, 3, n).astype(f),
        "u_rail_velocity": rng.uniform(-1, 1, n).astype(f), "prev_u_rail_velocity": rng.uniform(-1, 1, n).astype(f),
        "object_info": rng.uniform(-0.1, 1.2, (n, 2)).astype(f),
        "contact_force_norms": (rng.uniform(0, 2, (C, n)) * (rng.uniform(0, 1, (C, n)) < 0.3)).astype(f),
        "reset_buf_in": (rng.uniform(0, 1, n) < 0.2).astype(np.int64),
        "progress_buf": rng.integers(0, int(cfg["env"]["maxEpisodeLength"]) + 2, n).astype(np.int64),
    }
    # threshold cases: tips placed right around SUCCESS_DIST of the target, carts at +-RAIL_SOFT_LIMIT
    sd, lim = f(cfg["env"]["SUCCESS_DIST"]), f(cfg["env"]["RAIL_SOFT_LIMIT"])
    m = n // 4
    d = rng.normal(0, 1, (m, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    radius = (sd * (1 + rng.integers(-4, 5, m) * 2.0 ** -23)).astype(f)
    inp["tip_positions"][:m] = (inp["target_positions"][:m].astype(np.float64) + d * radius[:, None]).astype(f)
    inp["tip_positions"][m:m + 8] = inp["target_positions"][m:m + 8]          # dist == 0
    inp["tip_positions"][m + 8:m + 16, 1] = inp["target_positions"][m + 8:m + 16, 1]  # tip_y == target_y
    inp["cart_positions_y"][:16] = np.array([lim, -lim, np.nextafter(lim, f(1)), np.nextafter(-lim, f(-1)),
                                             np.nextafter(lim, f(0)), np.nextafter(-lim, f(0)), 0, -0.0] * 2, f)
    inp["contact_force_norms"][:, :8] = 0
    inp["progress_buf"][:6] = np.array([cfg["env"]["maxEpisodeLength"] - 2, cfg["env"]["maxEpisodeLength"] - 1,
                                        cfg["env"]["maxEpisodeLength"], 0, 1, 2])
    # load into the reference task's tensors / the fake gym caches
    ds = g.dof_state.view(n, 6, 2)
    ds[..., 0] = torch.from_numpy(inp["dof_pos"]); ds[..., 1] = torch.from_numpy(inp["dof_vel"])
    t.prev_dof_pos = torch.from_numpy(inp["prev_dof_pos"].copy())
    g.c_tip[:] = inp["tip_positions"]; g.c_tipvel[:] = inp["tip_velocities"]; g.c_cart_y[:] = inp["cart_positions_y"]
    t.prev_tip_positions = torch.from_numpy(inp["prev_tip_positions"].copy())
    t.target_positions = torch.from_numpy(inp["target_positions"].copy())
    t.target_velocities = torch.from_numpy(inp["target_velocities"].copy())
    t.smoothed_u_fpam = torch.from_numpy(inp["smoothed_u_fpam"].copy()).reshape(n, 1)
    t.u_fpam = torch.from_numpy(inp["u_fpam"].copy()).reshape(n, 1)
    t.u_rail_velocity = torch.from_numpy(inp["u_rail_velocity"].copy()).reshape(n, 1)
    t.prev_u_rail_velocity = torch.from_numpy(inp["prev_u_rail_velocity"].copy()).reshape(n, 1)
    t.rail_force = torch.zeros(n, 1)
    t.object_info = torch.from_numpy(inp["object_info"].copy())
    t.shelf_contact_force_norms = [torch.from_numpy(inp["contact_force_norms"][i].copy()) for i in range(C)]
    t.reset_buf[:] = torch.from_numpy(inp["reset_buf_in"]); t.progress_buf[:] = torch.from_numpy(inp["progress_buf"])
    rt._patch()
    try:
        t.compute_observations(); t.compute_reward()
    finally:
        rt._unpatch()
    timeout = (t.progress_buf >= t.max_episode_length - 1) & (t.reset_buf != 0)   # VT:366
    # the reward matrix comes straight from the reference's jit function on the same tensors
    dist = torch.linalg.norm(t.tip_positions - t.target_positions, dim=-1)
    reached = dist < cfg["env"]["SUCCESS_DIST"]
    cart_y = t.cart_positions[:, 1]
    limit_hit = torch.logical_or(cart_y > cfg["env"]["RAIL_SOFT_LIMIT"], cart_y < -cfg["env"]["RAIL_SOFT_LIMIT"])
    tip_limit_hit = t.tip_positions[:, 1] < t.target_positions[:, 1]
    if cfg["env"]["CREATE_SHELF"]:
        cn = torch.mean(torch.stack(t.shelf_contact_force_norms, dim=0), dim=0)
    else:
        cn = torch.zeros(n)
    _, rmat, _ = rt.v5.compute_reward_jit(dist, reached, t.tip_velocities, t.target_velocities, t.u_rail_velocity,
                                          t.u_fpam, t.prev_u_rail_velocity, t.smoothed_u_fpam, limit_hit,
                                          tip_limit_hit, cart_y, cn, t.reward_weights, rt.v5.REWARD_NAMES)
    noise = None
    if cfg["task"]["vine_randomize"] and cfg["task"]["randomization_parameters"]["OBSERVATION_NOISE_STD"] != 0:
        noise = rt.feed.randn_like(t.obs_buf).numpy()
    out = dict(inp)
    out.update({"obs_buf": t.obs_buf.numpy().copy(), "rew_buf": t.rew_buf.numpy().copy(),
                "reward_matrix": rmat.numpy().copy(), "reset_buf_out": t.reset_buf.numpy().copy(),
                "timeout_buf": timeout.numpy().astype(np.uint8),
                "target_reached": reached.numpy(), "limit_hit": limit_hit.numpy(), "tip_limit_hit": tip_limit_hit.numpy(),
                "overrides": np.array(json.dumps(["num_envs=%d" % n] + list(overrides)))})
    if noise is not None:
        out["obs_noise"] = noise
    np.savez_compressed(os.path.join(HERE, "fn_post_%s.npz" % name), **out)
    print("fn_post_%-16s reached=%d limit=%d tiplimit=%d resets=%d" % (
        name, int(reached.sum()), int(limit_hit.sum()), int(tip_limit_hit.sum()), int(t.reset_buf.sum())))


def gen_fn_pre_and_actuation(name, overrides, n=256, T=6, seed=11):
    """pre_physics_step action path (V5:927-940) and the actuation law (V5:1028-1106)."""
    cfg = vcfg.task_config(["num_envs=%d" % n] + list(overrides))
    rt = H.ReferenceTask(cfg, seed=seed)
    t, g = rt.task, rt.gym
    rng = np.random.default_rng(seed)
    f = np.float32
    D = int(cfg["env"]["ACTION_DELAY"])
    rand = bool(cfg["task"]["vine_randomize"])
    rec = {k: [] for k in ("actions", "action_noise", "history_in", "smoothed_in", "history_out", "u_rail_velocity",
                           "u_fpam", "smoothed_out", "dof_pos", "dof_vel", "cart_vel_y", "u_fpam_to_use",
                           "prev_cart_vel", "prev_cart_vel_error", "dynamics_scaling", "dof_efforts",
                           "prev_cart_vel_out", "prev_cart_vel_error_out")}
    hist = lambda: (np.stack([np.concatenate([a.numpy(), b.numpy()], 1) for a, b in t.actions_history], 1).astype(f)  # noqa: E731
                    if D > 0 else np.zeros((n, 1, 2), f))
    for step in range(T):
        a = np.clip(rng.uniform(-1.2, 1.2, (n, 2)), -1, 1).astype(f)
        rec["actions"].append(a)
        rec["history_in"].append(hist()); rec["smoothed_in"].append(t.smoothed_u_fpam.numpy().reshape(n).copy())
        rec["action_noise"].append(rt.feed.randn_like(torch.zeros(n, 2)).numpy() if rand else np.zeros((n, 2), f))
        rt.feed.sim_i = 0
        rt._patch()
        try:
            t.pre_physics_step(torch.from_numpy(a))
            rec["history_out"].append(hist()); rec["u_rail_velocity"].append(t.u_rail_velocity.numpy().reshape(n).copy())
            rec["u_fpam"].append(t.u_fpam.numpy().reshape(n).copy()); rec["smoothed_out"].append(t.smoothed_u_fpam.numpy().reshape(n).copy())
            # synthetic joint state for the actuation law; some velocity errors right at the 0.1 switch
            q = rng.normal(0, 0.3, (n, 6)).astype(f); qd = rng.normal(0, 2.0, (n, 6)).astype(f)
            cv = rng.normal(0, 0.5, n).astype(f)
            u_r = t.u_rail_velocity.numpy().reshape(n)
            cv[:32] = (u_r[:32] - np.array([0.1, -0.1, 0.1000001, -0.1000001, 0.0999999, -0.0999999, 0.0, 1e-9] * 4, f)).astype(f)
            ds = g.dof_state.view(n, 6, 2)
            ds[..., 0] = torch.from_numpy(q); ds[..., 1] = torch.from_numpy(qd)
            g.c_cart_vy[:] = cv
            pv, pe = rng.normal(0, 0.5, n).astype(f), rng.normal(0, 0.5, n).astype(f)
            t.prev_cart_vel = torch.from_numpy(pv.copy()).reshape(n, 1); t.prev_cart_vel_error = torch.from_numpy(pe.copy()).reshape(n, 1)
            t.refresh_state_tensors()
            t.compute_and_set_dof_actuation_force_tensor()
        finally:
            rt._unpatch()
        use = t.smoothed_u_fpam if cfg["env"]["USE_SMOOTHED_FPAM"] else t.u_fpam
        rec["dof_pos"].append(q); rec["dof_vel"].append(qd); rec["cart_vel_y"].append(cv)
        rec["u_fpam_to_use"].append(use.numpy().reshape(n).copy())
        rec["prev_cart_vel"].append(pv); rec["prev_cart_vel_error"].append(pe)
        rec["dynamics_scaling"].append(rt.feed.last_scale.copy() if rand else np.ones((n, 5, 4), f))
        rec["dof_efforts"].append(g.efforts.numpy().copy())
        rec["prev_cart_vel_out"].append(t.prev_cart_vel.numpy().reshape(n).copy())
        rec["prev_cart_vel_error_out"].append(t.prev_cart_vel_error.numpy().reshape(n).copy())
        rt.feed.step += 1
    out = {k: np.stack(v) for k, v in rec.items()}
    out["overrides"] = np.array(json.dumps(["num_envs=%d" % n] + list(overrides)))
    np.savez_compressed(os.path.join(HERE, "fn_pre_act_%s.npz" % name), **out)
    print("fn_pre_act_%-12s T=%d |efforts|max=%.3g" % (name, T, float(np.abs(out["dof_efforts"]).max())))


REFERENCE_CFG_UNCOMPARED = ("wandb_entity", "wandb_project", "wandb_group", "wandb_name", "wandb_tags", "wandb_logcode_dir")


def gen_reference_cfg():
    """reference_cfg.json: the reference's own cfg/ YAML files (config.yaml + task + train), composed and resolved, minus the
    author's wandb settings."""
    cfg = vcfg.compose(["task=Vine5LinkMovingBase", "train=Vine5LinkMovingBasePPO"],
                       cfg_dir=os.path.join(H.REF_ROOT, "isaacgymenvs", "cfg"))
    cfg = {k: v for k, v in cfg.items() if k not in REFERENCE_CFG_UNCOMPARED}
    with open(os.path.join(HERE, "reference_cfg.json"), "w") as f:
        json.dump(cfg, f, indent=1, sort_keys=True)
        f.write("\n")


def main():
    gen_reference_cfg()
    for name, (ov, n, T, mode) in STEP_SCENARIOS.items():
        gen_step(name, ov, n, T, mode)
    gen_fn_post_physics("default28", NO_OBST)
    gen_fn_post_physics("fstr18", FSTR_SNAPSHOT)
    gen_fn_post_physics("shelf_noise", ["task.env.CREATE_SHELF=True", "task.env.CREATE_PIPE=False",
                                        "task.env.USE_NONZERO_CONTACT_FORCE_RESET=True",
                                        "task.env.USE_TIP_LIMIT_HIT_RESET=True"] + FULL_DR)
    gen_fn_post_physics("weights", STEP_SCENARIOS["flags"][0])
    for ot in ("POS_ONLY", "POS_AND_VEL", "POS_AND_FD_VEL", "POS_AND_PREV_POS"):
        gen_fn_post_physics(ot.lower(), NO_OBST + ["OBSERVATION_TYPE=" + ot, "task.env.SCALE_OBSERVATIONS=False"], n=64)
    gen_fn_pre_and_actuation("default", NO_OBST)
    gen_fn_pre_and_actuation("dr_delay2", NO_OBST + FULL_DR + ["task.env.ACTION_DELAY=2", "task.env.RAIL_D_GAIN=0.25"])
    gen_fn_pre_and_actuation("nodelay_force", NO_OBST + ["task.env.ACTION_DELAY=0", "task.env.FORCE_U_FPAM=True",
                                                         "task.env.USE_SMOOTHED_FPAM=False", "vine_randomize=False"])


if __name__ == "__main__":
    main()
