"""ctypes mirror of ``include/vine_b200.h`` and the loader of ``libvine_b200.so``.

The product path has no CPU fallback: if the CUDA library is missing, ``load_library`` raises.
Field order below must match the header exactly (checked by ``struct_size`` in ``vine_create``
and by tests/test_abi.py).
"""
import ctypes as C
import os

NUM_DOFS = 6
NUM_ACTIONS = 2
NUM_REWARDS = 13
NUM_OBJECT_INFO = 2
MAX_ACTION_DELAY = 8
ABI_VERSION = 8

OK = 0
ERR_INVALID_ARG = -1
ERR_UNSUPPORTED = -2
ERR_CUDA = -3
ERR_NOT_BOUND = -4
ERR_ABI_MISMATCH = -5

# ObservationType (reference: isaacgymenvs/tasks/Vine5LinkMovingBase.py:67-73)
OBSERVATION_TYPES = {
    "POS_ONLY": 0,
    "POS_AND_VEL": 1,
    "POS_AND_FD_VEL": 2,
    "POS_AND_PREV_POS": 3,
    "POS_AND_FD_VEL_AND_OBJ_INFO": 4,
    "TIP_AND_CART_AND_OBJ_INFO": 5,
}
NUM_OBSERVATIONS = {0: 14, 1: 26, 2: 26, 3: 26, 4: 28, 5: 18}
TORQUE_LAW_INTEGRATION = {"zoh": 0, "implicit": 1}

# REWARD_NAMES order (reference: Vine5LinkMovingBase.py:78-81) -> cfg["env"] weight keys (:186-200)
REWARD_NAMES = ["Position", "Const Negative", "Position Success", "Velocity Success", "Velocity",
                "Rail Velocity Control", "FPAM Control", "Rail Velocity Change", "FPAM Change",
                "Rail Limit", "Cart Y", "Tip Y", "Contact Force"]
REWARD_WEIGHT_KEYS = ["POSITION_REWARD_WEIGHT", "CONST_NEGATIVE_REWARD_WEIGHT",
                      "POSITION_SUCCESS_REWARD_WEIGHT", "VELOCITY_SUCCESS_REWARD_WEIGHT",
                      "VELOCITY_REWARD_WEIGHT", "U_RAIL_VELOCITY_CONTROL_REWARD_WEIGHT",
                      "U_FPAM_CONTROL_REWARD_WEIGHT", "RAIL_VELOCITY_CHANGE_REWARD_WEIGHT",
                      "U_FPAM_CHANGE_REWARD_WEIGHT", "RAIL_LIMIT_REWARD_WEIGHT",
                      "CART_Y_REWARD_WEIGHT", "TIP_Y_REWARD_WEIGHT", "CONTACT_FORCE_REWARD_WEIGHT"]

_i32, _f64 = C.c_int32, C.c_double
_fp = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_u8p = C.POINTER(C.c_uint8)


class VineConfig(C.Structure):
    _fields_ = [
        ("struct_size", _i32), ("substeps", _i32), ("dt", _f64), ("gravity_z", _f64),
        ("control_freq_inv", _i32), ("max_episode_length", _i32),
        ("clip_observations", _f64), ("clip_actions", _f64),
        ("observation_type", _i32), ("scale_observations", _i32),
        ("create_shelf", _i32), ("create_pipe", _i32),
        ("use_smoothed_fpam", _i32), ("force_u_fpam", _i32), ("force_u_rail_velocity", _i32),
        ("action_delay", _i32),
        ("smoothing_alpha_inflate", _f64), ("smoothing_alpha_deflate", _f64),
        ("fpam_min", _f64), ("fpam_max", _f64), ("rail_velocity_scale", _f64),
        ("damping", _f64), ("stiffness", _f64),
        ("rail_soft_limit", _f64), ("rail_p_gain", _f64), ("rail_d_gain", _f64),
        ("rail_acceleration", _f64),
        ("randomize_dof_init", _i32), ("randomize_targets", _i32),
        ("random_init_cart_min_y", _f64), ("random_init_cart_max_y", _f64),
        ("success_dist", _f64),
        ("min_target_depth_in_obstacle", _f64), ("max_target_depth_in_obstacle", _f64),
        ("min_target_y", _f64), ("max_target_y", _f64),
        ("min_target_z", _f64), ("max_target_z", _f64),
        ("reward_weights", _f64 * NUM_REWARDS),
        ("use_target_reached_reset", _i32), ("use_tip_limit_hit_reset", _i32),
        ("use_nonzero_contact_force_reset", _i32),
        ("vine_randomize", _i32),
        ("dynamics_scaling_min", _f64), ("dynamics_scaling_max", _f64),
        ("observation_noise_std", _f64), ("action_noise_std", _f64),
        ("accel_target_scaling_min", _f64), ("accel_target_scaling_max", _f64),
        ("torque_law_integration", _i32), ("emulate_stale_body_state", _i32),
        ("armature", _f64),
        ("revolute_lower", _f64), ("revolute_upper", _f64),
        ("prismatic_lower", _f64), ("prismatic_upper", _f64),
        ("contact_stiffness", _f64), ("contact_damping", _f64), ("contact_rest_offset", _f64),
        ("contact_cull_slack", _f64), ("contact_binning", _i32),
    ]

    def copy(self):
        out = VineConfig()
        C.memmove(C.byref(out), C.byref(self), C.sizeof(VineConfig))
        return out


class VineStateView(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "dof_pos", "dof_vel", "tip_positions", "cart_body_vel_y", "target_positions", "object_info",
        "smoothed_u_fpam", "prev_cart_vel", "prev_cart_vel_error", "shelf_contact_force",
        "actions_history", "aggregated_rew_buf")] + [("step_count", _i64p)] + [(n, _fp) for n in (
        "u_rail_velocity", "u_fpam", "prev_u_rail_velocity", "rail_force", "tip_velocities",
        "reward_matrix", "finite_difference_dof_vel", "finite_difference_tip_velocities", "cart_body_pos_y")]


class VinePostPhysicsIO(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "dof_pos", "dof_vel", "prev_dof_pos", "tip_positions", "prev_tip_positions", "tip_velocities",
        "cart_positions_y", "target_positions", "target_velocities", "smoothed_u_fpam", "u_fpam",
        "u_rail_velocity", "prev_u_rail_velocity", "object_info", "contact_force_norms", "obs_noise")] + [
        ("reset_buf_in", _i64p), ("progress_buf", _i64p),
        ("obs_buf", _fp), ("rew_buf", _fp), ("reward_matrix", _fp),
        ("reset_buf_out", _i64p), ("timeout_buf", _u8p)]


class VinePrePhysicsIO(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "actions", "action_noise", "history_in", "smoothed_in", "history_out", "u_rail_velocity",
        "u_fpam", "smoothed_out")]


class VineActuationIO(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "dof_pos", "dof_vel", "cart_vel_y", "u_rail_velocity", "u_fpam_to_use", "prev_cart_vel",
        "prev_cart_vel_error", "dynamics_scaling", "accel_scaling", "dof_efforts",
        "prev_cart_vel_out", "prev_cart_vel_error_out")]


class VineSimulateIO(C.Structure):
    _fields_ = [(n, _fp) for n in (
        "dof_pos", "dof_vel", "dof_efforts", "dynamics_scaling", "u_fpam_to_use", "target_positions",
        "object_info", "tip_positions", "tip_velocities", "shelf_contact_force")]


# every symbol include/vine_b200.h declares
EXPORTED_SYMBOLS = [
    "vine_abi_version", "vine_config_defaults", "vine_num_observations", "vine_create",
    "vine_destroy", "vine_last_error", "vine_bind_io", "vine_step", "vine_step_range", "vine_route_counts", "vine_reset_idx",
    "vine_get_state", "vine_set_state", "vine_set_debug_outputs", "vine_metrics", "vine_post_physics",
    "vine_pre_physics", "vine_actuation", "vine_simulate", "vine_philox_debug", "vine_gae",
    "vine_mlp_pack", "vine_mlp_forward",
    "vine_ppo_num_params", "vine_ppo_max_ctas", "vine_ppo_minibatch", "vine_ppo_reduce", "vine_ppo_adam",
    "vine_p2p_alloc", "vine_p2p_open", "vine_p2p_close", "vine_p2p_free", "vine_p2p_channel_create", "vine_p2p_channel_status",
    "vine_p2p_channel_timing", "vine_p2p_allreduce_f64", "vine_p2p_channel_destroy",
    "vine_policy_act", "vine_rollout_post", "vine_ppo_moments", "vine_ppo_finalize",
    "vine_lstm_cell_fwd", "vine_lstm_cell_bwd", "vine_lstm_pack", "vine_lstm_step", "vine_lstm_mask", "vine_lstm_head", "vine_lstm_head_train", "vine_lstm_cell_bwd_tiles", "vine_lstm_bwd_gemm",
    "vine_set_programmatic_launch", "vine_lstm_gather", "vine_abi_struct_size", "vine_lstm_num_params", "vine_lstm_wgrad", "vine_lstm_reduce", "vine_lstm_adam",
    "vine_grad_clip", "vine_ppo_adam_clipped", "vine_lstm_adam_clipped",
]
METRIC_SUMS, METRIC_MAXES = 45, 30
METRIC_SCALARS = ["dist_tip_to_target", "target_reached", "limit_hit", "tip_limit_hit", "abs_tip_y", "tip_z", "tip_velocities",
                  "u_rail_velocity", "prev_u_rail_velocity", "rail_force", "u_fpam", "smoothed_u_fpam",
                  "tip_target_velocity_difference", "progress_buf", "contact_forces", "nonzero_contact_force"]
MLP_PACKED_BYTES = 102208
LSTM_PACKED_BYTES = 795664
LSTM_HEAD_GRAD_FLOATS = 1296
LSTM_HEAD_GRAD_PARTS = 1184
LSTM_WGRAD_BLOCK_FLOATS = 12 * 128 * 256      # per K split
LSTM_TILE_BYTES = 32768          # one [128 x 128] bf16 activation tile
PPO_WS_FLOATS = 49664
PPO_STATE_FLOATS = 16
PPO_STATE_CLIP_COEF, PPO_STATE_GRAD_NORM = 9, 10   # slots of the state block written by vine_grad_clip
PPO_STATE_EPOCH, PPO_STATE_EPOCH_KL_SUM, PPO_STATE_EPOCH_KL_COUNT = 11, 12, 13   # learning-rate schedule (vine_ppo_minibatch)
GRAD_CLIP_WS_FLOATS = 1024


class VinePolicyAct(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in (
        "packed", "obs", "obs_mean", "obs_inv_std", "value_stats", "mu", "value", "logstd", "rng_counter", "actions",
        "neglogp", "obs_copy", "env_actions")]
        + [("n", C.c_int64), ("num_obs", C.c_int32), ("raw_obs", C.c_int32), ("seed", C.c_uint64),
           ("global_env_offset", C.c_int64), ("u_out", C.c_void_p), ("u_step_rows", C.c_int32), ("u_step_seqs", C.c_int32),
           ("raw_value", C.c_int32), ("u_no_obs", C.c_int32)])


class VineLstmStep(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("params", "u", "hm", "c_prev", "not_done", "not_done_next", "c", "hh", "hm_next",
                                          "act")] + [("n", C.c_int64), ("hm_next_rows", C.c_int64)]


class VineLstmHead(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("params", "hh", "value_stats", "mu", "value", "logstd", "rng_counter", "actions",
                                           "neglogp", "env_actions")]
                + [("n", C.c_int64), ("seed", C.c_uint64), ("global_env_offset", C.c_int64), ("raw_value", C.c_int32),
                   ("no_layer_norm", C.c_int32)])


class VineLstmHeadTrain(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("params", "hh", "scalars", "logstd", "logstd_old", "dh", "grads", "debug_out")]
                + [("n", C.c_int64)]
                + [(n, C.c_float) for n in ("e_clip", "critic_coef", "entropy_coef", "bounds_loss_coef", "inv_B")]
                + [("step_rows", C.c_int32), ("mu_writeback", C.c_void_p)]
                + [(n, C.c_int64) for n in ("wb_seq_len", "wb_chunks", "wb_num_envs", "wb_env_begin", "wb_env_count")]
                + [("value_loss_unclipped", C.c_int32), ("step_seqs", C.c_int32), ("no_layer_norm", C.c_int32),
                   ("reserved", C.c_int32)])


class VineLstmCellBwd(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("act", "c_prev", "c", "not_done", "dh", "dh_rec", "dc_next", "dg", "dc_prev")] + [("n", C.c_int64)]


class VineLstmBwdGemm(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("params", "dg", "not_done", "dh3", "dh_rec")] + [("n", C.c_int64), ("dh3_rows", C.c_int64)]


class VineLstmGather(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("obs", "scalars", "not_done", "c_saved", "hh_saved", "mb_obs", "mb_scalars", "mb_not_done",
                                           "c0", "hm0")]
                + [(n, C.c_int32) for n in ("seq_len", "chunks", "num_envs", "env_begin", "env_count", "num_obs",
                                             "step_rows", "reserved")])


class VineLstmWgrad(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("u", "hm", "dg", "workspace")] + [("ntiles", C.c_int64), ("splits", C.c_int32), ("reserved", C.c_int32)]


class VineRolloutPost(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in (
        "rewards", "resets", "timeouts", "values", "shaped_rewards", "dones_next", "ep_return", "ep_length", "ep_stats",
        "rng_counter")]
        + [("n", C.c_int64), ("reward_scale", C.c_float), ("gamma", C.c_float), ("value_bootstrap", C.c_int32),
           ("success_reward_threshold", C.c_float), ("not_done_next", C.c_void_p),
           ("reward_shift", C.c_float), ("reward_min", C.c_float), ("reward_max", C.c_float), ("reward_clamp", C.c_int32)])


class VinePpoPrologue(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in (
        "obs", "values", "returns", "moments", "obs_mean", "obs_var", "obs_count", "val_mean", "val_var", "val_count",
        "obs_mean_f", "obs_inv_std_f", "value_stats", "adv_stats", "values_n", "returns_n", "advantages_n")]
        + [("count", C.c_int64), ("num_obs", C.c_int32), ("world", C.c_int32), ("normalize_advantage", C.c_int32),
           ("raw_obs", C.c_int32), ("raw_value", C.c_int32), ("reserved", C.c_int32)])


class VinePpoMinibatch(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in (
        "packed", "obs", "actions", "mu_old", "neglogp_old", "values_old", "returns", "advantages", "obs_mean",
        "obs_inv_std", "logstd", "logstd_old", "workspace", "state", "debug_out")]
        + [(n, C.c_int32) for n in ("horizon", "num_envs", "env_begin", "env_count", "num_obs", "workspace_ctas",
                                    "adaptive_lr", "reserved")]
        + [(n, C.c_float) for n in ("e_clip", "critic_coef", "entropy_coef", "bounds_loss_coef", "kl_threshold",
                                    "lr_min", "lr_max", "reserved_f")]
        + [("dh3_ext", C.c_void_p)]
        + [(n, C.c_int32) for n in ("lr_linear", "schedule_standard", "epoch_begin", "mini_epoch_begin", "max_epochs",
                                    "value_loss_unclipped")]
        + [("lr0", C.c_float), ("raw_obs", C.c_int32)])

# argument structs of the PPO entry points in the order of vine_abi_struct_size()
PPO_STRUCTS = [VinePolicyAct, VineRolloutPost, VinePpoPrologue, VinePpoMinibatch, VineLstmStep, VineLstmHead, VineLstmHeadTrain,
               VineLstmCellBwd, VineLstmBwdGemm, VineLstmWgrad, VineLstmGather]

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "csrc", "libvine_b200.so")
_lib = None


def _declare(lib):
    vp = C.c_void_p
    lib.vine_abi_version.restype = C.c_int
    lib.vine_config_defaults.argtypes = [C.POINTER(VineConfig)]
    lib.vine_num_observations.argtypes = [C.c_int]
    lib.vine_create.argtypes = [C.POINTER(VineConfig), C.c_int64, C.c_int64, C.c_int, C.c_uint64,
                                C.POINTER(vp)]
    lib.vine_destroy.argtypes = [vp]
    lib.vine_destroy.restype = None
    lib.vine_last_error.argtypes = [vp]
    lib.vine_last_error.restype = C.c_char_p
    lib.vine_bind_io.argtypes = [vp] + [vp] * 7
    lib.vine_step.argtypes = [vp, vp]
    lib.vine_step_range.argtypes = [vp, C.c_int64, C.c_int64, vp]
    lib.vine_route_counts.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.vine_reset_idx.argtypes = [vp, vp, C.c_int64, vp]
    lib.vine_get_state.argtypes = [vp, C.POINTER(VineStateView), vp]
    lib.vine_set_state.argtypes = [vp, C.POINTER(VineStateView), vp]
    lib.vine_set_debug_outputs.argtypes = [vp, C.c_int]
    lib.vine_metrics.argtypes = [vp, vp, vp, vp]
    lib.vine_post_physics.argtypes = [vp, C.POINTER(VinePostPhysicsIO), vp]
    lib.vine_pre_physics.argtypes = [vp, C.POINTER(VinePrePhysicsIO), vp]
    lib.vine_actuation.argtypes = [vp, C.POINTER(VineActuationIO), vp]
    lib.vine_simulate.argtypes = [vp, C.POINTER(VineSimulateIO), vp]
    lib.vine_philox_debug.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                      C.c_int64, vp, vp]
    lib.vine_gae.argtypes = [vp, vp, vp, vp, vp, C.c_int64, C.c_int64, C.c_double, C.c_double,
                             vp, vp, vp]
    lib.vine_mlp_pack.argtypes = [vp] * 10 + [C.c_int, vp, vp]
    lib.vine_mlp_forward.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int, vp, vp, vp, vp]
    lib.vine_policy_act.argtypes = [C.POINTER(VinePolicyAct), vp]
    lib.vine_rollout_post.argtypes = [C.POINTER(VineRolloutPost), vp]
    lib.vine_ppo_moments.argtypes = [C.POINTER(VinePpoPrologue), vp]
    lib.vine_ppo_finalize.argtypes = [C.POINTER(VinePpoPrologue), vp]
    lib.vine_lstm_cell_fwd.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int, vp, vp, vp, vp, vp]
    lib.vine_lstm_cell_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.c_int64, C.c_int, vp, vp, vp]
    lib.vine_lstm_pack.argtypes = [vp] * 10 + [C.c_int, vp, vp]
    lib.vine_lstm_step.argtypes = [C.POINTER(VineLstmStep), vp]
    lib.vine_lstm_mask.argtypes = [vp, vp, C.c_int64, vp, vp]
    lib.vine_lstm_head.argtypes = [C.POINTER(VineLstmHead), vp]
    lib.vine_lstm_head_train.argtypes = [C.POINTER(VineLstmHeadTrain), vp]
    lib.vine_lstm_cell_bwd_tiles.argtypes = [C.POINTER(VineLstmCellBwd), vp]
    lib.vine_lstm_bwd_gemm.argtypes = [C.POINTER(VineLstmBwdGemm), vp]
    lib.vine_lstm_gather.argtypes = [C.POINTER(VineLstmGather), vp]
    lib.vine_abi_struct_size.argtypes = [C.c_int]
    lib.vine_set_programmatic_launch.argtypes = [C.c_int]
    lib.vine_lstm_num_params.argtypes = [C.c_int]
    lib.vine_lstm_wgrad.argtypes = [C.POINTER(VineLstmWgrad), vp]
    lib.vine_lstm_reduce.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, vp, vp, vp]
    lib.vine_lstm_adam.argtypes = [vp, C.c_float, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_float, C.c_float, vp, vp]
    lib.vine_ppo_num_params.argtypes = [C.c_int]
    lib.vine_ppo_max_ctas.argtypes = []
    lib.vine_ppo_minibatch.argtypes = [C.POINTER(VinePpoMinibatch), vp]
    lib.vine_ppo_reduce.argtypes = [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp]
    lib.vine_ppo_adam.argtypes = [vp, C.c_float, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp]
    lib.vine_ppo_adam_clipped.argtypes = [vp, C.c_float, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, vp, vp, vp]
    lib.vine_lstm_adam_clipped.argtypes = [vp, C.c_float, vp, vp, vp, vp, vp, C.c_int, C.c_float, C.c_float, C.c_float, vp, vp, vp]
    lib.vine_grad_clip.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_float, C.c_float, vp, vp, vp, vp, vp]
    lib.vine_p2p_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p), vp]
    lib.vine_p2p_open.argtypes = [vp, C.POINTER(C.c_void_p)]
    lib.vine_p2p_close.argtypes = [vp]
    lib.vine_p2p_free.argtypes = [vp]
    lib.vine_p2p_channel_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_void_p)]
    lib.vine_p2p_channel_status.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    lib.vine_p2p_channel_timing.argtypes = [vp, C.POINTER(C.c_double), C.c_int]
    lib.vine_p2p_allreduce_f64.argtypes = [vp, vp, C.c_int, vp]
    lib.vine_p2p_channel_destroy.argtypes = [vp]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("vine_destroy", "vine_last_error"):
            fn.restype = C.c_int
    return lib


def load_library(path=None):
    """Load libvine_b200.so (built in-tree by ``__graft_entry__.build()``).  No fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("VINE_B200_LIB") or LIB_PATH   # env override: kernel-variant experiments
    if not os.path.exists(p):
        raise RuntimeError(
            f"{p} not found: the Vine5LinkMovingBase hot path is CUDA-only (sm_100a) and has no "
            "CPU fallback. Build it with `python -c 'import __graft_entry__ as g; g.build()'`.")
    lib = _declare(C.CDLL(p))
    v = lib.vine_abi_version()
    if v != ABI_VERSION:
        raise RuntimeError(f"libvine_b200.so ABI version {v} != expected {ABI_VERSION}")
    if path is None:
        _lib = lib
    return lib


def default_config():
    """Defaults of cfg/task/Vine5LinkMovingBase.yaml, as produced by the library itself."""
    cfg = VineConfig()
    rc = load_library().vine_config_defaults(C.byref(cfg))
    if rc != OK:
        raise RuntimeError(f"vine_config_defaults failed: {rc}")
    return cfg
