/*
 * vine_b200.h — C ABI of the B200-native Vine5LinkMovingBase hot path.
 *
 * The reference (tylerlum/Vine_Robot_IsaacGymEnvs) has no native code and no FFI of its
 * own: its per-control-step pipeline is Python/torch (isaacgymenvs/tasks/Vine5LinkMovingBase.py,
 * "V5") on top of the closed Isaac Gym binary (gymapi.simulate & friends) and the
 * VecTask base class (isaacgymenvs/tasks/base/vec_task.py, "VT").  This header is the
 * boundary a maintainer would bind (ctypes, see INTEGRATION.md) to replace that pipeline.
 * Every entry point cites the reference interface it stands in for.
 *
 * Conventions
 *   - plain C, no torch types; all array arguments are DEVICE pointers unless the
 *     name ends in `_host`; row-major; the caller (PyTorch) owns every I/O buffer.
 *   - every function returns 0 (VINE_OK) or a negative VineStatus; no C++ exception,
 *     exit() or abort() crosses the ABI (contrast VT:297-299 `quit()`).
 *   - all work is enqueued on the `stream` argument (a cudaStream_t passed as void*);
 *     no entry point synchronises the device or allocates after vine_create(), so
 *     vine_step() is CUDA-graph capturable.
 *   - one host thread per handle; handles on different devices are independent
 *     (one per rank; envs never communicate, V5:464).
 */
#ifndef VINE_B200_H_
#define VINE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VINE_ABI_VERSION 5

#define VINE_NUM_DOFS 6          /* 1 prismatic rail cart + 5 revolute links (V5:54,83) */
#define VINE_NUM_ACTIONS 2       /* u_rail_velocity, u_fpam (V5:171) */
#define VINE_NUM_REWARDS 13      /* REWARD_NAMES (V5:78-81) */
#define VINE_NUM_OBJECT_INFO 2   /* target depth, angle (V5:51) */
#define VINE_MAX_ACTION_DELAY 8
#define VINE_NUM_METRICS 96

typedef enum VineStatus {
  VINE_OK = 0,
  VINE_ERR_INVALID_ARG = -1,
  VINE_ERR_UNSUPPORTED = -2,     /* e.g. SCALE_OBSERVATIONS with a type V5:267-268 rejects */
  VINE_ERR_CUDA = -3,
  VINE_ERR_NOT_BOUND = -4,
  VINE_ERR_ABI_MISMATCH = -5
} VineStatus;

/* ObservationType (V5:67-73); widths V5:152-171. */
typedef enum VineObservationType {
  VINE_OBS_POS_ONLY = 0,                    /* 14 */
  VINE_OBS_POS_AND_VEL = 1,                 /* 26 */
  VINE_OBS_POS_AND_FD_VEL = 2,              /* 26 */
  VINE_OBS_POS_AND_PREV_POS = 3,            /* 26 */
  VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO = 4, /* 28 */
  VINE_OBS_TIP_AND_CART_AND_OBJ_INFO = 5    /* 18 */
} VineObservationType;

/* How the reference's joint torque law tau = -(K q + C qd + b + B u) (V5:1042-1062)
 * enters the integrator. ZOH = literal reference semantics (efforts frozen for one sim
 * step, VT:346-356).  IMPLICIT = the spring/damper part is integrated implicitly per
 * substep (unconditionally stable; see DESIGN.md "R1"). */
typedef enum VineTorqueLawIntegration {
  VINE_TORQUE_LAW_ZOH = 0,
  VINE_TORQUE_LAW_IMPLICIT = 1
} VineTorqueLawIntegration;

/*
 * Mirror of the reference's configuration surface for this path:
 * cfg["env"], cfg["sim"], cfg["task"] of cfg/task/Vine5LinkMovingBase.yaml.
 * Real-valued knobs are `double` because the reference holds them as Python floats and
 * rounds to f32 only where they meet a tensor; the library derives its f32 constants the
 * same way.
 */
typedef struct VineConfig {
  int32_t struct_size;                 /* = sizeof(VineConfig), checked by vine_create */
  /* sim.* (YT:102-123) */
  int32_t substeps;
  double dt;
  double gravity_z;
  /* env.* (YT:7-100) */
  int32_t control_freq_inv;
  int32_t max_episode_length;
  double clip_observations;
  double clip_actions;
  int32_t observation_type;            /* VineObservationType */
  int32_t scale_observations;
  int32_t create_shelf;
  int32_t create_pipe;
  int32_t use_smoothed_fpam;
  int32_t force_u_fpam;
  int32_t force_u_rail_velocity;
  int32_t action_delay;
  double smoothing_alpha_inflate;
  double smoothing_alpha_deflate;
  double fpam_min;
  double fpam_max;
  double rail_velocity_scale;
  double damping;                      /* PhysX DOF damping on all 6 DOFs (V5:504) */
  double stiffness;                    /* PhysX DOF stiffness on revolutes (V5:511) */
  double rail_soft_limit;
  double rail_p_gain;
  double rail_d_gain;
  double rail_acceleration;
  int32_t randomize_dof_init;
  int32_t randomize_targets;
  double random_init_cart_min_y;
  double random_init_cart_max_y;
  double success_dist;
  double min_target_depth_in_obstacle;
  double max_target_depth_in_obstacle;
  double min_target_y;
  double max_target_y;
  double min_target_z;
  double max_target_z;
  double reward_weights[VINE_NUM_REWARDS];   /* REWARD_NAMES order (V5:186-203) */
  int32_t use_target_reached_reset;
  int32_t use_tip_limit_hit_reset;
  int32_t use_nonzero_contact_force_reset;
  /* task.* (YT:125-134; ACCEL_TARGET_SCALING_* only on README.md:63) */
  int32_t vine_randomize;
  double dynamics_scaling_min;
  double dynamics_scaling_max;
  double observation_noise_std;
  double action_noise_std;
  double accel_target_scaling_min;
  double accel_target_scaling_max;
  /* Simulator-side parameters the reference leaves to Isaac Gym (SURVEY App. F). */
  int32_t torque_law_integration;      /* VineTorqueLawIntegration */
  int32_t emulate_stale_body_state;    /* replicate rigid-body staleness after reset (V5:796) */
  double armature;                     /* added to every revolute joint-space inertia */
  double revolute_lower;               /* dof_props lower/upper of limit-less joints (V5:778-786) */
  double revolute_upper;
  double prismatic_lower;
  double prismatic_upper;
  double contact_stiffness;            /* penalty contact, N/m */
  double contact_damping;              /* N s/m */
  double contact_rest_offset;          /* YT:117 */
  /* Launch tuning of the library itself (no counterpart in the reference; results do not depend on them). */
  double contact_cull_slack;           /* obstacle variants: metres a chain may move before its candidate (link,
                                          rectangle) pairs are re-culled; <= 0 selects the default 0.01 */
  int32_t contact_binning;             /* obstacle variants: order envs by "had contact candidates" before launches of
                                          >= 98,304 envs (1 = default) or keep the identity order (0) */
} VineConfig;

typedef struct VineEnv VineEnv;

/* Version of this header the library was built against. */
int vine_abi_version(void);

/*
 * Programmatic dependent launch (process-wide, default OFF): when on, the short dependent kernels of the PPO iteration and
 * the single-launch env step are launched with cudaLaunchAttributeProgrammaticStreamSerialization and begin with
 * griddepcontrol.wait, so that a kernel's launch latency overlaps the tail of its predecessor in the stream (memory semantics
 * unchanged: nothing is read or written before the predecessors have completed).  0 = plain stream-ordered launches.
 * Returns the previous setting.  Launches already captured in a CUDA graph keep the mode they were captured with.
 */
int vine_set_programmatic_launch(int enabled);

/* Fill `cfg` with the defaults of cfg/task/Vine5LinkMovingBase.yaml (YT:7-134). */
int vine_config_defaults(VineConfig* cfg);

/* Observation width for a type (V5:152-171); negative on bad type. */
int vine_num_observations(int observation_type);

/*
 * Replaces Vine5LinkMovingBase.__init__ / create_sim / _create_envs /
 * initialize_state_tensors (V5:137-291, 299-362, 364-519) and VecTask.__init__
 * (VT:169-223): validates the config, bakes the model constants, allocates the private
 * SoA state for `num_envs` environments on CUDA device `device`.  Envs are numbered
 * global_env_offset .. global_env_offset+num_envs-1; the Philox key is (seed, global id)
 * so results do not depend on how envs are sharded over ranks.
 */
int vine_create(const VineConfig* cfg, int64_t num_envs, int64_t global_env_offset,
                int device, uint64_t seed, VineEnv** out);

void vine_destroy(VineEnv* env);

/* Last error text for this handle (or the last vine_create failure when env==NULL). */
const char* vine_last_error(const VineEnv* env);

/*
 * Borrow the VecTask buffers (VT:260-283): actions f32[N,2]; obs_buf f32[N,O];
 * rew_buf f32[N]; reset_buf i64[N]; progress_buf i64[N]; timeout_buf u8[N] (torch.bool);
 * obs_clamped f32[N,O] = clamp(obs_buf, +-clipObservations) (VT:374), may be NULL.
 */
int vine_bind_io(VineEnv* env, const float* actions, float* obs_buf, float* rew_buf,
                 int64_t* reset_buf, int64_t* progress_buf, uint8_t* timeout_buf,
                 float* obs_clamped);

/*
 * One control step == VecTask.step (VT:319-380): clamp actions, pre_physics_step
 * (V5:922-945), controlFrequencyInv x {forces V5:1028-1106, shelf contact sample
 * VT:348-351, simulate VT:356}, post_physics_step (V5:1110-1120: progress, deferred
 * reset_idx, observations, reward, reset), timeout (VT:366), obs clamp (VT:374).
 * ONE fused kernel launch; with obstacles (CREATE_SHELF / CREATE_PIPE) and at least 98,304 envs it is preceded by a
 * 8-byte memset and one ordering kernel (envs that had contact candidates in their last step share warps; results do not
 * depend on the order; VINE_CONTACT_BINNING=0 in the environment at vine_create turns it off). No allocation, no host
 * synchronisation, CUDA-graph capturable in either case.
 */
int vine_step(VineEnv* env, void* stream);

/*
 * The same step for the env sub-range [first, first+count) only (first a multiple of 128).
 * Envs are independent (V5:464), so a step may be issued as several range launches on different
 * streams to overlap host<->device copies of one chunk with the compute of another; the union of
 * ranges covering 0..num_envs is bit-identical to one vine_step.
 */
int vine_step_range(VineEnv* env, int64_t first, int64_t count, void* stream);
/* Obstacle variants, routed step: how the last vine_step binned its envs -- out = {near (near pass), far (far pass), given up by
 * the far pass and redone, 0}.  Zeros when the step is not routed.  Synchronises. */
int vine_route_counts(VineEnv* env, int64_t out[4]);

/*
 * reset_idx(env_ids) (V5:774-885) outside step, as VecTask.reset_done (VT:412-427)
 * and the 'R' key (V5:715-718) call it.  `env_ids` i64[n] device pointer, local ids.
 */
int vine_reset_idx(VineEnv* env, const int64_t* env_ids, int64_t n, void* stream);

/*
 * Structure-of-arrays snapshot of the private state, for identical-state parity tests
 * and for exposing dof_pos etc. as torch tensors. Any pointer may be NULL (skipped).
 */
typedef struct VineStateView {
  float* dof_pos;              /* [N,6]  (V5:303) */
  float* dof_vel;              /* [N,6]  (V5:304) */
  float* tip_positions;        /* [N,3]  rigid-body view as of the last simulate (V5:357) */
  float* cart_body_vel_y;      /* [N]    cart_velocities[:,1] as of the last simulate (V5:362) */
  float* target_positions;     /* [N,3]  (V5:179) */
  float* object_info;          /* [N,2]  (V5:238) */
  float* smoothed_u_fpam;      /* [N]    (V5:224) */
  float* prev_cart_vel;        /* [N]    (V5:235) */
  float* prev_cart_vel_error;  /* [N]    (V5:234) */
  float* shelf_contact_force;  /* [N]    |net contact force on shelf_link| of the last simulate (VT:349-350) */
  float* actions_history;      /* [N,ACTION_DELAY,2] oldest first (V5:288-291) */
  float* aggregated_rew_buf;   /* [N]    (V5:183) */
  int64_t* step_count;         /* [N]    control steps taken (Philox counter) */
  /* outputs of the last step only (ignored by vine_set_state) */
  float* u_rail_velocity;      /* [N] */
  float* u_fpam;               /* [N] */
  float* prev_u_rail_velocity; /* [N] */
  float* rail_force;           /* [N] */
  float* tip_velocities;       /* [N,3] */
  float* reward_matrix;        /* [N,13] unweighted terms of the last step (V5:1500) */
  float* finite_difference_dof_vel;          /* [N,6] (q - prev_q) / control_dt (V5:1347) */
  float* finite_difference_tip_velocities;   /* [N,3] (tip - prev_tip) / control_dt (V5:1348) */
  float* cart_body_pos_y;                    /* [N] cart_positions[:,1], the rigid-body view the reward reads (V5:1231): equals
                                                dof_pos[:,0] except on a reset step, where it is still the old episode's */
} VineStateView;

int vine_get_state(VineEnv* env, const VineStateView* view, void* stream);
int vine_set_state(VineEnv* env, const VineStateView* view, void* stream);

/* When enabled, vine_step also records the `outputs of the last step` block above. */
int vine_set_debug_outputs(VineEnv* env, int enabled);

/*
 * The aggregate entries of the reference's per-step wandb dict (compute_reward, V5:1250-1322) in ONE reduction
 * launch, no host synchronisation (the reference calls `.item()` ~100 times per step).  Needs
 * vine_set_debug_outputs(env, 1).  Over all envs of this handle:
 *   sums f64[VINE_METRIC_SUMS]:  [0..15] dist_tip_to_target, target_reached, limit_hit, tip_limit_hit, abs_tip_y,
 *     tip_z, tip_velocities, u_rail_velocity, prev_u_rail_velocity, rail_force, u_fpam, smoothed_u_fpam,
 *     tip_target_velocity_difference, progress_buf, contact_forces, nonzero_contact_force;
 *     [16..28] the 13 reward terms (REWARD_NAMES order, V5:78-81); [29..41] the same weighted; [42] total reward;
 *     [43] aggregated reward; [44] aggregated reward squared.   (divide by num_envs for the means)
 *   maxes f32[VINE_METRIC_MAXES]: [0] max_abs_tip_y, [1] max_tip_z, [2] tip_velocities_max, [3..15] max reward
 *     terms, [16..28] max weighted terms, [29] max total reward.
 * Multi-GPU: all-reduce sums (SUM) and maxes (MAX) across ranks.
 */
#define VINE_METRIC_SUMS 45
#define VINE_METRIC_MAXES 30
int vine_metrics(VineEnv* env, double* sums, float* maxes, void* stream);

/* ---- function-level entry points (same device code as the fused step; used for parity
 *      with the reference's own functions on identical inputs) ---- */

/*
 * compute_observations (V5:1339-1390) + compute_reward (V5:1218-1248, 1272-1278,
 * compute_reward_jit V5:1470-1537) + compute_reset_jit (V5:1540-1558) + timeout (VT:366).
 * Inputs are the tensors those functions read.  progress_buf is the value AFTER the
 * `+= 1` of V5:1111.
 */
typedef struct VinePostPhysicsIO {
  const float* dof_pos;              /* [N,6] */
  const float* dof_vel;              /* [N,6] */
  const float* prev_dof_pos;         /* [N,6] */
  const float* tip_positions;        /* [N,3] */
  const float* prev_tip_positions;   /* [N,3] */
  const float* tip_velocities;       /* [N,3] */
  const float* cart_positions_y;     /* [N] */
  const float* target_positions;     /* [N,3] */
  const float* target_velocities;    /* [N,3] */
  const float* smoothed_u_fpam;      /* [N] */
  const float* u_fpam;               /* [N] */
  const float* u_rail_velocity;      /* [N] */
  const float* prev_u_rail_velocity; /* [N] */
  const float* object_info;          /* [N,2] */
  const float* contact_force_norms;  /* [control_freq_inv,N] (VT:351) or NULL */
  const float* obs_noise;            /* [N,O] standard normals or NULL (V5:1389) */
  const int64_t* reset_buf_in;       /* [N] */
  const int64_t* progress_buf;       /* [N] */
  float* obs_buf;                    /* [N,O] out */
  float* rew_buf;                    /* [N] out */
  float* reward_matrix;              /* [N,13] out */
  int64_t* reset_buf_out;            /* [N] out */
  uint8_t* timeout_buf;              /* [N] out */
} VinePostPhysicsIO;

int vine_post_physics(VineEnv* env, const VinePostPhysicsIO* io, void* stream);

/*
 * pre_physics_step's action path (V5:927-940): raw_actions_to_actions, delay ring,
 * FORCE_* overrides, pressure smoothing.  action_noise: [N,2] standard normals or NULL.
 * history_in/out: [N,ACTION_DELAY,2] oldest first.
 */
typedef struct VinePrePhysicsIO {
  const float* actions;          /* [N,2] already clamped (VT:333) */
  const float* action_noise;     /* [N,2] or NULL */
  const float* history_in;       /* [N,D,2] */
  const float* smoothed_in;      /* [N] */
  float* history_out;            /* [N,D,2] */
  float* u_rail_velocity;        /* [N] */
  float* u_fpam;                 /* [N] */
  float* smoothed_out;           /* [N] */
} VinePrePhysicsIO;

int vine_pre_physics(VineEnv* env, const VinePrePhysicsIO* io, void* stream);

/*
 * compute_and_set_dof_actuation_force_tensor (V5:1028-1106).  dynamics_scaling: [N,5,4]
 * multipliers of (K,C,b,B) per joint or NULL (=1); accel_scaling [N] or NULL.
 */
typedef struct VineActuationIO {
  const float* dof_pos;              /* [N,6] */
  const float* dof_vel;              /* [N,6] */
  const float* cart_vel_y;           /* [N] cart_velocities[:,1] */
  const float* u_rail_velocity;      /* [N] */
  const float* u_fpam_to_use;        /* [N] smoothed or raw (V5:1059) */
  const float* prev_cart_vel;        /* [N] */
  const float* prev_cart_vel_error;  /* [N] */
  const float* dynamics_scaling;     /* [N,5,4] or NULL */
  const float* accel_scaling;        /* [N] or NULL */
  float* dof_efforts;                /* [N,6] out */
  float* prev_cart_vel_out;          /* [N] out */
  float* prev_cart_vel_error_out;    /* [N] out */
} VineActuationIO;

int vine_actuation(VineEnv* env, const VineActuationIO* io, void* stream);

/*
 * gym.simulate (VT:356) for one sim step (`substeps` substeps of dt/substeps) with the
 * given efforts held constant; replaces PhysX for this articulation.  obstacle state is
 * taken from target_positions/object_info.  In/out dof state [N,6]; outputs the
 * rigid-body views the task reads (tip pos/vel, shelf_link contact norm).
 */
typedef struct VineSimulateIO {
  float* dof_pos;                    /* [N,6] in/out */
  float* dof_vel;                    /* [N,6] in/out */
  const float* dof_efforts;          /* [N,6] */
  const float* dynamics_scaling;     /* [N,5,4] or NULL; used only by IMPLICIT mode */
  const float* u_fpam_to_use;        /* [N] used only by IMPLICIT mode */
  const float* target_positions;     /* [N,3] */
  const float* object_info;          /* [N,2] */
  float* tip_positions;              /* [N,3] out */
  float* tip_velocities;             /* [N,3] out */
  float* shelf_contact_force;        /* [N] out */
} VineSimulateIO;

int vine_simulate(VineEnv* env, const VineSimulateIO* io, void* stream);

/* Raw Philox4x32-10 stream used for all domain randomization (north_star f):
 * out u32[n_blocks*4] for counter (gid, site, step, block0+i), key = seed. */
int vine_philox_debug(uint64_t seed, uint32_t gid, uint32_t site, uint32_t step,
                      uint32_t block0, int64_t n_blocks, uint32_t* out, void* stream);

/* ---- PPO side (rl_games 1.5.2 A2CAgent pieces; in-repo analogue
 *      isaacgymenvs/learning/common_agent.py:413-425) ---- */

/*
 * discount_values: GAE over the horizon. rewards/values/dones f32[T,N] (dones as 0/1),
 * last_values f32[N], last_dones f32[N]; out advantages f32[T,N], returns f32[T,N].
 *   delta_t = r_t + gamma V_{t+1} (1-d_{t+1}) - V_t ;  A_t = delta_t + gamma tau (1-d_{t+1}) A_{t+1}
 */
int vine_gae(const float* rewards, const float* values, const float* dones,
             const float* last_values, const float* last_dones, int64_t horizon,
             int64_t num_envs, double gamma, double tau, float* advantages, float* returns,
             void* stream);

/*
 * Actor-critic MLP of cfg/train/Vine5LinkMovingBasePPO.yaml:10-30 (rl_games `actor_critic` network:
 * shared MLP [256,128,64] ELU, mu head [2], value head [1]) as ONE fused tcgen05/TMEM kernel for
 * rollout inference (rl_games A2CAgent.get_action_values; in-repo analogue
 * learning/common_agent.py:257-314).  Weights are nn.Linear layout f32 [out,in]; vine_mlp_pack
 * converts them to bf16 in the tensor-core operand layout (call it after every optimizer step).
 *   x = clamp((obs - obs_mean) * obs_inv_std, +-5);  mu f32[N,2];  value f32[N] de-normalised as
 *   clamp(v, +-5) * value_stats[1] + value_stats[0]  (rl_games RunningMeanStd, normalize_input /
 *   normalize_value; value_stats = device pointer to {mean, std} so a captured CUDA graph sees updates).
 */
#define VINE_MLP_PACKED_BYTES 102208
int vine_mlp_pack(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3,
                  const float* b3, const float* w_mu, const float* b_mu, const float* w_v, const float* b_v,
                  int num_obs, void* packed, void* stream);
int vine_mlp_forward(const void* packed, const float* obs, const float* obs_mean, const float* obs_inv_std,
                     int64_t n, int num_obs, const float* value_stats, float* mu, float* value,
                     void* stream);

/*
 * One rollout step of the policy in ONE launch (rl_games A2CAgent.get_action_values + the buffer writes of
 * play_steps; in-repo analogue learning/common_agent.py:257-314): vine_mlp_forward's network, then
 *   action = mu + exp(logstd) * N(0,1)   Philox4x32-10, key = seed, counter = (global env id, 16, *rng_counter, 0)
 *   neglogp = 0.5 sum(eps^2) + log(2 pi) + sum(logstd);   env_actions = clamp(action, +-1)  (preprocess_actions)
 * and a copy of the raw observation row.  Every output pointer is optional (NULL = skip); with actions == NULL
 * the call is pure inference (== vine_mlp_forward).  The Philox stream is keyed by the GLOBAL env id, so sampled
 * actions do not depend on how envs are sharded over GPUs.
 */
typedef struct VinePolicyAct {
  const void* packed;            /* VINE_MLP_PACKED_BYTES */
  const float* obs;              /* [n, O] */
  const float* obs_mean;         /* [O] */
  const float* obs_inv_std;      /* [O] */
  const float* value_stats;      /* {mean, std} */
  float* mu;                     /* [n, 2] */
  float* value;                  /* [n] de-normalised */
  const float* logstd;           /* [2]; required when sampling */
  const uint32_t* rng_counter;   /* device word, advanced by vine_rollout_post */
  float* actions;                /* [n, 2] raw sampled actions; NULL = no sampling */
  float* neglogp;                /* [n] */
  float* obs_copy;               /* [n, O] */
  float* env_actions;            /* [n, 2] clamped to [-1, 1] */
  int64_t n;
  int32_t num_obs, reserved;
  uint64_t seed;
  int64_t global_env_offset;
  void* u_out;                   /* NULL, or [ceil(n/128)] tiles [128 x 128] bf16 (UMMA row-blocked): the LSTM input
                                    [MLP output (64) | normalised obs (32, col 31 == 1) | 0]; heads and sampling are
                                    skipped (they follow the LSTM: vine_lstm_step / vine_lstm_head) */
} VinePolicyAct;
int vine_policy_act(const VinePolicyAct* args, void* stream);

/*
 * After the env step (rl_games play_steps tail): shaped = reward * reward_scale (YP:58-59)
 * [+ gamma * value on time-outs, value_bootstrap YP:56], dones, per-env episode return/length and the
 * device-side episode statistics ep_stats f64[4] += {episodes, successes, sum return, sum length}.
 * The whole rl_games DefaultRewardsShaper (without log_val): shaped = clamp((reward + reward_shift) * reward_scale,
 * reward_min, reward_max), the shift added only when it is non-zero (reward + 0 would turn -0 into +0) and the clamp applied
 * only with reward_clamp != 0; a NaN reward stays NaN, as with torch.clamp.
 */
typedef struct VineRolloutPost {
  const float* rewards;          /* env rew_buf [n] */
  const int64_t* resets;         /* env reset_buf [n] */
  const uint8_t* timeouts;       /* env timeout_buf [n] (bool) */
  const float* values;           /* [n] value estimates of this step */
  float* shaped_rewards;         /* [n] out */
  float* dones_next;             /* [n] out, 0/1 */
  float* ep_return;              /* [n] in/out */
  float* ep_length;              /* [n] in/out */
  double* ep_stats;              /* [4] accumulated */
  uint32_t* rng_counter;         /* incremented once per call (may be NULL) */
  int64_t n;
  float reward_scale, gamma;
  int32_t value_bootstrap;
  float success_reward_threshold;
  float* not_done_next;          /* NULL or [n] out: 1 - dones_next (the mask of the recurrent state) */
  float reward_shift;            /* reward_shaper.shift_value (0: none) */
  float reward_min, reward_max;  /* reward_shaper.min_val / max_val, used when reward_clamp != 0 */
  int32_t reward_clamp;
} VineRolloutPost;
int vine_rollout_post(const VineRolloutPost* args, void* stream);

/*
 * Update prologue (once per PPO iteration): rl_games RunningMeanStd updates of observations and values
 * (values and returns pooled), advantage mean/std, then values_n/returns_n = clamp((x - mean)/std, +-5) and
 * advantages_n = ((returns - values) - mean) / (std + 1e-8).  vine_ppo_moments accumulates f64 sufficient
 * statistics into `moments` (2*O + 4 doubles, zero on first use; all-reduce it across ranks and set `world`),
 * vine_ppo_finalize merges them into the running statistics (f64, in place), writes the f32 copies the
 * kernels read, normalises, and clears `moments`.
 */
typedef struct VinePpoPrologue {
  const float* obs;              /* [count, O] */
  const float* values;           /* [count] */
  const float* returns;          /* [count] */
  double* moments;               /* [2*O + 4] */
  double *obs_mean, *obs_var, *obs_count;     /* [O], [O], [1] */
  double *val_mean, *val_var, *val_count;     /* scalars */
  float *obs_mean_f, *obs_inv_std_f;          /* [O] out */
  float *value_stats, *adv_stats;             /* {mean, std}, {mean, 1/(std+1e-8)} out */
  float *values_n, *returns_n, *advantages_n; /* [count] out */
  int64_t count;
  int32_t num_obs, world, normalize_advantage, reserved;
} VinePpoPrologue;
int vine_ppo_moments(const VinePpoPrologue* args, void* stream);
int vine_ppo_finalize(const VinePpoPrologue* args, void* stream);

/*
 * The recurrent half of the reference's network (Vine5LinkMovingBasePPO.yaml:32-40: lstm 256, concat_input,
 * layer_norm; rl_games A2CBuilder.Network.forward) on hand-written kernels.  Activations live in HBM as 128-row
 * tiles in the UMMA row-blocked layout (one bulk-TMA copy per GEMM operand): u / hm / hh = [tiles][...] as described
 * in csrc/vine_lstm_net.cu; c = f32 [n, 256] row-major.
 *   vine_lstm_pack : torch-layout f32 parameters (W_ih [1024, 64+O], W_hh [1024, 256], b_ih, b_hh, LayerNorm gamma/beta,
 *                    W_mu [2,256], b_mu, W_v [1,256], b_v) -> the packed block (bf16 weight pieces + f32 vectors).
 *   vine_lstm_step : one time step: gates = u W_ih^T + hm W_hh^T + b (tcgen05, TMEM accumulator), c = f c_prev*nd + i g,
 *                    h = o tanh(c); writes c, hh (bf16 tiles), optionally hm_next = hh * not_done_next and the activated
 *                    gates (for backward).  Grid = (tiles, 8 slices of 32 hidden units).
 *   vine_lstm_mask : hm = hh * not_done (rollout: the done flag arrives after the step has run).
 *   vine_lstm_head : LayerNorm + mu/value heads per row (+ Philox Gaussian sampling, neglogp, clamped env action: the
 *                    same outputs and Philox keying as vine_policy_act).
 */
#define VINE_LSTM_PACKED_BYTES 795664
typedef struct VineLstmStep {
  const void* params;            /* VINE_LSTM_PACKED_BYTES */
  const void* u;                 /* [tiles][128 x 128] bf16 */
  const void* hm;                /* [tiles][2][128 x 128] bf16: not_done * h_prev */
  const float* c_prev;           /* [n, 256] */
  const float* not_done;         /* [n] mask of c_prev (NULL = 1) */
  const float* not_done_next;    /* [n] mask for hm_next (NULL = 1) */
  float* c;                      /* [n, 256] out */
  void* hh;                      /* [tiles][2][128 x 128] bf16 out */
  void* hm_next;                 /* NULL or like hh */
  void* act;                     /* NULL or [tiles][16][128 x 64] bf16 activated gates */
  int64_t n;
} VineLstmStep;
typedef struct VineLstmHead {
  const void* params;
  const void* hh;
  const float* value_stats;      /* {mean, std} */
  float* mu;                     /* [n, 2] or NULL */
  float* value;                  /* [n] de-normalised, or NULL */
  const float* logstd;           /* [2]; required when sampling */
  const uint32_t* rng_counter;
  float* actions;                /* [n, 2] or NULL (no sampling) */
  float* neglogp;                /* [n] */
  float* env_actions;            /* [n, 2] clamped */
  int64_t n;
  uint64_t seed;
  int64_t global_env_offset;
} VineLstmHead;
int vine_lstm_pack(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, const float* ln_gamma,
                   const float* ln_beta, const float* w_mu, const float* b_mu, const float* w_v, const float* b_v,
                   int num_obs, void* packed, void* stream);
int vine_lstm_step(const VineLstmStep* args, void* stream);
int vine_lstm_mask(const void* hh, const float* not_done, int64_t n, void* hm, void* stream);
int vine_lstm_head(const VineLstmHead* args, void* stream);

/*
 * Training counterpart of vine_lstm_head over all rows of a minibatch (rows = [step][sequence]): LayerNorm + heads,
 * the PPO losses of vine_ppo_minibatch (same formulas), and the backward down to dh (bf16 tiles like hh).
 * scalars f32 [n, 8] per row: action0, action1, mu_old0, mu_old1, neglogp_old, value_old (normalised), return
 * (normalised), advantage (normalised).  grads f32 [VINE_LSTM_HEAD_GRAD_PARTS + 1][VINE_LSTM_HEAD_GRAD_FLOATS] receives one
 * partial per thread block (the call returns how many; vine_lstm_reduce sums them): d(LayerNorm gamma)[256],
 * d(beta)[256], d(W_mu0, W_mu1, W_v)[3][256], d(b)[3] (+1 pad), d(logstd)[2], loss statistics a_loss, c_loss, kl,
 * b_loss (means), padding.
 */
#define VINE_LSTM_HEAD_GRAD_FLOATS 1296
#define VINE_LSTM_HEAD_GRAD_PARTS 1184  /* max per-block gradient partials one vine_lstm_head_train call writes */
typedef struct VineLstmHeadTrain {
  const void* params;
  const void* hh;                /* [tiles][2][128 x 128] bf16 */
  const float* scalars;          /* [n, 8] */
  const float* logstd;           /* [2] */
  const float* logstd_old;       /* [2] */
  void* dh;                      /* out, tiles like hh */
  float* grads;                  /* [VINE_LSTM_HEAD_GRAD_PARTS][VINE_LSTM_HEAD_GRAD_FLOATS] per-block partials */
  float* debug_out;              /* NULL or [n, 4]: mu0, mu1, normalised value, neglogp */
  int64_t n;
  float e_clip, critic_coef, entropy_coef, bounds_loss_coef, inv_B, reserved_f;
  /* rl_games dataset.update_mu_sigma: NULL, or the [T, N, 8] scalars buffer this minibatch was gathered from; the kernel
   * stores this pass's mu into columns 2,3 of the source row of every minibatch row (rows = [step in chunk][chunk][env]) */
  float* mu_writeback;
  int64_t wb_seq_len, wb_chunks, wb_num_envs, wb_env_begin, wb_env_count;
  int32_t value_loss_unclipped;  /* 0: clipped value loss (rl_games clip_value True); 1: c_loss = (return - v)^2 */
  int32_t reserved2;             /* 0 */
} VineLstmHeadTrain;
int vine_lstm_head_train(const VineLstmHeadTrain* args, void* stream);

/*
 * Backward through one LSTM time step of a minibatch (truncated BPTT, steps visited in reverse):
 *   vine_lstm_cell_bwd_tiles : pointwise; from the activated gates, c_prev, c, dh (from the head) [+ dh_rec from the
 *       following step, already masked] and dc_next -> dG (bf16 tiles like act) and dc_prev.
 *   vine_lstm_bwd_gemm : d[u(:, 0:64) | hm] = dG W (tcgen05; the 1024 gate rows streamed as 16 pieces through a 3-stage
 *       ring of bulk-TMA copies; the forward weight pieces are read as MN-major operands): dh3 f32 [n, 64] = gradient of
 *       the MLP output, dh_rec = not_done * d(hm) as bf16 tiles for the previous step (NULL at the first step).
 */
typedef struct VineLstmCellBwd {
  const void* act;               /* [tiles][16][128 x 64] bf16 */
  const float* c_prev;           /* [n, 256] */
  const float* c;                /* [n, 256] */
  const float* not_done;         /* [n] or NULL */
  const void* dh;                /* tiles like hh: dh from the head */
  const void* dh_rec;            /* tiles like hh or NULL */
  const float* dc_next;          /* [n, 256] or NULL */
  void* dg;                      /* out, tiles like act */
  float* dc_prev;                /* out [n, 256] */
  int64_t n;
} VineLstmCellBwd;
typedef struct VineLstmBwdGemm {
  const void* params;
  const void* dg;
  const float* not_done;         /* [n] mask applied to dh_rec (NULL = 1) */
  float* dh3;                    /* out [n, 64] */
  void* dh_rec;                  /* out tiles like hh, or NULL */
  int64_t n;
} VineLstmBwdGemm;
int vine_lstm_cell_bwd_tiles(const VineLstmCellBwd* args, void* stream);
int vine_lstm_bwd_gemm(const VineLstmBwdGemm* args, void* stream);

/*
 * Weight gradients and optimiser of the recurrent half.  Flat f32 parameter vector (torch layouts, this order):
 *   W_ih[1024, 64+O] W_hh[1024, 256] b_ih[1024] b_hh[1024] ln_gamma[256] ln_beta[256] W_mu[2,256] b_mu[2] W_v[1,256]
 *   b_v[1] logstd[2]                                   (vine_lstm_num_params(O) floats)
 *   vine_lstm_wgrad : dW^T = in^T dG over all (step, sequence) rows of the minibatch (tcgen05, both operands MN-major,
 *       rows streamed through a 2-stage bulk-TMA ring); grid = 12 output blocks x `splits` K ranges; partials go to
 *       workspace f32 [splits][12][128][256].  ntiles = number of 128-row tiles of u / hm / dg (all steps).
 *   vine_lstm_reduce : flat[p] = gradient of parameter p (sum of the partials; b_ih/b_hh from the constant-1 column
 *       of u; LayerNorm / heads / logstd from the head gradient buffer); flat[P..P+3] = a_loss, c_loss, kl, b_loss.
 *   vine_lstm_adam : torch.optim.Adam on the flat vector + in-place update of the packed block + the loss / KL
 *       bookkeeping in `state` (same layout and meaning as vine_ppo_adam, which then runs with bookkeeping = 0).
 */
/*
 * Minibatch assembly of the recurrent update in one launch: envs [env_begin, env_begin+env_count) x all horizon steps of
 * the [T, N] rollout buffers -> rows ordered [step in chunk][chunk, env] (T = chunks * seq_len; sequences = chunks *
 * env_count), plus the initial cell state and the masked initial hidden-state tiles of every sequence from the snapshots the
 * rollout took at the chunk starts.  num_envs, env_begin and env_count must be multiples of 128.
 */
typedef struct VineLstmGather {
  const float* obs;              /* [T, N, O] */
  const float* scalars;          /* [T, N, 8] */
  const float* not_done;         /* [T, N] */
  const float* c_saved;          /* [chunks, N, 256] */
  const void* hh_saved;          /* [chunks][N/128][2][128 x 128] bf16 */
  float* mb_obs;                 /* [L, S, O] out */
  float* mb_scalars;             /* [L, S, 8] out */
  float* mb_not_done;            /* [L, S] out */
  float* c0;                     /* [S, 256] out */
  void* hm0;                     /* [S/128][2][128 x 128] bf16 out: not_done[first step] * h */
  int32_t seq_len, chunks, num_envs, env_begin, env_count, num_obs;
} VineLstmGather;
int vine_lstm_gather(const VineLstmGather* args, void* stream);

typedef struct VineLstmWgrad {
  const void* u;                 /* [ntiles][128 x 128] bf16 */
  const void* hm;                /* [ntiles][2][128 x 128] bf16 */
  const void* dg;                /* [ntiles][16][128 x 64] bf16 */
  float* workspace;              /* [splits][12][128][256] f32 */
  int64_t ntiles;
  int32_t splits, reserved;
} VineLstmWgrad;
int vine_lstm_num_params(int num_obs);
int vine_lstm_wgrad(const VineLstmWgrad* args, void* stream);
/* head_grads: the partials of vine_lstm_head_train; its last row is scratch for their sum.  p2p_channel (NULL on one GPU):
 * see "gradient all-reduce over peer memory" below */
int vine_lstm_reduce(const float* workspace, int splits, float* head_grads, int head_parts, int num_obs, float* flat,
                     void* p2p_channel, void* stream);
int vine_lstm_adam(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed,
                   float* state, int num_obs, float beta1, float beta2, float eps, void* p2p_channel, void* stream);
/* the same with the gradient-clipping coefficient clip_coef (device, NULL = none), see vine_grad_clip */
int vine_lstm_adam_clipped(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq, void* packed,
                           float* state, int num_obs, float beta1, float beta2, float eps, const float* clip_coef,
                           void* p2p_channel, void* stream);

/*
 * Pointwise half of the LSTM layer of the reference's network (Vine5LinkMovingBasePPO.yaml:32-38; rl_games
 * LSTMWithDones, torch gate order i,f,g,o), one fused launch per time step and direction.  `gates` bf16 [S, 4H] are
 * the pre-activations (input projection + recurrent GEMM + biases); not_done [S] multiplies the incoming state
 * (hidden state zeroed where an episode ended before this observation).  Forward writes c, h (f32), the bf16
 * h * not_done_next that feeds the next recurrent GEMM, and the activated gates (bf16 [S, 4H]) for backward.
 * Backward takes dh_out (f32, from the layers above), the raw recurrent dh of step t+1 (bf16, = dG_{t+1} W_hh, masked
 * here with not_done_next) and dc_next, and writes dG (bf16 [S, 4H]) and dc_prev.  Optional pointers may be NULL.
 */
int vine_lstm_cell_fwd(const void* gates_bf16, const float* c_prev, const float* not_done, const float* not_done_next,
                       int64_t num_seqs, int hidden, float* c, float* h, void* h_next_bf16, void* acts_bf16, void* stream);
int vine_lstm_cell_bwd(const void* acts_bf16, const float* c_prev, const float* c, const float* not_done, const float* dh_out,
                       const void* dh_rec_bf16, const float* not_done_next, const float* dc_next, int64_t num_seqs, int hidden,
                       void* dgates_bf16, float* dc_prev, void* stream);

/*
 * PPO minibatch update of the same network as ONE fused tcgen05/TMEM kernel: forward, the PPO losses of
 * Vine5LinkMovingBasePPO.yaml:46-81 (e_clip actor loss, clipped -- with value_loss_unclipped plain -- value loss
 * x critic_coef / 2, bounds loss, entropy), backward and weight gradients (rl_games A2CAgent.calc_gradients + autograd; in-repo analogue
 * learning/common_agent.py:319-435, 482-517), then the gradient reduction and torch.optim.Adam.
 *
 * Parameters live in ONE flat f32 vector in torch layouts, in this order:
 *   W1[256,O] b1[256] W2[128,256] b2[128] W3[64,128] b3[64] Wmu[2,64] bmu[2] Wv[1,64] bv[1] logstd[2]
 * (vine_ppo_num_params(O) floats); `packed` is their tensor-core copy (vine_mlp_pack format), which
 * vine_ppo_adam rewrites in place, so vine_mlp_forward always sees the current policy.
 *
 * A minibatch is rl_games' env-major slice: envs [env_begin, env_begin+env_count) x all `horizon` steps of the
 * [T, N] rollout buffers.  values_old / returns are value-normalised, advantages are batch-normalised (both
 * done by the caller once per iteration), obs is raw and normalised inside like vine_mlp_forward.
 *
 * state (device, >= 16 floats): [0] learning rate, [1] Adam step count, [2] KL of the last minibatch,
 * [3] "KL pending" flag, [4..7] running sums of a_loss, c_loss, kl, b_loss, [8] minibatches summed,
 * [9] gradient-clipping coefficient and [10] gradient norm of the last vine_grad_clip call (untouched without clipping),
 * [11] training iteration (rl_games epoch_num: +1 by every launch with epoch_begin), [12] sum and [13] count of the
 * minibatch KLs of the current mini-epoch (schedule_standard).
 * The learning-rate schedule runs on the device between optimiser steps, in block 0 of vine_ppo_minibatch: no host
 * synchronisation anywhere, the whole update is CUDA-graph capturable.  One run of the rule (rl_games scheduler.update):
 *   adaptive_lr: lr /= 1.5 if kl > 2 kl_threshold, lr *= 1.5 if kl < kl_threshold / 2, clamped to [lr_min, lr_max];
 *   lr_linear:   lr = lr_min + (lr0 - lr_min) * max(0, max_epochs - epoch) / max_epochs (epoch = state[11]);
 *   neither:     lr unchanged.
 * When: schedule_standard = 0 (rl_games `legacy`): with the KL of every minibatch, before the next optimiser step;
 * schedule_standard = 1 (`standard`): once per mini-epoch with the mean KL of its minibatches, applied by the first launch of
 * the next mini-epoch (mini_epoch_begin).  A launch first applies what is pending, then counts epoch_begin.
 */
#define VINE_PPO_WS_FLOATS 49664   /* floats per CTA gradient partial */
typedef struct VinePpoMinibatch {
  const void* packed;            /* VINE_MLP_PACKED_BYTES */
  const float* obs;              /* [T, N, O] raw observations */
  const float* actions;          /* [T, N, 2] */
  float* mu_old;                 /* [T, N, 2] in: mean of the policy the row was last evaluated with (rollout, or the previous
                                    mini-epoch); out: this pass's mean (rl_games dataset.update_mu_sigma) */
  const float* neglogp_old;      /* [T, N] */
  const float* values_old;       /* [T, N] normalised */
  const float* returns;          /* [T, N] normalised */
  const float* advantages;       /* [T, N] normalised */
  const float* obs_mean;         /* [O] */
  const float* obs_inv_std;      /* [O] */
  const float* logstd;           /* [2] current (points into the flat parameter vector) */
  const float* logstd_old;       /* [2] log-std these rows were last evaluated with (see vine_ppo_reduce) */
  float* workspace;              /* [workspace_ctas][VINE_PPO_WS_FLOATS] gradient partials, 16-B aligned */
  float* state;                  /* device optimiser state, see above */
  float* debug_out;              /* NULL or [T*env_count, 4]: mu0, mu1, normalised value, neglogp per sample */
  int32_t horizon, num_envs, env_begin, env_count, num_obs, workspace_ctas, adaptive_lr;
  int32_t reserved;              /* 0; 2 selects two (instead of four) epilogue threads per row, an A/B switch for profiling */
  float e_clip, critic_coef, entropy_coef, bounds_loss_coef, kl_threshold, lr_min, lr_max, reserved_f;
  const float* dh3_ext;          /* NULL, or f32 [T*env_count, 64]: d(loss)/d(MLP output) supplied by the LSTM backward
                                    (vine_lstm_bwd_gemm); the heads and losses are skipped and the loss pointers may be
                                    NULL -- the kernel recomputes the MLP forward and back-propagates from there */
  int32_t lr_linear;             /* 1: linear schedule (adaptive_lr must be 0; max_epochs > 0) */
  int32_t schedule_standard;     /* 0: rl_games schedule_type legacy, 1: standard (see above) */
  int32_t epoch_begin;           /* 1: this launch opens a training iteration */
  int32_t mini_epoch_begin;      /* 1: this launch opens a mini-epoch */
  int32_t max_epochs;            /* lr_linear: the schedule's length in iterations */
  int32_t value_loss_unclipped;  /* 0: clipped value loss (rl_games clip_value True); 1: c_loss = (return - v)^2 */
  float lr0;                     /* lr_linear: the initial learning rate */
  float reserved_f2;             /* 0 */
} VinePpoMinibatch;

int vine_ppo_num_params(int num_obs);
int vine_ppo_max_ctas(void);     /* upper bound of gradient partials one vine_ppo_minibatch call writes */
/* returns the number of partials written (> 0) or a negative error */
int vine_ppo_minibatch(const VinePpoMinibatch* batch, void* stream);
/* flat[p] = sum of the partials in parameter order, flat[P..P+3] = a_loss, c_loss, kl, b_loss (means).
 * logstd_old_out (NULL or [2]) receives a copy of logstd (the parameter, [2]): the sigma half of rl_games'
 * dataset.update_mu_sigma -- this launch sits between the minibatch kernel (last reader) and Adam (writer). */
int vine_ppo_reduce(const float* workspace, int n_partials, int num_obs, float* flat, const float* logstd,
                    float* logstd_old_out, void* p2p_channel, void* stream);
/* Adam step with g = flat * grad_scale (1/world after an all-reduce); updates params, moments, packed, state */
/* bookkeeping != 0: also record the loss statistics / pending KL in `state` (0 when vine_lstm_adam does it) */
int vine_ppo_adam(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq,
                  void* packed, float* state, int num_obs, float beta1, float beta2, float eps, int bookkeeping,
                  void* p2p_channel, void* stream);
/* the same with g = flat * grad_scale * clip_coef[0]: clip_coef (device, NULL = no clipping) is the coefficient
 * vine_grad_clip writes to state + 9 */
int vine_ppo_adam_clipped(const float* flat, float grad_scale, float* params, float* exp_avg, float* exp_avg_sq,
                          void* packed, float* state, int num_obs, float beta1, float beta2, float eps, int bookkeeping,
                          const float* clip_coef, void* p2p_channel, void* stream);

/*
 * Gradient-norm clipping before Adam (rl_games truncate_grads / grad_norm: torch.nn.utils.clip_grad_norm_ over the model's
 * parameters).  One or two flat gradient vectors (flat2 = NULL, count2 = length2 = 0 for one); entries [0, count) of each
 * count towards the norm, all `length` floats (gradient + loss statistics) are carried: with the reference network, flat =
 * the MLP half with count = vine_ppo_num_params(O) - 197 (its unused head slots excluded), flat2 = the recurrent half with
 * count2 = vine_lstm_num_params(O); length = count of floats of each vector (P + 4).  With g = flat * grad_scale:
 *   state[10] = total = sqrt(sum g^2) (f32, fixed summation order: the same bits on every rank holding the same sum),
 *   state[9]  = min(max_norm / (total + 1e-6), 1) (NaN stays NaN),
 * which vine_ppo_adam_clipped / vine_lstm_adam_clipped multiply in (pass state + 9).  workspace: device,
 * VINE_GRAD_CLIP_WS_FLOATS floats, zeroed once before the first call (the kernel leaves it ready for the next one; one
 * workspace per stream).  Multi-GPU over peer memory, this call is the consumer of the channels (one per vector): it writes
 * the rank-order sum over the ranks into flat / flat2, and the Adam launches then run without a channel.
 */
#define VINE_GRAD_CLIP_WS_FLOATS 1024
int vine_grad_clip(float* flat, int count, int length, float* flat2, int count2, int length2, float grad_scale,
                   float max_norm, float* state, float* workspace, void* p2p_channel, void* p2p_channel2, void* stream);

/*
 * Gradient all-reduce over peer memory (multi-GPU PPO; replaces the per-minibatch all-reduce of the flattened gradients the
 * reference gets from rl_games / Horovod: learning/common_agent.py:125-126,219).  One process per GPU of ONE node:
 *   vine_p2p_alloc(count, &region, handle)   cudaMalloc of this rank's region (two buffers of `count` f32 + flags) and its
 *                                            64-byte CUDA IPC handle; the caller exchanges the handles (torch.distributed);
 *   vine_p2p_open(peer_handle, &region)      maps a peer's region (NVLink peer access);
 *   vine_p2p_channel_create(regions[world] in rank order (own region at [rank]), world, rank, count, &channel)
 * and the channel is passed to the producer (vine_ppo_reduce / vine_lstm_reduce: the rank's gradient sum goes into its own
 * region; `flat` may then be NULL) and to the consumer (vine_ppo_adam / vine_lstm_adam: waits until every rank has
 * published, adds the `world` buffers in rank order -- bit-identical sums, hence bit-identical parameters, on all ranks --
 * and applies Adam to the sum; grad_scale = 1 / world gives the mean).  One channel per (producer, consumer) pair; every
 * rank must issue the same launches.  No host synchronisation, CUDA-graph capturable; csrc/vine_p2p.cuh has the protocol.
 */
#define VINE_P2P_HANDLE_BYTES 64
#define VINE_P2P_MAX_WORLD 16
int vine_p2p_alloc(int64_t count, void** region, void* ipc_handle_out);
int vine_p2p_open(const void* ipc_handle, void** region);
int vine_p2p_close(void* region);      /* a region obtained from vine_p2p_open */
int vine_p2p_free(void* region);       /* a region obtained from vine_p2p_alloc */
int vine_p2p_channel_create(void* const* regions, int world, int rank, int64_t count, void** channel);
/* buf[i] <- sum over the ranks of buf[i] (f64, rank order) for a short vector, e.g. the running-statistics moments between
 * vine_ppo_moments and vine_ppo_finalize; one single-block launch; the channel needs count >= 2 n */
int vine_p2p_allreduce_f64(void* channel, double* buf, int n, void* stream);
int vine_p2p_channel_status(const void* channel, uint32_t* exchanges_done, uint32_t* timed_out);   /* synchronises */
/* mean ns per exchange seen by block 0 of the consumer kernel, then reset: out[0] = entry -> own flag stored at every peer,
 * out[1 + r] = entry -> rank r's flag seen here, out[17] = entry -> last block of the consumer done, out[18] = entry -> block 0's
 * sums ready; n_out >= 1 + VINE_P2P_MAX_WORLD (17) or 19.  Synchronises. */
int vine_p2p_channel_timing(void* channel, double* out, int n_out);
int vine_p2p_channel_destroy(void* channel);

/* sizeof of the argument structs of the PPO entry points, in declaration order (VinePolicyAct = 0, VineRolloutPost,
 * VinePpoPrologue, VinePpoMinibatch, VineLstmStep, VineLstmHead, VineLstmHeadTrain, VineLstmCellBwd, VineLstmBwdGemm,
 * VineLstmWgrad, VineLstmGather = 10): lets a foreign-function binding verify its mirror of the layouts. */
int vine_abi_struct_size(int which);

#ifdef __cplusplus
}
#endif
#endif /* VINE_B200_H_ */
