/*
 * vine_oracle.c — CPU ORACLE (test infrastructure; see vine_oracle.h for the rules).
 *
 * A plain-C restatement of the reference's per-control-step pipeline.  Abbreviations:
 *   V5 = /root/reference/isaacgymenvs/tasks/Vine5LinkMovingBase.py
 *   VT = /root/reference/isaacgymenvs/tasks/base/vec_task.py
 *   YT = /root/reference/isaacgymenvs/cfg/task/Vine5LinkMovingBase.yaml
 *   URDF = /root/reference/assets/urdf/Vine5LinkMovingBase.urdf
 * Task logic is IEEE f32 in the operation order torch's CPU kernels use (pinned by
 * tests/golden/).  Build with -ffp-contract=off: every fused multiply-add is explicit.
 */
#include "vine_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ------------------------------------------------------------------------------------------
 * Model constants (URDF; SURVEY Appendix B)
 * ---------------------------------------------------------------------------------------- */
#define NL 5
static const double LINK_LEN = 0.0885;       /* URDF:294-326 joint origins */
static const double LINK_COM = 0.04425;      /* URDF:83 inertial origin */
static const double LINK_MASS[NL] = {0.005, 0.005, 0.005, 0.005, 0.1};           /* URDF:84.. */
static const double LINK_INERTIA[NL] = {6.89246e-6, 6.89246e-6, 6.89246e-6, 6.89246e-6,
                                        1.01559e-4};                              /* ixx */
static const double CART_MASS = 0.4;         /* URDF:69 */
static const double BASE_ANGLE = 3.1415;     /* URDF:289 rpy of cart_to_link_0 (not exactly pi) */
static const double PIVOT_Z = 1.0 - 0.025 - 0.01; /* INIT_Z (V5:85) + joint origins URDF:275,289 */
static const double LINK_RADIUS = 0.0381;    /* URDF:98 */
static const double FPAM_RADIUS = 0.0169;    /* URDF:113 */
static const double FPAM_OFFSET = 0.055;     /* URDF:111 */
/* torque law tau = -(K q + C qd + b + B u), V5:1045-1048 */
static const float TL_K[NL] = {0.8385f, 1.5400f, 1.5109f, 1.2887f, 0.4347f};
static const float TL_C[NL] = {0.0178f, 0.0304f, 0.0528f, 0.0367f, 0.0223f};
static const float TL_b[NL] = {0.0007f, 0.0062f, 0.0402f, 0.0160f, 0.0133f};
static const float TL_B[NL] = {0.0247f, 0.0616f, 0.0779f, 0.0498f, 0.0268f};
/* pipe (V5:45,88,487; STL dims SURVEY App. B) */
static const double PIPE_RADIUS_PARAM = 0.07 * 1.05;
static const double PIPE_R_IN = 0.069 * 1.05, PIPE_R_OUT = 0.074 * 1.05, PIPE_LEN = 0.325 * 1.05;
static const double PIPE_MESH_CENTER = 0.074 * 1.05;

/* observation scaling rows, V5:246-266 */
static const float OBS_SCALE_28[28] = {0.12f, 0.269f, 0.148f, 0.249f, 0.148f, 0.344f,
                                       0.67f, 2.22f, 1.47f, 1.14f, 0.903f, 0.716f,
                                       0.0656f, 0.238f, 0.0656f, 0.732f, 2.0f, 0.732f,
                                       0.02f, 0.0235f, 0.02f, 0.732f, 2.0f, 0.732f,
                                       0.845f, 0.86f, 0.0385f, 0.5f};
static const float OBS_SCALE_18[18] = {0.12f, 0.67f, 0.0656f, 0.238f, 0.0656f, 0.732f, 2.0f,
                                       0.732f, 0.02f, 0.0235f, 0.02f, 0.732f, 2.0f, 0.732f,
                                       0.845f, 0.86f, 0.0385f, 0.5f};

enum { SITE_ACTION_NOISE = 1, SITE_DYNAMICS = 2, SITE_OBS_NOISE = 3, SITE_RESET = 4 };

int oracle_num_observations(int t) {
  switch (t) { /* V5:152-171 */
    case VINE_OBS_POS_ONLY: return 14;
    case VINE_OBS_POS_AND_VEL:
    case VINE_OBS_POS_AND_FD_VEL:
    case VINE_OBS_POS_AND_PREV_POS: return 26;
    case VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO: return 28;
    case VINE_OBS_TIP_AND_CART_AND_OBJ_INFO: return 18;
    default: return -1;
  }
}

void oracle_config_defaults(VineConfig* c) { /* YT:7-134 */
  memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(*c);
  c->substeps = 10; c->dt = 0.00833; c->gravity_z = -9.81;
  c->control_freq_inv = 4; c->max_episode_length = 500;
  c->clip_observations = 5.0; c->clip_actions = 1.0;
  c->observation_type = VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO; c->scale_observations = 1;
  c->create_shelf = 0; c->create_pipe = 1;
  c->use_smoothed_fpam = 1; c->force_u_fpam = 0; c->force_u_rail_velocity = 0;
  c->action_delay = 1;
  c->smoothing_alpha_inflate = 0.81; c->smoothing_alpha_deflate = 0.86;
  c->fpam_min = -0.1; c->fpam_max = 3.0; c->rail_velocity_scale = 1.0;
  c->damping = 2e-2; c->stiffness = 0.0;
  c->rail_soft_limit = 0.3; c->rail_p_gain = 10.0; c->rail_d_gain = 0.0;
  c->rail_acceleration = 8.0;
  c->randomize_dof_init = 1; c->randomize_targets = 1;
  c->random_init_cart_min_y = -0.1 * 0.3; c->random_init_cart_max_y = 0.3;
  c->success_dist = 0.08;
  c->min_target_depth_in_obstacle = -0.05; c->max_target_depth_in_obstacle = 0.2;
  c->min_target_y = -0.48; c->max_target_y = -0.4;
  c->min_target_z = 0.58; c->max_target_z = 0.67;
  {
    const double w[VINE_NUM_REWARDS] = {0, 0, 1, 0, 0.1, 0, 0, 0, 0, 1, 0, 0, 0.10};
    memcpy(c->reward_weights, w, sizeof(w));
  }
  c->use_target_reached_reset = 1; c->use_tip_limit_hit_reset = 0;
  c->use_nonzero_contact_force_reset = 0;
  c->vine_randomize = 1;
  c->dynamics_scaling_min = 0.999; c->dynamics_scaling_max = 1.001;
  c->observation_noise_std = 0.0; c->action_noise_std = 0.0;
  c->accel_target_scaling_min = 1.0; c->accel_target_scaling_max = 1.0;
  c->torque_law_integration = VINE_TORQUE_LAW_IMPLICIT;
  c->emulate_stale_body_state = 1;
  c->armature = 0.0;
  c->revolute_lower = -3.4e38; c->revolute_upper = 3.4e38;
  c->prismatic_lower = -3.4e38; c->prismatic_upper = 3.4e38;
  c->contact_stiffness = 2000.0; c->contact_damping = 2.0; c->contact_rest_offset = 0.001;
  c->contact_cull_slack = 0.01; c->contact_binning = 1;  /* launch tuning of the CUDA library: unused here */
}

/* ------------------------------------------------------------------------------------------
 * Philox4x32-10 (Salmon et al., SC'11).  ctr = (gid, site, step, block), key = seed.
 * ---------------------------------------------------------------------------------------- */
void oracle_philox(uint64_t seed, uint32_t gid, uint32_t site, uint32_t step, uint32_t block,
                   uint32_t out[4]) {
  uint32_t c0 = gid, c1 = site, c2 = step, c3 = block;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

static inline float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; } /* [0,1) */

void oracle_uniform4(uint64_t seed, uint32_t gid, uint32_t site, uint32_t step, uint32_t block,
                     float out[4]) {
  uint32_t r[4];
  oracle_philox(seed, gid, site, step, block, r);
  for (int i = 0; i < 4; ++i) out[i] = u01(r[i]);
}

/* The 24 uniforms of one sim step's dynamics draw (V5:1053-1055 needs 20, the accel scaling 1): 16 random bits each, two per
 * Philox word of blocks 8 i .. 8 i + 2, low half first. */
void oracle_dynamics_uniforms(uint64_t seed, uint32_t gid, uint32_t step, uint32_t sim_i, float out[24]) {
  for (uint32_t b = 0; b < 3; ++b) {
    uint32_t r[4];
    oracle_philox(seed, gid, SITE_DYNAMICS, step, sim_i * 8u + b, r);
    for (int w = 0; w < 4; ++w) {
      out[8 * b + 2 * w] = (float)(r[w] & 0xffffu) * 1.52587890625e-05f;      /* 2^-16: [0,1) */
      out[8 * b + 2 * w + 1] = (float)(r[w] >> 16) * 1.52587890625e-05f;
    }
  }
}

/* Box-Muller: 4 u32 -> 4 standard normals. */
void oracle_normal4(uint64_t seed, uint32_t gid, uint32_t site, uint32_t step, uint32_t block,
                    float out[4]) {
  uint32_t r[4];
  oracle_philox(seed, gid, site, step, block, r);
  for (int p = 0; p < 2; ++p) {
    float u1 = (float)((r[2 * p] >> 8) + 1u) * 5.9604644775390625e-08f; /* (0,1] */
    float u2 = u01(r[2 * p + 1]);
    float rad = sqrtf(-2.0f * logf(u1));
    float ang = 6.283185307179586f * u2;
    out[2 * p] = rad * cosf(ang);
    out[2 * p + 1] = rad * sinf(ang);
  }
}

static inline float uniform_ab(float u, float a, float b) { return fmaf(u, b - a, a); }

/* ------------------------------------------------------------------------------------------
 * Derived f32 constants: where a Python float meets an f32 tensor in the reference it is
 * rounded to f32 at that point; arithmetic between Python floats happens in double first.
 * ---------------------------------------------------------------------------------------- */
typedef struct Derived {
  int O, C, S, D;
  float clip_act, clip_obs;
  float act_noise, obs_noise;
  float rail_scale, fpam_range, fpam_min;       /* V5:1458-1463 */
  float alpha_inf, alpha_def;                   /* V5:1001-1002 */
  float dt, control_dt;                         /* V5:227-228 */
  float rail_force_max, rail_accel, p_gain, d_gain; /* V5:1074-1091 */
  float dyn_min, dyn_max, acc_min, acc_max;
  float soft_limit, success_dist;
  float w[VINE_NUM_REWARDS];
  float rev_lo, rev_hi, cart_lo, cart_hi;       /* V5:778-786 */
  float ty_lo, ty_hi, tz_lo, tz_hi, dep_lo, dep_hi;
  const float* obs_scale;                       /* NULL = ones */
} Derived;

static int derive(const VineConfig* c, Derived* d) {
  if (c->struct_size != (int32_t)sizeof(VineConfig)) return VINE_ERR_ABI_MISMATCH;
  memset(d, 0, sizeof(*d));
  d->O = oracle_num_observations(c->observation_type);
  if (d->O < 0) return VINE_ERR_INVALID_ARG;
  d->C = c->control_freq_inv; d->S = c->substeps; d->D = c->action_delay;
  if (d->C < 1 || d->S < 1 || d->D < 0 || d->D > VINE_MAX_ACTION_DELAY) return VINE_ERR_INVALID_ARG;
  d->obs_scale = NULL;
  if (c->scale_observations) { /* V5:242-268 */
    if (c->observation_type == VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO) d->obs_scale = OBS_SCALE_28;
    else if (c->observation_type == VINE_OBS_TIP_AND_CART_AND_OBJ_INFO) d->obs_scale = OBS_SCALE_18;
    else return VINE_ERR_UNSUPPORTED;
  }
  d->clip_act = (float)c->clip_actions; d->clip_obs = (float)c->clip_observations;
  d->act_noise = (float)c->action_noise_std; d->obs_noise = (float)c->observation_noise_std;
  d->rail_scale = (float)c->rail_velocity_scale;
  d->fpam_range = (float)(c->fpam_max - c->fpam_min); d->fpam_min = (float)c->fpam_min;
  d->alpha_inf = (float)c->smoothing_alpha_inflate; d->alpha_def = (float)c->smoothing_alpha_deflate;
  d->dt = (float)c->dt; d->control_dt = (float)(c->dt * (double)c->control_freq_inv);
  d->rail_force_max = (float)(c->rail_acceleration / 2.0); d->rail_accel = (float)c->rail_acceleration;
  d->p_gain = (float)c->rail_p_gain; d->d_gain = (float)c->rail_d_gain;
  d->dyn_min = (float)c->dynamics_scaling_min; d->dyn_max = (float)c->dynamics_scaling_max;
  d->acc_min = (float)c->accel_target_scaling_min; d->acc_max = (float)c->accel_target_scaling_max;
  d->soft_limit = (float)c->rail_soft_limit; d->success_dist = (float)c->success_dist;
  for (int i = 0; i < VINE_NUM_REWARDS; ++i) d->w[i] = (float)c->reward_weights[i];
  {
    const double ten = 10.0 * 3.14159265358979323846 / 180.0; /* math.radians(10) */
    d->rev_lo = (float)fmax(c->revolute_lower, -ten);
    d->rev_hi = (float)fmin(c->revolute_upper, ten);
    d->cart_lo = (float)fmax(c->prismatic_lower, c->random_init_cart_min_y);
    d->cart_hi = (float)fmin(c->prismatic_upper, c->random_init_cart_max_y);
  }
  d->ty_lo = (float)c->min_target_y; d->ty_hi = (float)c->max_target_y;
  d->tz_lo = (float)c->min_target_z; d->tz_hi = (float)c->max_target_z;
  d->dep_lo = (float)c->min_target_depth_in_obstacle; d->dep_hi = (float)c->max_target_depth_in_obstacle;
  return VINE_OK;
}

/* ------------------------------------------------------------------------------------------
 * Action path — pre_physics_step V5:927-940, raw_actions_to_actions V5:984-997,
 * rescale_to_u V5:1458-1459, u_fpam_to_smoothed_u_fpam V5:999-1005, manual_intervention V5:1023-1026
 * ---------------------------------------------------------------------------------------- */
static inline void pre_physics_env(const VineConfig* c, const Derived* d, float a0, float a1,
                                   const float noise[2], float* hist /* [D,2] oldest first */,
                                   float* smoothed, float* u_rail_out, float* u_fpam_out) {
  if (c->vine_randomize && noise) { /* V5:930-932 */
    a0 = a0 + d->act_noise * noise[0];
    a1 = a1 + d->act_noise * noise[1];
  }
  float new_rail = a0 * d->rail_scale;
  float new_fpam = ((a1 + 1.0f) / 2.0f) * d->fpam_range + d->fpam_min;
  float u_rail, u_fpam;
  if (d->D == 0) { /* append then pop(0) on an empty list returns the new element */
    u_rail = new_rail; u_fpam = new_fpam;
  } else {         /* V5:936-937 */
    u_rail = hist[0]; u_fpam = hist[1];
    for (int k = 0; k + 1 < d->D; ++k) { hist[2 * k] = hist[2 * k + 2]; hist[2 * k + 1] = hist[2 * k + 3]; }
    hist[2 * (d->D - 1)] = new_rail; hist[2 * (d->D - 1) + 1] = new_fpam;
  }
  if (c->force_u_fpam) u_fpam = 0.0f;
  if (c->force_u_rail_velocity) u_rail = 0.0f;
  float s = *smoothed;
  float alpha = (u_fpam > s) ? d->alpha_inf : d->alpha_def;
  *smoothed = alpha * s + (1.0f - alpha) * u_fpam;
  *u_rail_out = u_rail; *u_fpam_out = u_fpam;
}

/* ------------------------------------------------------------------------------------------
 * compute_and_set_dof_actuation_force_tensor, V5:1028-1106
 * scale: [5][4] multipliers of (K,C,b,B) (V5:1053-1055) or NULL; acc_scale multiplies accel_target.
 * ---------------------------------------------------------------------------------------- */
static inline void actuation_env(const Derived* d, const float q[6], const float qd[6],
                                 float cart_vel_y, float u_rail, float u_use,
                                 const float* scale, float acc_scale,
                                 float* prev_cart_vel, float* prev_err, float efforts[6]) {
  for (int j = 0; j < NL; ++j) {
    float sK = scale ? scale[4 * j + 0] : 1.0f, sC = scale ? scale[4 * j + 1] : 1.0f;
    float sb = scale ? scale[4 * j + 2] : 1.0f, sB = scale ? scale[4 * j + 3] : 1.0f;
    float t = (TL_K[j] * sK) * q[j + 1];
    t = t + (TL_C[j] * sC) * qd[j + 1];
    t = t + (TL_b[j] * sb);
    t = t + (TL_B[j] * sB) * u_use;
    efforts[j + 1] = -t;
  }
  float err = u_rail - cart_vel_y;
  float minmax = (err > 0.0f) ? d->rail_force_max : -d->rail_force_max;
  float accel = (cart_vel_y - *prev_cart_vel) / d->dt;
  float accel_target = (err > 0.0f) ? d->rail_accel : -d->rail_accel;
  accel_target = accel_target * acc_scale;           /* ACCEL_TARGET_SCALING (README.md:63); 1.0 = no-op */
  float adjustment = 0.30f * (accel_target - accel); /* COURSE_P_GAIN V5:1083 */
  minmax = minmax + adjustment;
  float pid = d->p_gain * err + d->d_gain * (err - *prev_err);
  efforts[0] = (fabsf(err) > 0.1f) ? minmax : pid;   /* V5:1094 */
  *prev_err = err; *prev_cart_vel = cart_vel_y;
}

/* ------------------------------------------------------------------------------------------
 * Obstacles as 2-D rectangles in the (y,z) plane of motion.
 * ---------------------------------------------------------------------------------------- */
typedef struct Rect { double cy, cz, ay, az, ha, hn; int sensing; } Rect; /* axis a (unit), normal n=(-az,ay) */

static int build_rects(const VineConfig* c, const float target[3], const float obj[2], Rect r[5]) {
  int n = 0;
  if (c->create_shelf) { /* custom_shelf.urdf:82-93,139-152; pose V5:818-829 */
    double ry = (double)target[1] + (-0.2 + (double)obj[0]), rz = (double)target[2] - 0.01;
    r[n++] = (Rect){ry - 0.001, rz, 1, 0, 0.1995, 0.005, 0};
    r[n++] = (Rect){ry, rz + 0.2, 1, 0, 0.2, 0.005, 0};
    r[n++] = (Rect){ry + 0.199, rz, 1, 0, 0.001, 0.005, 1};
  }
  if (c->create_pipe) { /* V5:841-885; mesh dims SURVEY App. B */
    double th = (double)obj[1], d = (double)obj[0];
    double ct = cos(th), st = sin(th);
    double off = PIPE_RADIUS_PARAM - PIPE_MESH_CENTER;
    double ey = (double)target[1] + d * ct + off * st, ez = (double)target[2] + d * st - off * ct;
    double ay = -ct, az = -st, ny = -az, nz = ay;
    double dx = -PIPE_RADIUS_PARAM + PIPE_MESH_CENTER; /* axis offset from the plane x=0 */
    double win = sqrt(PIPE_R_IN * PIPE_R_IN - dx * dx), wout = sqrt(PIPE_R_OUT * PIPE_R_OUT - dx * dx);
    double mid = 0.5 * (win + wout), hn = 0.5 * (wout - win), ha = 0.5 * PIPE_LEN;
    for (int s = -1; s <= 1; s += 2)
      r[n++] = (Rect){ey + ay * ha + s * mid * ny, ez + az * ha + s * mid * nz, ay, az, ha, hn, 0};
  }
  return n;
}

/* instantiate the dynamics for double and float */
#define REAL double
#define SUF(x) x##_f64
#include "vine_oracle_dyn.inc"
#undef REAL
#undef SUF
#define REAL float
#define SUF(x) x##_f32
#include "vine_oracle_dyn.inc"
#undef REAL
#undef SUF

typedef struct BodyState { float tip[3], tipvel[3], cart_y, cart_vy, lip; } BodyState;

static inline void simulate_env(const VineConfig* c, int use_f64, float q[6], float qd[6],
                                const float efforts[6], const float* scale, float u_use,
                                const float target[3], const float obj[2], BodyState* b) {
  if (use_f64) simulate_env_f64(c, q, qd, efforts, scale, u_use, target, obj, b->tip, b->tipvel, &b->lip);
  else simulate_env_f32(c, q, qd, efforts, scale, u_use, target, obj, b->tip, b->tipvel, &b->lip);
  b->cart_y = q[0]; b->cart_vy = qd[0];
}

/* ------------------------------------------------------------------------------------------
 * compute_observations V5:1339-1390, compute_reward V5:1218-1248 + compute_reward_jit
 * V5:1470-1537, compute_reset_jit V5:1540-1558, timeout VT:366
 * ---------------------------------------------------------------------------------------- */
static inline float norm3(float x, float y, float z) { /* torch CPU linalg.norm: nested fma */
  return sqrtf(fmaf(z, z, fmaf(y, y, x * x)));
}

typedef struct PostIn {
  const float *q, *qd, *prev_q, *tip, *prev_tip, *tipvel, *target, *target_vel, *obj;
  float cart_y, smoothed, u_fpam, u_rail, prev_u_rail;
  const float* contact; int contact_stride; /* contact[i*stride], i<C, or NULL */
  const float* obs_noise;                    /* [O] or NULL */
  int64_t reset_in, progress;
} PostIn;

static inline void post_physics_env(const VineConfig* c, const Derived* d, const PostIn* in,
                                    float* obs, float* rew, float* rmat /* [13] or NULL */,
                                    int64_t* reset_out, uint8_t* timeout) {
  float fdq[6], fdt[3], raw[28];
  for (int i = 0; i < 6; ++i) fdq[i] = (in->q[i] - in->prev_q[i]) / d->control_dt;      /* V5:1347 */
  for (int i = 0; i < 3; ++i) fdt[i] = (in->tip[i] - in->prev_tip[i]) / d->control_dt;  /* V5:1348 */
  int k = 0;
  const int t = c->observation_type;
  if (t == VINE_OBS_TIP_AND_CART_AND_OBJ_INFO) { /* V5:1375-1378 */
    raw[k++] = in->q[0]; raw[k++] = fdq[0];
  } else {
    for (int i = 0; i < 6; ++i) raw[k++] = in->q[i];
    if (t == VINE_OBS_POS_AND_VEL) for (int i = 0; i < 6; ++i) raw[k++] = in->qd[i];
    else if (t == VINE_OBS_POS_AND_PREV_POS) for (int i = 0; i < 6; ++i) raw[k++] = in->prev_q[i];
    else if (t != VINE_OBS_POS_ONLY) for (int i = 0; i < 6; ++i) raw[k++] = fdq[i];
  }
  for (int i = 0; i < 3; ++i) raw[k++] = in->tip[i];
  if (t == VINE_OBS_POS_AND_VEL) for (int i = 0; i < 3; ++i) raw[k++] = in->tipvel[i];
  else if (t == VINE_OBS_POS_AND_PREV_POS) for (int i = 0; i < 3; ++i) raw[k++] = in->prev_tip[i];
  else if (t != VINE_OBS_POS_ONLY) for (int i = 0; i < 3; ++i) raw[k++] = fdt[i];
  for (int i = 0; i < 3; ++i) raw[k++] = in->target[i];
  if (t != VINE_OBS_POS_ONLY) for (int i = 0; i < 3; ++i) raw[k++] = in->target_vel[i];
  raw[k++] = in->smoothed; raw[k++] = in->prev_u_rail;
  if (t == VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO || t == VINE_OBS_TIP_AND_CART_AND_OBJ_INFO) {
    raw[k++] = in->obj[0]; raw[k++] = in->obj[1];
  }
  for (int i = 0; i < d->O; ++i) {
    float v = raw[i] / (d->obs_scale ? d->obs_scale[i] : 1.0f);                 /* V5:1385 */
    if (c->vine_randomize && in->obs_noise) v = v + d->obs_noise * in->obs_noise[i]; /* V5:1388-1390 */
    obs[i] = v;
  }
  /* reward */
  float dist = norm3(in->tip[0] - in->target[0], in->tip[1] - in->target[1], in->tip[2] - in->target[2]);
  int reached = dist < d->success_dist;                                         /* V5:1228 */
  int limit_hit = (in->cart_y > d->soft_limit) || (in->cart_y < -d->soft_limit); /* V5:1232-1233 */
  int tip_limit_hit = in->tip[1] < in->target[1];                               /* V5:1237 */
  float contact = 0.0f; int nonzero = 0;
  if (c->create_shelf && in->contact) {                                         /* V5:1240-1244 */
    float s = in->contact[0];
    for (int i = 1; i < d->C; ++i) s = s + in->contact[i * in->contact_stride];
    contact = s / (float)d->C;
    nonzero = contact > 0.0f;
  }
  float r[VINE_NUM_REWARDS];
  r[0] = 0.0f - dist;
  r[1] = -1.0f;
  r[2] = reached ? 1000.0f : 0.0f;
  {
    float vs = norm3(in->tipvel[0] - in->target_vel[0], in->tipvel[1] - in->target_vel[1],
                     in->tipvel[2] - in->target_vel[2]);
    r[3] = 0.0f - (reached ? vs : 0.0f);
  }
  r[4] = norm3(in->tipvel[0], in->tipvel[1], in->tipvel[2]);
  r[5] = 0.0f - fabsf(in->u_rail);
  r[6] = 0.0f - fabsf(in->u_fpam);
  r[7] = 0.0f - fabsf(in->u_rail - in->prev_u_rail);
  r[8] = 0.0f - fabsf(in->u_fpam - in->smoothed);
  r[9] = limit_hit ? -100.0f : 0.0f;
  r[10] = 0.0f - fabsf(in->cart_y);
  r[11] = tip_limit_hit ? -100.0f : 0.0f;
  r[12] = 0.0f - ((contact > 0.0f) ? contact : 0.0f);
  float wr[VINE_NUM_REWARDS];
  for (int i = 0; i < VINE_NUM_REWARDS; ++i) wr[i] = r[i] * d->w[i];
  /* torch.sum(dim=-1) over 13 contiguous f32 on CPU: tail 8..12 first, then the 8 vector lanes */
  float acc = 0.0f;
  for (int i = 8; i < 13; ++i) acc = acc + wr[i];
  for (int i = 0; i < 8; ++i) acc = acc + wr[i];
  *rew = acc;
  if (rmat) memcpy(rmat, r, sizeof(r));
  /* compute_reset_jit */
  int64_t reset = (in->progress >= (int64_t)c->max_episode_length - 1) ? 1 : in->reset_in;
  if (reached && c->use_target_reached_reset) reset = 1;
  if (tip_limit_hit && c->use_tip_limit_hit_reset) reset = 1;
  if (limit_hit) reset = 1;
  if (nonzero && c->use_nonzero_contact_force_reset) reset = 1;
  *reset_out = reset;
  *timeout = (uint8_t)((in->progress >= (int64_t)c->max_episode_length - 1) && (reset != 0));
}

/* ------------------------------------------------------------------------------------------
 * reset_idx V5:774-885 (+ sample_target_positions V5:887-914).  Draw k of the reference's
 * call order maps to Philox block k/4, lane k%4: joints 1..5, cart, target x,y,z, depth.
 * ---------------------------------------------------------------------------------------- */
typedef struct ResetDraws { float u[12]; } ResetDraws;

static inline void reset_draws(uint64_t seed, uint32_t gid, uint32_t step, ResetDraws* r) {
  for (uint32_t b = 0; b < 3; ++b) oracle_uniform4(seed, gid, SITE_RESET, step, b, &r->u[4 * b]);
}

static inline void reset_env(const VineConfig* c, const Derived* d, const ResetDraws* r,
                             float q[6], float qd[6], float target[3], float obj[2]) {
  if (c->randomize_dof_init) {
    for (int j = 0; j < NL; ++j) q[j + 1] = uniform_ab(r->u[j], d->rev_lo, d->rev_hi);
    q[0] = uniform_ab(r->u[5], d->cart_lo, d->cart_hi);
  } else {
    for (int j = 0; j < 6; ++j) q[j] = 0.0f;
  }
  for (int j = 0; j < 6; ++j) qd[j] = 0.0f;
  if (c->randomize_targets) { /* V5:901-909 */
    target[0] = uniform_ab(r->u[6], 0.0f, 0.0f);
    target[1] = uniform_ab(r->u[7], d->ty_lo, d->ty_hi);
    target[2] = uniform_ab(r->u[8], d->tz_lo, d->tz_hi);
  } else {                    /* V5:911-912 */
    target[0] = 0.0f; target[1] = d->ty_hi; target[2] = d->tz_lo;
  }
  if (c->create_shelf) obj[0] = uniform_ab(r->u[9], d->dep_lo, d->dep_hi); /* V5:822-839 */
  if (c->create_pipe) {       /* V5:854-885 */
    float ez = 1.0f - target[2];
    /* np.polyval (Horner) with float64 coefficients on the f32 effective_z, then f32 */
    double x = (double)ez, y = 0.0;
    const double p[4] = {1.0e4 * 1.3199, 1.0e4 * -1.2276, 1.0e4 * 0.4045, 1.0e4 * -0.0447};
    for (int i = 0; i < 4; ++i) y = y * x + p[i];
    float theta_prime = (float)y * (float)(3.14159265358979323846 / 180.0); /* torch.deg2rad */
    obj[0] = uniform_ab(r->u[9 + (c->create_shelf ? 1 : 0)], d->dep_lo, d->dep_hi); /* V5:863: one more draw */
    obj[1] = theta_prime;
  }
}

/* forward kinematics of the tip in f32-rounded output (used on reset when not emulating staleness) */
static void fk_tip(const float q[6], float tip[3]) {
  double phi = BASE_ANGLE, y = q[0], z = PIVOT_Z;
  for (int k = 0; k < NL; ++k) { phi += (double)q[k + 1]; y += LINK_LEN * -sin(phi); z += LINK_LEN * cos(phi); }
  tip[0] = 0.0f; tip[1] = (float)y; tip[2] = (float)z;
}

/* ------------------------------------------------------------------------------------------
 * Whole control step: VecTask.step VT:319-380 with V5's hooks.
 * ---------------------------------------------------------------------------------------- */
static void step_env(const VineConfig* c, const Derived* d, OracleArrays* A, int64_t e, int use_f64) {
  const int O = d->O, C = d->C, D = d->D;
  const uint32_t gid = (uint32_t)(A->global_env_offset + e);
  const uint32_t step = (uint32_t)A->step_count[e];
  float* q = A->dof_pos + 6 * e; float* qd = A->dof_vel + 6 * e;
  float* target = A->target + 3 * e; float* obj = A->object_info + 2 * e;
  BodyState body;
  memcpy(body.tip, A->tip_body + 3 * e, 12); memcpy(body.tipvel, A->tipvel_body + 3 * e, 12);
  body.cart_y = A->cart_body_y[e]; body.cart_vy = A->cart_body_vy[e]; body.lip = A->lip_force[e];

  /* VT:333 */
  float a0 = fminf(fmaxf(A->actions[2 * e], -d->clip_act), d->clip_act);
  float a1 = fminf(fmaxf(A->actions[2 * e + 1], -d->clip_act), d->clip_act);
  /* pre_physics_step */
  float noise[4]; const float* np_ = NULL;
  if (c->vine_randomize && d->act_noise != 0.0f) { oracle_normal4(A->seed, gid, SITE_ACTION_NOISE, step, 0, noise); np_ = noise; }
  float u_rail, u_fpam;
  pre_physics_env(c, d, a0, a1, np_, A->history + (size_t)2 * D * e, &A->smoothed[e], &u_rail, &u_fpam);
  const float smoothed = A->smoothed[e];
  float prev_q[6]; memcpy(prev_q, q, sizeof(prev_q));           /* V5:943 */
  float prev_tip[3]; memcpy(prev_tip, body.tip, sizeof(prev_tip)); /* V5:944 (tensor as of last refresh) */
  float prev_u_rail = u_rail;                                   /* V5:945 */
  const float u_use = c->use_smoothed_fpam ? smoothed : u_fpam; /* V5:1059 */

  float contact[16]; float tip_before_last[3]; float rail_force = 0.0f;
  for (int i = 0; i < C; ++i) { /* VT:338-356 */
    /* refresh_state_tensors: rigid-body views = state after the previous simulate */
    memcpy(tip_before_last, body.tip, 12);
    float scale[20]; const float* sp = NULL; float acc_scale = 1.0f;
    if (c->vine_randomize) { /* V5:1053-1055: redrawn every sim step */
      float u[24];
      oracle_dynamics_uniforms(A->seed, gid, step, (uint32_t)i, u);
      for (int k = 0; k < 20; ++k) scale[k] = uniform_ab(u[k], d->dyn_min, d->dyn_max);
      acc_scale = uniform_ab(u[20], d->acc_min, d->acc_max);
      sp = scale;
    }
    float efforts[6];
    actuation_env(d, q, qd, body.cart_vy, u_rail, u_use, sp, acc_scale, &A->prev_cart_vel[e],
                  &A->prev_cart_vel_error[e], efforts);
    rail_force = efforts[0];
    if (i < 16) contact[i] = body.lip;                         /* VT:348-351 */
    simulate_env(c, use_f64, q, qd, efforts, sp, u_use, target, obj, &body); /* VT:356 */
  }

  /* post_physics_step V5:1110-1120 */
  int64_t progress = A->progress[e] + 1;
  int64_t reset_in = A->reset[e];
  float rew_dummy;
  if (reset_in != 0) {
    ResetDraws rd; reset_draws(A->seed, gid, step, &rd);
    reset_env(c, d, &rd, q, qd, target, obj);
    memcpy(prev_q, q, sizeof(prev_q));                          /* V5:794 */
    if (c->emulate_stale_body_state) {
      memcpy(prev_tip, tip_before_last, 12);                    /* V5:797: tensor last refreshed before the final simulate */
    } else {
      fk_tip(q, body.tip); memset(body.tipvel, 0, 12);
      body.cart_y = q[0]; body.cart_vy = 0.0f; body.lip = 0.0f;
      memcpy(prev_tip, body.tip, 12);
      A->prev_cart_vel[e] = 0.0f;
      for (int i = 0; i < C && i < 16; ++i) contact[i] = 0.0f;
    }
    prev_u_rail = 0.0f;                                         /* V5:798 */
    A->prev_cart_vel_error[e] = 0.0f;                           /* V5:799 */
    reset_in = 0; progress = 0; A->agg_rew[e] = 0.0f;           /* V5:807-810 */
  }
  (void)rew_dummy;
  float tvel[3] = {0.0f, 0.0f, 0.0f};                           /* V5:916-918 */
  float obs_noise[32]; const float* on = NULL;
  if (c->vine_randomize && d->obs_noise != 0.0f) {
    for (uint32_t b = 0; b < (uint32_t)((O + 3) / 4); ++b) oracle_normal4(A->seed, gid, SITE_OBS_NOISE, step, b, &obs_noise[4 * b]);
    on = obs_noise;
  }
  PostIn in = {q, qd, prev_q, body.tip, prev_tip, body.tipvel, target, tvel, obj,
               body.cart_y, smoothed, u_fpam, u_rail, prev_u_rail, contact, 1, on, reset_in, progress};
  float rmat[VINE_NUM_REWARDS];
  post_physics_env(c, d, &in, A->obs + (size_t)O * e, &A->rew[e], rmat, &A->reset[e], &A->timeout[e]);
  A->agg_rew[e] = A->agg_rew[e] + A->rew[e];                    /* V5:1278 */
  A->progress[e] = progress;
  if (A->obs_clamped)                                           /* VT:374 */
    for (int i = 0; i < O; ++i) A->obs_clamped[(size_t)O * e + i] = fminf(fmaxf(A->obs[(size_t)O * e + i], -d->clip_obs), d->clip_obs);
  memcpy(A->tip_body + 3 * e, body.tip, 12); memcpy(A->tipvel_body + 3 * e, body.tipvel, 12);
  A->cart_body_y[e] = body.cart_y; A->cart_body_vy[e] = body.cart_vy; A->lip_force[e] = body.lip;
  A->step_count[e] += 1;
  if (A->u_rail) A->u_rail[e] = u_rail;
  if (A->u_fpam) A->u_fpam[e] = u_fpam;
  if (A->prev_u_rail) A->prev_u_rail[e] = prev_u_rail;
  if (A->rail_force) A->rail_force[e] = rail_force;
  if (A->reward_matrix) memcpy(A->reward_matrix + VINE_NUM_REWARDS * e, rmat, sizeof(rmat));
}

int oracle_step(const VineConfig* cfg, OracleArrays* a, int use_f64, int nthreads) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  if (d.C > 16) return VINE_ERR_INVALID_ARG;
#ifdef _OPENMP
  int nt = nthreads > 0 ? nthreads : omp_get_max_threads();
#pragma omp parallel for schedule(static) num_threads(nt)
#endif
  for (int64_t e = 0; e < a->n; ++e) step_env(cfg, &d, a, e, use_f64);
  (void)nthreads;
  return VINE_OK;
}

/* State right after Vine5LinkMovingBase.__init__ (V5:178-291) + allocate_buffers (VT:260-283):
 * q = qd = 0, rigid-body views at the q = 0 pose, reset_buf = 1, targets sampled (V5:179) from
 * Philox (site RESET, step 0x40000000, draws 6..8). */
int oracle_init(const VineConfig* cfg, OracleArrays* a) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  for (int64_t e = 0; e < a->n; ++e) {
    float q0[6] = {0, 0, 0, 0, 0, 0};
    memset(a->dof_pos + 6 * e, 0, 24); memset(a->dof_vel + 6 * e, 0, 24);
    fk_tip(q0, a->tip_body + 3 * e); memset(a->tipvel_body + 3 * e, 0, 12);
    a->cart_body_y[e] = 0; a->cart_body_vy[e] = 0; a->lip_force[e] = 0;
    a->smoothed[e] = 0; a->prev_cart_vel[e] = 0; a->prev_cart_vel_error[e] = 0; a->agg_rew[e] = 0;
    a->object_info[2 * e] = 0; a->object_info[2 * e + 1] = 0;
    for (int k = 0; k < 2 * d.D; ++k) a->history[(size_t)2 * d.D * e + k] = 0;
    a->step_count[e] = 0; a->reset[e] = 1; a->progress[e] = 0; a->timeout[e] = 0; a->rew[e] = 0;
    for (int k = 0; k < d.O; ++k) a->obs[(size_t)d.O * e + k] = 0;
    ResetDraws rd; reset_draws(a->seed, (uint32_t)(a->global_env_offset + e), 0x40000000u, &rd);
    float* t = a->target + 3 * e;
    if (cfg->randomize_targets) {
      t[0] = uniform_ab(rd.u[6], 0.0f, 0.0f); t[1] = uniform_ab(rd.u[7], d.ty_lo, d.ty_hi);
      t[2] = uniform_ab(rd.u[8], d.tz_lo, d.tz_hi);
    } else { t[0] = 0.0f; t[1] = d.ty_hi; t[2] = d.tz_lo; }
  }
  return VINE_OK;
}

/* reset_idx called outside step (VT:412-427 reset_done): rigid-body views are not refreshed. */
int oracle_reset_idx(const VineConfig* cfg, OracleArrays* a, const int64_t* env_ids, int64_t n) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  for (int64_t i = 0; i < n; ++i) {
    int64_t e = env_ids[i];
    if (e < 0 || e >= a->n) return VINE_ERR_INVALID_ARG;
    ResetDraws rd;
    reset_draws(a->seed, (uint32_t)(a->global_env_offset + e), (uint32_t)a->step_count[e] | 0x80000000u, &rd);
    reset_env(cfg, &d, &rd, a->dof_pos + 6 * e, a->dof_vel + 6 * e, a->target + 3 * e, a->object_info + 2 * e);
    if (!cfg->emulate_stale_body_state) {
      fk_tip(a->dof_pos + 6 * e, a->tip_body + 3 * e); memset(a->tipvel_body + 3 * e, 0, 12);
      a->cart_body_y[e] = a->dof_pos[6 * e]; a->cart_body_vy[e] = 0.0f; a->lip_force[e] = 0.0f;
      a->prev_cart_vel[e] = 0.0f;
    }
    a->prev_cart_vel_error[e] = 0.0f;
    a->reset[e] = 0; a->progress[e] = 0; a->rew[e] = 0.0f; a->agg_rew[e] = 0.0f;
  }
  return VINE_OK;
}

/* ------------------------------------------------------------------------------------------
 * Function-level array wrappers
 * ---------------------------------------------------------------------------------------- */
int oracle_pre_physics(const VineConfig* cfg, int64_t n, const VinePrePhysicsIO* io) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  for (int64_t e = 0; e < n; ++e) {
    float hist[2 * VINE_MAX_ACTION_DELAY + 2];
    if (d.D) memcpy(hist, io->history_in + (size_t)2 * d.D * e, sizeof(float) * 2 * d.D);
    float s = io->smoothed_in[e];
    pre_physics_env(cfg, &d, io->actions[2 * e], io->actions[2 * e + 1],
                    io->action_noise ? io->action_noise + 2 * e : NULL, hist, &s,
                    &io->u_rail_velocity[e], &io->u_fpam[e]);
    io->smoothed_out[e] = s;
    if (d.D) memcpy(io->history_out + (size_t)2 * d.D * e, hist, sizeof(float) * 2 * d.D);
  }
  return VINE_OK;
}

int oracle_actuation(const VineConfig* cfg, int64_t n, const VineActuationIO* io) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  for (int64_t e = 0; e < n; ++e) {
    float pv = io->prev_cart_vel[e], pe = io->prev_cart_vel_error[e];
    actuation_env(&d, io->dof_pos + 6 * e, io->dof_vel + 6 * e, io->cart_vel_y[e],
                  io->u_rail_velocity[e], io->u_fpam_to_use[e],
                  io->dynamics_scaling ? io->dynamics_scaling + 20 * e : NULL,
                  io->accel_scaling ? io->accel_scaling[e] : 1.0f, &pv, &pe, io->dof_efforts + 6 * e);
    io->prev_cart_vel_out[e] = pv; io->prev_cart_vel_error_out[e] = pe;
  }
  return VINE_OK;
}

int oracle_simulate(const VineConfig* cfg, int64_t n, const VineSimulateIO* io, int use_f64) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
  for (int64_t e = 0; e < n; ++e) {
    BodyState b; memset(&b, 0, sizeof(b));
    simulate_env(cfg, use_f64, io->dof_pos + 6 * e, io->dof_vel + 6 * e, io->dof_efforts + 6 * e,
                 io->dynamics_scaling ? io->dynamics_scaling + 20 * e : NULL,
                 io->u_fpam_to_use ? io->u_fpam_to_use[e] : 0.0f, io->target_positions + 3 * e,
                 io->object_info + 2 * e, &b);
    if (io->tip_positions) memcpy(io->tip_positions + 3 * e, b.tip, 12);
    if (io->tip_velocities) memcpy(io->tip_velocities + 3 * e, b.tipvel, 12);
    if (io->shelf_contact_force) io->shelf_contact_force[e] = b.lip;
  }
  return VINE_OK;
}

int oracle_post_physics(const VineConfig* cfg, int64_t n, const VinePostPhysicsIO* io) {
  Derived d; int rc = derive(cfg, &d);
  if (rc) return rc;
  for (int64_t e = 0; e < n; ++e) {
    PostIn in = {io->dof_pos + 6 * e, io->dof_vel + 6 * e, io->prev_dof_pos + 6 * e,
                 io->tip_positions + 3 * e, io->prev_tip_positions + 3 * e, io->tip_velocities + 3 * e,
                 io->target_positions + 3 * e, io->target_velocities + 3 * e, io->object_info + 2 * e,
                 io->cart_positions_y[e], io->smoothed_u_fpam[e], io->u_fpam[e], io->u_rail_velocity[e],
                 io->prev_u_rail_velocity[e],
                 io->contact_force_norms ? io->contact_force_norms + e : NULL, (int)n,
                 io->obs_noise ? io->obs_noise + (size_t)d.O * e : NULL,
                 io->reset_buf_in[e], io->progress_buf[e]};
    post_physics_env(cfg, &d, &in, io->obs_buf + (size_t)d.O * e, &io->rew_buf[e],
                     io->reward_matrix ? io->reward_matrix + VINE_NUM_REWARDS * e : NULL,
                     &io->reset_buf_out[e], &io->timeout_buf[e]);
  }
  return VINE_OK;
}

/* GAE: rl_games A2CBase.discount_values; in-repo analogue learning/common_agent.py:413-425 */
int oracle_gae(const float* rewards, const float* values, const float* dones,
               const float* last_values, const float* last_dones, int64_t T, int64_t N,
               double gamma_d, double tau_d, float* adv, float* ret) {
  /* Python: `self.gamma * nextvalues` and `self.gamma * self.tau * nextnonterminal` -> the
   * double product gamma*tau is rounded to f32 when it meets the tensor */
  const float gamma = (float)gamma_d, gt = (float)(gamma_d * tau_d);
  for (int64_t e = 0; e < N; ++e) {
    float lastgaelam = 0.0f;
    for (int64_t t = T - 1; t >= 0; --t) {
      float nonterm, nextv;
      if (t == T - 1) { nonterm = 1.0f - last_dones[e]; nextv = last_values[e]; }
      else { nonterm = 1.0f - dones[(t + 1) * N + e]; nextv = values[(t + 1) * N + e]; }
      float delta = rewards[t * N + e] + gamma * nextv * nonterm - values[t * N + e];
      lastgaelam = delta + gt * nonterm * lastgaelam;
      adv[t * N + e] = lastgaelam;
      ret[t * N + e] = lastgaelam + values[t * N + e];
    }
  }
  return VINE_OK;
}

void oracle_mass_matrix(const double q[6], double M[36]) { mass_matrix_rel_f64(q, M); }
double oracle_energy(const VineConfig* cfg, const double q[6], const double qd[6]) {
  return energy_f64(cfg, q, qd);
}
