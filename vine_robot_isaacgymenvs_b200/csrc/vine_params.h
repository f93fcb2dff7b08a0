// vine_params.h — f32 constants derived from VineConfig, passed to kernels by value
// (__grid_constant__), plus the baked model constants of the URDF.
//
// Reference abbreviations used in all csrc/ files:
//   V5 = isaacgymenvs/tasks/Vine5LinkMovingBase.py, VT = isaacgymenvs/tasks/base/vec_task.py,
//   YT = isaacgymenvs/cfg/task/Vine5LinkMovingBase.yaml, URDF = assets/urdf/Vine5LinkMovingBase.urdf
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include "../../include/vine_b200.h"

#define VINE_NL 5
#define VINE_MAX_OBS 28
#define VINE_MAX_CFI 8   // controlFrequencyInv upper bound (contact samples kept in registers)
#define VINE_MAX_RECTS 5

// Philox stream ids (ctr.y)
enum { VINE_SITE_ACTION_NOISE = 1, VINE_SITE_DYNAMICS = 2, VINE_SITE_OBS_NOISE = 3, VINE_SITE_RESET = 4 };

struct VineParams {
  // shapes / switches
  int O, C, S, D;
  int obs_type, scaled;
  int shelf, pipe;
  int use_smoothed, force_fpam, force_rail;
  int randomize, implicit_law, stale;
  int rand_dof_init, rand_targets;
  int reach_reset, tip_reset, contact_reset;
  int64_t max_len_m1;            // max_episode_length - 1 (V5:1544)
  // action path (V5:984-1005, 1458-1463)
  float clip_act, clip_obs, act_noise, obs_noise;
  float rail_scale, fpam_range, fpam_min, alpha_inf, alpha_def;
  // controller (V5:1064-1098)
  float dt, control_dt, rail_force_max, rail_accel, p_gain, d_gain;
  float dyn_min, dyn_rng, acc_min, acc_rng;
  float cull_slack;   // contact variant: how far a chain may move before its candidate pairs are re-culled (m)
  // reward / reset (V5:1218-1248)
  float soft_limit, success_dist;
  float w[VINE_NUM_REWARDS];
  float obs_scale[VINE_MAX_OBS];
  // reset sampling (V5:774-914)
  float rev_lo, rev_rng, cart_lo, cart_rng, ty_lo, ty_rng, tz_lo, tz_rng, dep_lo, dep_rng;
  float ty_hi, tz_lo_fixed;
  // dynamics (gym.simulate, VT:356)
  float h, g, damping, stiffness, armature;
  float kc, dc, rest;            // penalty contact
  float beta[VINE_NL], alpha[VINE_NL], mtot;
  float Lbeta[VINE_NL], gbeta[VINE_NL], inv_L;  // L*beta_j, g*beta_j, 1/L (hoisted products)
  float tip0_y, tip0_z;          // tip pose at q = 0
};

// ---- model constants (URDF; SURVEY Appendix B) ----
static const double kLinkLen = 0.0885, kLinkCom = 0.04425, kCartMass = 0.4, kBaseAngle = 3.1415;
static const double kPivotZ = 1.0 - 0.025 - 0.01;
static const double kLinkMass[VINE_NL] = {0.005, 0.005, 0.005, 0.005, 0.1};
static const double kLinkInertia[VINE_NL] = {6.89246e-6, 6.89246e-6, 6.89246e-6, 6.89246e-6, 1.01559e-4};
#define VINE_LINK_LEN 0.0885f
#define VINE_BASE_ANGLE 3.1415f   // kBaseAngle
#define VINE_PIVOT_Z 0.965f
#define VINE_LINK_RADIUS 0.0381f
#define VINE_FPAM_RADIUS 0.0169f
#define VINE_FPAM_OFFSET 0.055f

static const float kObsScale28[28] = {0.12f, 0.269f, 0.148f, 0.249f, 0.148f, 0.344f, 0.67f, 2.22f, 1.47f, 1.14f,
                                      0.903f, 0.716f, 0.0656f, 0.238f, 0.0656f, 0.732f, 2.0f, 0.732f, 0.02f,
                                      0.0235f, 0.02f, 0.732f, 2.0f, 0.732f, 0.845f, 0.86f, 0.0385f, 0.5f};  // V5:246-255
static const float kObsScale18[18] = {0.12f, 0.67f, 0.0656f, 0.238f, 0.0656f, 0.732f, 2.0f, 0.732f, 0.02f, 0.0235f,
                                      0.02f, 0.732f, 2.0f, 0.732f, 0.845f, 0.86f, 0.0385f, 0.5f};           // V5:257-266

static inline int vine_obs_width(int t) {  // V5:152-171
  switch (t) {
    case VINE_OBS_POS_ONLY: return 14;
    case VINE_OBS_POS_AND_VEL:
    case VINE_OBS_POS_AND_FD_VEL:
    case VINE_OBS_POS_AND_PREV_POS: return 26;
    case VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO: return 28;
    case VINE_OBS_TIP_AND_CART_AND_OBJ_INFO: return 18;
    default: return -1;
  }
}

// Where a Python float meets an f32 tensor in the reference it is rounded to f32 there;
// arithmetic between Python floats is done in double first (e.g. FPAM_MAX - FPAM_MIN, V5:1459).
static inline int vine_derive_params(const VineConfig* c, VineParams* p, const char** why) {
  *why = "";
  if (c->struct_size != (int32_t)sizeof(VineConfig)) { *why = "VineConfig.struct_size mismatch"; return VINE_ERR_ABI_MISMATCH; }
  memset(p, 0, sizeof(*p));
  p->O = vine_obs_width(c->observation_type);
  if (p->O < 0) { *why = "unknown OBSERVATION_TYPE"; return VINE_ERR_INVALID_ARG; }
  p->C = c->control_freq_inv; p->S = c->substeps; p->D = c->action_delay;
  if (p->C < 1 || p->C > VINE_MAX_CFI) { *why = "controlFrequencyInv must be in 1..8"; return VINE_ERR_INVALID_ARG; }
  if (p->S < 1) { *why = "sim.substeps must be >= 1"; return VINE_ERR_INVALID_ARG; }
  if (p->D < 0 || p->D > VINE_MAX_ACTION_DELAY) { *why = "ACTION_DELAY must be in 0..8"; return VINE_ERR_INVALID_ARG; }
  if (!(c->dt > 0)) { *why = "sim.dt must be > 0"; return VINE_ERR_INVALID_ARG; }
  p->obs_type = c->observation_type; p->scaled = c->scale_observations != 0;
  for (int i = 0; i < VINE_MAX_OBS; ++i) p->obs_scale[i] = 1.0f;
  if (p->scaled) {  // V5:242-268
    if (c->observation_type == VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO) memcpy(p->obs_scale, kObsScale28, sizeof(kObsScale28));
    else if (c->observation_type == VINE_OBS_TIP_AND_CART_AND_OBJ_INFO) memcpy(p->obs_scale, kObsScale18, sizeof(kObsScale18));
    else { *why = "Observation scaling not implemented for this OBSERVATION_TYPE (V5:267-268)"; return VINE_ERR_UNSUPPORTED; }
  }
  p->shelf = c->create_shelf != 0; p->pipe = c->create_pipe != 0;
  p->use_smoothed = c->use_smoothed_fpam != 0; p->force_fpam = c->force_u_fpam != 0; p->force_rail = c->force_u_rail_velocity != 0;
  p->randomize = c->vine_randomize != 0;
  p->implicit_law = c->torque_law_integration == VINE_TORQUE_LAW_IMPLICIT;
  p->stale = c->emulate_stale_body_state != 0;
  p->rand_dof_init = c->randomize_dof_init != 0; p->rand_targets = c->randomize_targets != 0;
  p->reach_reset = c->use_target_reached_reset != 0; p->tip_reset = c->use_tip_limit_hit_reset != 0;
  p->contact_reset = c->use_nonzero_contact_force_reset != 0;
  p->max_len_m1 = (int64_t)c->max_episode_length - 1;
  p->clip_act = (float)c->clip_actions; p->clip_obs = (float)c->clip_observations;
  p->act_noise = (float)c->action_noise_std; p->obs_noise = (float)c->observation_noise_std;
  p->rail_scale = (float)c->rail_velocity_scale;
  p->fpam_range = (float)(c->fpam_max - c->fpam_min); p->fpam_min = (float)c->fpam_min;
  p->alpha_inf = (float)c->smoothing_alpha_inflate; p->alpha_def = (float)c->smoothing_alpha_deflate;
  p->dt = (float)c->dt; p->control_dt = (float)(c->dt * (double)c->control_freq_inv);
  p->rail_force_max = (float)(c->rail_acceleration / 2.0); p->rail_accel = (float)c->rail_acceleration;
  p->p_gain = (float)c->rail_p_gain; p->d_gain = (float)c->rail_d_gain;
  p->dyn_min = (float)c->dynamics_scaling_min; p->dyn_rng = (float)c->dynamics_scaling_max - p->dyn_min;
  p->acc_min = (float)c->accel_target_scaling_min; p->acc_rng = (float)c->accel_target_scaling_max - p->acc_min;
  p->soft_limit = (float)c->rail_soft_limit; p->success_dist = (float)c->success_dist;
  for (int i = 0; i < VINE_NUM_REWARDS; ++i) p->w[i] = (float)c->reward_weights[i];
  {
    const double ten = 10.0 * 3.14159265358979323846 / 180.0;  // math.radians(10), V5:778-779
    float lo = (float)fmax(c->revolute_lower, -ten), hi = (float)fmin(c->revolute_upper, ten);
    p->rev_lo = lo; p->rev_rng = hi - lo;
    lo = (float)fmax(c->prismatic_lower, c->random_init_cart_min_y); hi = (float)fmin(c->prismatic_upper, c->random_init_cart_max_y);
    p->cart_lo = lo; p->cart_rng = hi - lo;
  }
  p->ty_lo = (float)c->min_target_y; p->ty_rng = (float)c->max_target_y - p->ty_lo; p->ty_hi = (float)c->max_target_y;
  p->tz_lo = (float)c->min_target_z; p->tz_rng = (float)c->max_target_z - p->tz_lo; p->tz_lo_fixed = p->tz_lo;
  p->dep_lo = (float)c->min_target_depth_in_obstacle; p->dep_rng = (float)c->max_target_depth_in_obstacle - p->dep_lo;
  p->h = (float)(c->dt / (double)c->substeps); p->g = (float)(-c->gravity_z);
  p->damping = (float)c->damping; p->stiffness = (float)c->stiffness; p->armature = (float)c->armature;
  p->kc = (float)c->contact_stiffness; p->dc = (float)c->contact_damping; p->rest = (float)c->contact_rest_offset;
  double tail = 0;
  for (int j = VINE_NL - 1; j >= 0; --j) {
    p->beta[j] = (float)(kLinkLen * tail + kLinkCom * kLinkMass[j]);
    p->alpha[j] = (float)(kLinkInertia[j] + kLinkMass[j] * kLinkCom * kLinkCom + kLinkLen * kLinkLen * tail);
    tail += kLinkMass[j];
  }
  p->mtot = (float)(kCartMass + tail);
  for (int j = 0; j < VINE_NL; ++j) { p->Lbeta[j] = (float)kLinkLen * p->beta[j]; p->gbeta[j] = p->g * p->beta[j]; }
  p->inv_L = (float)(1.0 / kLinkLen);
  p->tip0_y = (float)(-5.0 * kLinkLen * sin(kBaseAngle)); p->tip0_z = (float)(kPivotZ + 5.0 * kLinkLen * cos(kBaseAngle));
  return VINE_OK;
}
