// vine_b200.cu — kernels and the C ABI (include/vine_b200.h) of the Vine5LinkMovingBase hot path.
// Target: sm_100a (B200). One fused kernel per control step; one environment per thread with the
// whole articulation state in registers across controlFrequencyInv x substeps integrator steps.
//
// HBM layout (private to the library, structure-of-arrays of 16-byte planes, index = env):
//   S0 = q0..q3 | S1 = q4,q5,qd0,qd1 | S2 = qd2..qd5
//   S3 = smoothed_u_fpam, prev_cart_vel, prev_cart_vel_error, |F_shelf_link|
//   S4 = tip_y, tip_z (rigid-body view), cart body vel y, aggregated reward
//   S5 = target_y, target_z, object depth, object angle        (target_x == 0, V5:892)
//   ring[slot][env] = (u_rail, u_fpam) delay ring, slot = step % ACTION_DELAY | ctr[env] = step count
// VecTask buffers (obs/rew/reset/progress/timeout) are torch-owned row-major tensors (VT:260-283).
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "vine_device.cuh"
#include "vine_launch.cuh"

#define VINE_BLOCK 128
#ifndef VINE_STEP_MIN_BLOCKS
#define VINE_STEP_MIN_BLOCKS 0   // 0 = unspecified: the compiler's own choice (125 registers, 16 warps/SM) is the fastest measured (1 -> 167 registers, -8 %; 4 -> 121, -3 %; 5 -> 96 + spills, -6 %)
#endif
#ifndef VINE_STEP_MIN_BLOCKS_CONTACT
#define VINE_STEP_MIN_BLOCKS_CONTACT 12  // contact variant (1-warp blocks): 160 registers (no spills) instead of 200 -> 12 warps/SM; measured
#endif                                   // +14 % (shelf) / +11 % (pipe): hides the per-warp load imbalance of the narrow phase
#ifndef VINE_STEP2_MIN_BLOCKS
#define VINE_STEP2_MIN_BLOCKS 0  // two-envs-per-thread kernel: the compiler's own register choice
#endif
#define VINE_DBG_W 28  // u_rail,u_fpam,prev_u_rail,rail_force,tipvel y,z, reward_matrix[13], pad, fd dof vel[6], fd tip vel y,z

struct StepArgs {
  int64_t n, gid0;
  int64_t first, end;  // env range [first, end) of this launch (vine_step: 0..n; vine_step_range: a chunk)
  uint32_t k0, k1;
  float4 *S0, *S1, *S2, *S3, *S4, *S5;
  float2* ring;
  uint32_t* ctr;
  const float2* actions;
  float* obs; float* obs_clamped; float* rew;
  int64_t* reset; int64_t* progress; uint8_t* timeout;
  float* dbg;  // [N, VINE_DBG_W] or nullptr
  // contact variant only (else nullptr): per-env "had contact candidates in its last step" flag, the env order of this launch
  // (envs with the flag first, so that they share warps) and the two cursors the binning kernel fills it with
  uint8_t* near; int32_t* perm; int32_t* bin_cursor;
  // obstacle variants, routed step: the launch takes its envs from list[0 .. *list_count) (list_reversed: from the END of the
  // n-entry array backwards); the far pass appends the envs it had to give up to redo_list / redo_count
  const int32_t* list; const int32_t* list_count; int list_reversed;
  int32_t* redo_list; int32_t* redo_count;
};

struct VineEnv {
  VineParams p;
  VineConfig cfg;
  StepArgs a;
  int device;
  int bound;
  // routed step of the obstacle variants: the near pass runs beside the far pass on this stream (forked from and joined back
  // into the caller's stream with the two events, so the whole step stays one capturable unit of the caller's stream)
  cudaStream_t side;
  cudaEvent_t ev_fork, ev_join;
  int prio_hi;
  char err[256];
};

static char g_create_err[256] = "";

#define CUDA_TRY(env, call)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      snprintf((env) ? (env)->err : g_create_err, 256, "%s failed: %s", #call, cudaGetErrorString(_e)); \
      return VINE_ERR_CUDA;                                                                   \
    }                                                                                         \
  } while (0)

// ------------------------------------------------------------------------------------------
// coalesced store of a block's observation rows staged in shared memory
// ------------------------------------------------------------------------------------------
template <int ROWS, int THREADS>
__device__ __forceinline__ void store_obs_block(const float* s_obs, int O, int64_t first, int64_t end, float clip,
                                                float* __restrict__ obs, float* __restrict__ obs_clamped) {
  const int64_t row0 = first + (int64_t)blockIdx.x * ROWS;
  const int rows = (int)min((int64_t)ROWS, end - row0);
  const int count2 = rows * O / 2;  // O is even for every ObservationType
  float2* g = reinterpret_cast<float2*>(obs + row0 * O);
  float2* gc = obs_clamped ? reinterpret_cast<float2*>(obs_clamped + row0 * O) : nullptr;
  const float inv_O = 1.0f / (float)O;
  for (int i = threadIdx.x; i < count2; i += THREADS) {
    // r0 = e0 / O without the 20-instruction integer division (exact: e0 < 256 * 32, the quotient is far from a rounding boundary)
    const int e0 = 2 * i, r0 = (int)(((float)e0 + 0.5f) * inv_O), c0 = e0 - r0 * O;  // c0 even, c0+1 < O
    float2 v;
    v.x = s_obs[r0 * (VINE_MAX_OBS + 1) + c0];
    v.y = s_obs[r0 * (VINE_MAX_OBS + 1) + c0 + 1];
    g[i] = v;
    if (gc) {  // VT:374 torch.clamp(obs_buf, -clip, clip)
      v.x = fminf(fmaxf(v.x, -clip), clip); v.y = fminf(fmaxf(v.y, -clip), clip);
      gc[i] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// The control step of ONE environment, cut at the points where the integrator runs, so that the one-env-per-thread
// kernel (contact variant) and the two-envs-per-thread kernel (free space, packed FP32) share every line of task logic.
// ------------------------------------------------------------------------------------------
struct EnvStep {   // what one env carries in registers across the sim steps of a control step
  float smoothed, prev_cart_vel, prev_err, lip, cart_body_vy;
  float u_rail, u_fpam, u_use, rail_force;
  float new_rail, new_fpam;         // this step's command, pushed into the delay ring at the end of the step
  float tipb_y, tipb_z;             // rigid-body tip as of the refresh before the LAST simulate (V5:797 on reset steps)
  float contact[VINE_MAX_CFI];      // VT:348-351 samples (shelf only)
  uint32_t step, gid;
  bool reset_in;
};

// load + VT:333 + pre_physics_step V5:922-945; returns the env's dynamics state in absolute coordinates
__device__ __forceinline__ void env_begin(const VineParams& p, const StepArgs& a, int64_t e, EnvStep& E, Dyn& d) {
  const float4 s0 = a.S0[e], s1 = a.S1[e], s2 = a.S2[e], s3 = a.S3[e], s4 = a.S4[e];
  const float q[6] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y};
  const float qd[6] = {s1.z, s1.w, s2.x, s2.y, s2.z, s2.w};
  E.smoothed = s3.x; E.prev_cart_vel = s3.y; E.prev_err = s3.z; E.lip = s3.w;
  E.tipb_y = s4.x; E.tipb_z = s4.y; E.cart_body_vy = s4.z;
  E.step = a.ctr[e];
  E.gid = (uint32_t)(a.gid0 + e);
  const float2 act = a.actions[e];
  E.reset_in = a.reset[e] != 0;
  float a0 = fminf(fmaxf(act.x, -p.clip_act), p.clip_act);
  float a1 = fminf(fmaxf(act.y, -p.clip_act), p.clip_act);
  if (p.randomize && p.act_noise != 0.f) {  // V5:930-932 (noise after the clamp)
    float nz[4];
    normal4(philox4x32(a.k0, a.k1, E.gid, VINE_SITE_ACTION_NOISE, E.step, 0), nz);
    a0 = __fadd_rn(a0, __fmul_rn(p.act_noise, nz[0]));
    a1 = __fadd_rn(a1, __fmul_rn(p.act_noise, nz[1]));
  }
  rescale_actions(p, a0, a1, E.u_rail, E.u_fpam);
  E.new_rail = E.u_rail; E.new_fpam = E.u_fpam;
  if (p.D > 0) {  // V5:936-937 FIFO of ACTION_DELAY control steps; the push happens in env_end (nothing is written before the
    const float2 old = a.ring[(int64_t)(E.step % (uint32_t)p.D) * a.n + e];   // step is complete, so a pass may give an env up)
    E.u_rail = old.x; E.u_fpam = old.y;
  }
  apply_overrides_and_smooth(p, E.u_rail, E.u_fpam, E.smoothed);
  E.u_use = p.use_smoothed ? E.smoothed : E.u_fpam;                // V5:1059
  E.rail_force = 0.f;
#pragma unroll
  for (int i = 0; i < VINE_MAX_CFI; ++i) E.contact[i] = 0.f;
  rel_to_abs(q, qd, d);
}

// head of sim step i (VT:338-351): dynamics-scaling draws, rail controller, contact sample, integrator constants
__device__ __forceinline__ void env_sim_step_begin(const VineParams& p, const StepArgs& a, int i, EnvStep& E, const Dyn& d, JointImp& J) {
  if (i > 0 && i == p.C - 1 && E.reset_in && p.stale) {  // only needed by V5:797 on reset steps
    float vy, vz; tip_fk(d, E.tipb_y, E.tipb_z, vy, vz);
  }
  JointLaw law; joint_law_unscaled(law);
  float acc_scale = 1.f;
  if (p.randomize) {  // V5:1053-1055: 20 multipliers re-drawn every sim step (+1 for accel scaling)
    // 16 random bits per multiplier (two per Philox word): 3 Philox calls per sim step instead of 6; multiplier k uses
    // half k of the 24 halves of blocks 8 i .. 8 i + 2, low half first
    const float dyn_rng16 = p.dyn_rng * 1.52587890625e-05f, acc_rng16 = p.acc_rng * 1.52587890625e-05f;   // 2^-16
    uint32_t u[12];
#pragma unroll
    for (uint32_t b = 0; b < 3; ++b) {
      const uint4 r = philox4x32(a.k0, a.k1, E.gid, VINE_SITE_DYNAMICS, E.step, (uint32_t)i * 8u + b);
      u[4 * b] = r.x; u[4 * b + 1] = r.y; u[4 * b + 2] = r.z; u[4 * b + 3] = r.w;
    }
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) {
      law.K[j] = __fmul_rn(law.K[j], uniform_ab16(u[2 * j] & 0xffffu, p.dyn_min, dyn_rng16));
      law.Cd[j] = __fmul_rn(law.Cd[j], uniform_ab16(u[2 * j] >> 16, p.dyn_min, dyn_rng16));
      law.b[j] = __fmul_rn(law.b[j], uniform_ab16(u[2 * j + 1] & 0xffffu, p.dyn_min, dyn_rng16));
      law.B[j] = __fmul_rn(law.B[j], uniform_ab16(u[2 * j + 1] >> 16, p.dyn_min, dyn_rng16));
    }
    acc_scale = uniform_ab16(u[10] & 0xffffu, p.acc_min, acc_rng16);
  }
  // rigid-body cart velocity: stale on the first sim step after a reset (V5:1069, SURVEY D.2)
  const float cart_vel = (i == 0) ? E.cart_body_vy : d.v[0];
  float efforts[6];
  efforts[0] = rail_controller(p, cart_vel, E.u_rail, acc_scale, E.prev_cart_vel, E.prev_err);
  E.rail_force = efforts[0];
  if (!p.implicit_law) {
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) {
      const float th = j == 0 ? d.x[1] : d.x[j + 1] - d.x[j];
      const float thd = j == 0 ? d.v[1] : d.v[j + 1] - d.v[j];
      efforts[j + 1] = joint_torque(law, j, th, thd, E.u_use);
    }
  } else {
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) efforts[j + 1] = 0.f;
  }
  if (p.shelf) {
#pragma unroll
    for (int k = 0; k < VINE_MAX_CFI; ++k) if (k == i) E.contact[k] = E.lip;  // VT:348-351: force of the PREVIOUS simulate
  }
  joint_implicit_consts(p, law, E.u_use, efforts, J);
}

// post_physics_step V5:1110-1120 + VT:366-374 + write-back; the observation row goes to `row` (shared memory).
// Values that the step only needs here (the joint positions and rigid-body tip at the start of the step = prev_dof_pos /
// prev_tip_positions V5:943-944, targets, object info, progress, the reward sum) are re-read from their planes instead of
// being carried in registers across the 40 substeps: the planes still hold the step's input until the write-back below.
__device__ __forceinline__ void env_end(const VineParams& p, const StepArgs& a, int64_t e, EnvStep& E, const Dyn& d, float* row) {
  float q[6], qd[6];
  float tip_y, tip_z, tipvel_y, tipvel_z;
  tip_fk(d, tip_y, tip_z, tipvel_y, tipvel_z);
  float cart_y_body = d.x[0];
  float cart_body_vy = d.v[0];
  abs_to_rel(d, q, qd);
  const float4 s0 = a.S0[e], s1 = a.S1[e], s4 = a.S4[e], s5 = a.S5[e];
  float target[3] = {0.f, s5.x, s5.y};
  float obj[2] = {s5.z, s5.w};
  float agg = s4.w;
  PostIn in;
  in.prev_q[0] = s0.x; in.prev_q[1] = s0.y; in.prev_q[2] = s0.z; in.prev_q[3] = s0.w; in.prev_q[4] = s1.x; in.prev_q[5] = s1.y;  // V5:943
  in.prev_tip[0] = 0.f; in.prev_tip[1] = s4.x; in.prev_tip[2] = s4.y;     // V5:944
  in.prev_u_rail = E.u_rail;                                             // V5:945
  int64_t progress = a.progress[e] + 1;                                  // V5:1111
  int64_t reset_in = E.reset_in ? 1 : 0;
  if (E.reset_in) {  // deferred reset of envs flagged at the end of the previous step (V5:1114-1116)
    reset_env(p, a.k0, a.k1, E.gid, E.step, q, qd, target, obj);
#pragma unroll
    for (int i = 0; i < 6; ++i) in.prev_q[i] = q[i];                     // V5:794
    if (p.stale) {                                                       // V5:796-797 stale rigid-body views
      in.prev_tip[1] = E.tipb_y; in.prev_tip[2] = E.tipb_z;
    } else {                                                             // "as if FK were done": clean episode boundary
      Dyn dn; rel_to_abs(q, qd, dn);
      tip_fk(dn, tip_y, tip_z, tipvel_y, tipvel_z);
      in.prev_tip[1] = tip_y; in.prev_tip[2] = tip_z;
      cart_y_body = q[0]; cart_body_vy = 0.f; E.lip = 0.f; E.prev_cart_vel = 0.f;
#pragma unroll
      for (int i = 0; i < VINE_MAX_CFI; ++i) E.contact[i] = 0.f;
    }
    in.prev_u_rail = 0.f;                                                // V5:798
    E.prev_err = 0.f;                                                    // V5:799
    reset_in = 0; progress = 0; agg = 0.f;                               // V5:807-810
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) { in.q[i] = q[i]; in.qd[i] = qd[i]; }
  in.tip[0] = 0.f; in.tip[1] = tip_y; in.tip[2] = tip_z;
  in.tipvel[0] = 0.f; in.tipvel[1] = tipvel_y; in.tipvel[2] = tipvel_z;
  in.target[0] = target[0]; in.target[1] = target[1]; in.target[2] = target[2];
  in.target_vel[0] = in.target_vel[1] = in.target_vel[2] = 0.f;          // V5:916-918
  in.obj[0] = obj[0]; in.obj[1] = obj[1];
  in.cart_y = cart_y_body; in.smoothed = E.smoothed; in.u_fpam = E.u_fpam; in.u_rail = E.u_rail;
#pragma unroll
  for (int i = 0; i < VINE_MAX_CFI; ++i) in.contact[i] = E.contact[i];
  in.reset_in = reset_in; in.progress = progress;
  float noise[VINE_MAX_OBS];
  const bool noisy = p.randomize && p.obs_noise != 0.f;
  if (noisy) {
#pragma unroll
    for (uint32_t b = 0; b < VINE_MAX_OBS / 4; ++b) {
      if ((int)(4 * b) < p.O) normal4(philox4x32(a.k0, a.k1, E.gid, VINE_SITE_OBS_NOISE, E.step, b), &noise[4 * b]);
    }
  }
  PostOut o;
  post_physics(p, in, noisy ? noise : nullptr, o);
  agg = __fadd_rn(agg, o.rew);                                           // V5:1278

  a.S0[e] = make_float4(q[0], q[1], q[2], q[3]);
  a.S1[e] = make_float4(q[4], q[5], qd[0], qd[1]);
  a.S2[e] = make_float4(qd[2], qd[3], qd[4], qd[5]);
  a.S3[e] = make_float4(E.smoothed, E.prev_cart_vel, E.prev_err, E.lip);
  a.S4[e] = make_float4(tip_y, tip_z, cart_body_vy, agg);
  if (E.reset_in) a.S5[e] = make_float4(target[1], target[2], obj[0], obj[1]);
  if (p.D > 0) a.ring[(int64_t)(E.step % (uint32_t)p.D) * a.n + e] = make_float2(E.new_rail, E.new_fpam);
  a.ctr[e] = E.step + 1u;
  a.rew[e] = o.rew;
  a.reset[e] = o.reset;
  a.progress[e] = progress;
  a.timeout[e] = o.timeout;
#pragma unroll
  for (int i = 0; i < VINE_MAX_OBS; ++i) if (i < p.O) row[i] = o.obs[i];
  if (a.dbg) {
    float* dbg = a.dbg + e * VINE_DBG_W;
    dbg[0] = E.u_rail; dbg[1] = E.u_fpam; dbg[2] = in.prev_u_rail; dbg[3] = E.rail_force;
    dbg[4] = tipvel_y; dbg[5] = tipvel_z;
    dbg[19] = cart_y_body;   // rigid-body cart position: the pre-reset one on a reset step (stale body views, V5:796)
#pragma unroll
    for (int i = 0; i < VINE_NUM_REWARDS; ++i) dbg[6 + i] = o.r[i];
    // finite_difference_dof_vel / finite_difference_tip_velocities (V5:1347-1348), what the reference's per-view-env wandb
    // traces show (V5:1283-1300): the same two expressions compute_observations uses
#pragma unroll
    for (int i = 0; i < 6; ++i) dbg[20 + i] = div_rn(__fsub_rn(in.q[i], in.prev_q[i]), p.control_dt);
    dbg[26] = div_rn(__fsub_rn(in.tip[1], in.prev_tip[1]), p.control_dt);
    dbg[27] = div_rn(__fsub_rn(in.tip[2], in.prev_tip[2]), p.control_dt);
  }
}

// ------------------------------------------------------------------------------------------
// THE fused control step == VecTask.step (VT:319-380), one environment per thread
// ------------------------------------------------------------------------------------------
// Block size: 128 for the free-space variant.  The contact variant uses one warp per block: its warps finish at very
// different times (the narrow phase runs only where something touches), and a block holds its registers until its slowest
// warp is done -- ncu showed 3.2 warps per issue slot parked at the block barrier with 128-thread blocks.
#ifndef VINE_BLOCK_CONTACT
#define VINE_BLOCK_CONTACT 32
#endif

// one observation row (O <= 32 floats) per warp-wide store: for launches whose envs are not consecutive
__device__ __forceinline__ void store_obs_rows_scattered(const VineParams& p, const StepArgs& a, const float* s_obs, int64_t mine) {
  const int lane = threadIdx.x & 31, w0 = threadIdx.x & ~31;
#pragma unroll 1
  for (int r = 0; r < 32; ++r) {
    const int64_t er = __shfl_sync(0xffffffffu, mine, r);
    if (er >= 0 && lane < p.O) {
      const float v = s_obs[(w0 + r) * (VINE_MAX_OBS + 1) + lane];
      a.obs[er * p.O + lane] = v;
      if (a.obs_clamped) a.obs_clamped[er * p.O + lane] = fminf(fmaxf(v, -p.clip_obs), p.clip_obs);
    }
  }
}

// env id of launch slot `slot` (< count): consecutive, or through the launch's list
__device__ __forceinline__ int64_t slot_env(const StepArgs& a, int64_t slot) {
  if (!a.list) return a.first + slot;
  return (int64_t)(a.list_reversed ? a.list[a.n - 1 - slot] : a.list[slot]);
}

template <bool CONTACT>
__global__ void __launch_bounds__(CONTACT ? VINE_BLOCK_CONTACT : VINE_BLOCK, CONTACT ? VINE_STEP_MIN_BLOCKS_CONTACT : VINE_STEP_MIN_BLOCKS)
vine_step_kernel(const __grid_constant__ VineParams p, const StepArgs a) {
  vine_launch::grid_dependency_sync();
  constexpr int BLOCK = CONTACT ? VINE_BLOCK_CONTACT : VINE_BLOCK;
  __shared__ float s_obs[BLOCK * (VINE_MAX_OBS + 1)];
  __shared__ ContactScratch s_contact[CONTACT ? BLOCK / 32 : 1];
  ContactScratch* cs = &s_contact[CONTACT ? threadIdx.x >> 5 : 0];
  const int64_t count = a.list_count ? (int64_t)*a.list_count : a.end - a.first;
  // Listed launches (near / redo pass) hold nothing but envs with contact work; when the list is short enough for the grid,
  // each warp takes only 8 of them (lanes 0..7) and the other 24 lanes are ghosts = workers of the pooled narrow phase.
  // (With a long list 32 envs per warp are faster: 16 -> +8 % / +24 %, 8 -> +22 % / +76 % step time, shelf / pipe at 1 M envs.)
  const int lanes = (CONTACT && a.list && count <= (int64_t)gridDim.x * 8) ? 8 : BLOCK;
  // grid-stride over the launch's slots: listed launches are sized without knowing the list length
#pragma unroll 1
  for (int64_t base = (int64_t)blockIdx.x * lanes; base < count; base += (int64_t)gridDim.x * lanes) {
    const int64_t slot = base + threadIdx.x;
    const bool live = slot < count && (int)threadIdx.x < lanes;
    // Contact variant: the lanes of the warp that have no env of their own (tail of the launch; lanes 8..31 of a short listed
    // launch) run along as ghosts on a copy of the warp's first env -- they never cull or touch, write nothing, and serve as
    // workers of the warp's pooled narrow phase (contact_forces)
    const bool ghost = CONTACT && !live;
    const int64_t e = live ? slot_env(a, slot) : (ghost ? slot_env(a, base) : -1);
    if (live || ghost) {
      EnvStep E; Dyn d;
      env_begin(p, a, e, E, d);
      Obstacles ob = {0, -1, 0.f, 0.f, 0.f, 0.f};
      ContactCache cc = {0u, ghost ? -1e30f : 1e30f, 0u};   // no candidate pairs yet: the first substep culls
      if (CONTACT) { const float4 s5 = a.S5[e]; build_obstacles(p, s5.x, s5.y, s5.z, s5.w, cs, ob); }
      const float m00 = fmaf(p.h, p.damping, p.mtot), m00inv = rcp_approx(m00);
      // ---- controlFrequencyInv x {forces, contact sample, simulate}  VT:338-356 ----
#pragma unroll 1
      for (int i = 0; i < p.C; ++i) {
        JointImp J;
        env_sim_step_begin(p, a, i, E, d, J);
#pragma unroll 1
        for (int s = 0; s < p.S; ++s) substep<CONTACT, float>(p, J, m00, m00inv, E.rail_force, ob, cs, cc, d, E.lip, ghost);
      }
      if (!ghost) {
        env_end(p, a, e, E, d, s_obs + threadIdx.x * (VINE_MAX_OBS + 1));
        if (CONTACT && a.near) a.near[e] = cc.seen != 0u;
      }
    }
    __syncthreads();
    if (CONTACT && a.list) store_obs_rows_scattered(p, a, s_obs, live ? e : -1);
    else store_obs_block<BLOCK, BLOCK>(s_obs, p.O, a.first + base - (int64_t)blockIdx.x * BLOCK, a.end, p.clip_obs, a.obs, a.obs_clamped);   // unlisted: lanes == BLOCK
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Far pass of the obstacle variants.  Most envs of a step are nowhere near their obstacle (random actions: ~2 % with the
// shelf, ~8 % with the pipe), and the contact variant charges them its 155 registers, its one-warp blocks and its 20 KB
// sim-step loop anyway.  So a routed step (vine_step with obstacles) sends the envs that were not near in their last step
// through THIS kernel: the free-space integrator (substep<false>) plus a bound on how far the chain has moved since its
// bounding box last had a gap to the obstacles' (7 instructions per substep).  An env whose boxes come to overlap is given up
// -- nothing has been written for it -- and appended to the redo list, which the contact variant runs afterwards.  An env
// that finishes here never had a contact candidate, so it computed exactly what the contact variant would have (same
// explicit round-to-nearest arithmetic, same link_trig of the same x): results do not depend on the routing.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(VINE_BLOCK) vine_step_far_kernel(const __grid_constant__ VineParams p, const StepArgs a) {
  __shared__ float s_obs[VINE_BLOCK * (VINE_MAX_OBS + 1)];
  const int64_t count = a.list_count ? a.n - (int64_t)*a.list_count : a.n;   // list_count = number of NEAR envs at the front
  const int64_t slot = (int64_t)blockIdx.x * VINE_BLOCK + threadIdx.x;
  if ((int64_t)blockIdx.x * VINE_BLOCK >= count) return;
  const bool live = slot < count;
  int64_t e = live ? slot_env(a, slot) : -1;
  if (live) {
    EnvStep E; Dyn d;
    env_begin(p, a, e, E, d);
    Obstacles ob;
    { const float4 s5 = a.S5[e]; obstacle_bbox(p, s5.x, s5.y, s5.z, s5.w, ob); }
    float gap = chain_obstacle_gap(p, ob, d);
    bool given_up = !(gap > 0.f);
    float disp = -gap;
    ContactCache cc = {0u, 0.f, 0u};
    const float m00 = fmaf(p.h, p.damping, p.mtot), m00inv = rcp_approx(m00);
#pragma unroll 1
    for (int i = 0; i < p.C && !given_up; ++i) {
      JointImp J;
      env_sim_step_begin(p, a, i, E, d, J);
#pragma unroll 1
      for (int s = 0; s < p.S; ++s) {
        substep<false, float>(p, J, m00, m00inv, E.rail_force, ob, nullptr, cc, d, E.lip);
        disp += chain_displacement_bound(p, d);
        if (disp > p.cull_slack) {          // the chain may have reached the boxes' gap: measure it again
          gap = chain_obstacle_gap(p, ob, d);
          if (!(gap > 0.f)) { given_up = true; break; }
          disp = -gap;
        }
      }
      E.lip = 0.f;                          // nothing touched during this simulate (VT:348-351 samples it next sim step)
    }
    if (given_up) {
      a.redo_list[atomicAdd(a.redo_count, 1)] = (int32_t)e;
      e = -1;                               // no observation row
    } else {
      env_end(p, a, e, E, d, s_obs + threadIdx.x * (VINE_MAX_OBS + 1));
      // (marking envs near ahead of time -- within one step's reach of the gap, or just reset -- was measured: the near pass
      // grows faster than the redo pass shrinks, 0.97 -> 1.13 ms per 1 M shelf envs)
      a.near[e] = 0;
    }
  }
  __syncthreads();
  store_obs_rows_scattered(p, a, s_obs, e);
}

// ------------------------------------------------------------------------------------------
// The free-space control step with TWO environments per thread: thread t of a block owns envs base + t and
// base + VINE_BLOCK2 + t (both coalesced), integrates them in the two lanes of FFMA2/FMUL2/FADD2 (substep<false, float2>)
// and runs the scalar task logic (bit-exact to the reference's torch kernels) once per env.
// ------------------------------------------------------------------------------------------
#define VINE_BLOCK2 128
__global__ void __launch_bounds__(VINE_BLOCK2, VINE_STEP2_MIN_BLOCKS)
vine_step2_kernel(const __grid_constant__ VineParams p, const StepArgs a) {
  __shared__ float s_obs[2 * VINE_BLOCK2 * (VINE_MAX_OBS + 1)];
  const int64_t eA = a.first + (int64_t)blockIdx.x * (2 * VINE_BLOCK2) + threadIdx.x;
  const int64_t eB0 = eA + VINE_BLOCK2;
  const bool liveA = eA < a.end, liveB = eB0 < a.end;
  const int64_t eB = liveB ? eB0 : eA;   // a ragged tail integrates env A in both lanes and stores it once
  if (liveA) {
    EnvStep EA, EB;
    DynT<float2> d2;
    {
      Dyn dA, dB;
      env_begin(p, a, eA, EA, dA);
      env_begin(p, a, eB, EB, dB);
      pack2(dA, dB, d2);
    }
    Obstacles ob = {0, -1, 0.f, 0.f, 0.f, 0.f};
    ContactCache cc = {0u, 1e30f, 0u};
    float lip_unused = 0.f;
    const float m00 = fmaf(p.h, p.damping, p.mtot), m00inv = rcp_approx(m00);
#pragma unroll 1
    for (int i = 0; i < p.C; ++i) {
      JointImpT<float2> J2;
      float2 rail;
      {
        Dyn dA, dB; unpack2(d2, dA, dB);
        JointImp JA, JB;
        env_sim_step_begin(p, a, i, EA, dA, JA);
        env_sim_step_begin(p, a, i, EB, dB, JB);
        pack2(JA, JB, J2);
        rail = make_float2(EA.rail_force, EB.rail_force);
      }
#pragma unroll 1
      for (int s = 0; s < p.S; ++s) substep<false, float2>(p, J2, m00, m00inv, rail, ob, nullptr, cc, d2, lip_unused);
    }
    Dyn dA, dB; unpack2(d2, dA, dB);
    env_end(p, a, eA, EA, dA, s_obs + threadIdx.x * (VINE_MAX_OBS + 1));
    if (liveB) env_end(p, a, eB, EB, dB, s_obs + (VINE_BLOCK2 + threadIdx.x) * (VINE_MAX_OBS + 1));
  }
  __syncthreads();
  store_obs_block<2 * VINE_BLOCK2, VINE_BLOCK2>(s_obs, p.O, a.first, a.end, p.clip_obs, a.obs, a.obs_clamped);
}

// Env order of a binned launch of the contact variant: envs that had contact candidates in their last step first, the others
// from the back. A warp then runs the narrow phase with most of its lanes or none; per-env results do not depend on the
// order (no cross-lane arithmetic), so the unordered cursors are fine.
__global__ void __launch_bounds__(1024) vine_bin_kernel(const StepArgs a) {
  __shared__ int s_near[32], s_far[32], s_base[2];
  const int64_t e = (int64_t)blockIdx.x * 1024 + threadIdx.x;
  const bool valid = e < a.n, nr = valid && a.near[e] != 0;
  const unsigned bn = __ballot_sync(0xffffffffu, nr), bf = __ballot_sync(0xffffffffu, valid && !nr);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_near[warp] = __popc(bn); s_far[warp] = __popc(bf); }
  __syncthreads();
  if (warp == 0) {
    const int cn = s_near[lane], cf = s_far[lane];
    int in = cn, jf = cf;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int tn = __shfl_up_sync(0xffffffffu, in, off), tf = __shfl_up_sync(0xffffffffu, jf, off);
      if (lane >= off) { in += tn; jf += tf; }
    }
    s_near[lane] = in - cn; s_far[lane] = jf - cf;   // exclusive prefix over the warps of this block
    if (lane == 31) { s_base[0] = atomicAdd(a.bin_cursor, in); s_base[1] = atomicAdd(a.bin_cursor + 1, jf); }
  }
  __syncthreads();
  if (!valid) return;
  const unsigned lt = (1u << lane) - 1u;
  if (nr) a.perm[s_base[0] + s_near[warp] + __popc(bn & lt)] = (int32_t)e;
  else a.perm[a.n - 1 - (s_base[1] + s_far[warp] + __popc(bf & lt))] = (int32_t)e;
}

// ------------------------------------------------------------------------------------------
// init / reset_idx / get / set state
// ------------------------------------------------------------------------------------------
__global__ void vine_init_kernel(const __grid_constant__ VineParams p, const StepArgs a) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.n) return;
  // state right after Vine5LinkMovingBase.__init__ (V5:178-291): q = 0, initial targets (V5:179)
  uint32_t u[12];
  for (uint32_t b = 0; b < 3; ++b) {
    const uint4 r = philox4x32(a.k0, a.k1, (uint32_t)(a.gid0 + e), VINE_SITE_RESET, 0x40000000u, b);
    u[4 * b] = r.x; u[4 * b + 1] = r.y; u[4 * b + 2] = r.z; u[4 * b + 3] = r.w;
  }
  float target[3]; sample_targets(p, u, target);
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  a.S0[e] = z; a.S1[e] = z; a.S2[e] = z; a.S3[e] = z;
  a.S4[e] = make_float4(p.tip0_y, p.tip0_z, 0.f, 0.f);
  a.S5[e] = make_float4(target[1], target[2], 0.f, 0.f);
  for (int k = 0; k < p.D; ++k) a.ring[(int64_t)k * a.n + e] = make_float2(0.f, 0.f);
  a.ctr[e] = 0u;
}

// reset_idx outside step (VT:412-427 reset_done; 'R' key V5:715-718): rigid-body views untouched
__global__ void vine_reset_idx_kernel(const __grid_constant__ VineParams p, const StepArgs a, const int64_t* ids, int64_t n_ids) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_ids) return;
  const int64_t e = ids[i];
  if (e < 0 || e >= a.n) return;
  float q[6], qd[6], target[3], obj[2];
  const float4 s5 = a.S5[e];
  target[0] = 0.f; target[1] = s5.x; target[2] = s5.y; obj[0] = s5.z; obj[1] = s5.w;
  reset_env(p, a.k0, a.k1, (uint32_t)(a.gid0 + e), a.ctr[e] | 0x80000000u, q, qd, target, obj);
  float4 s3 = a.S3[e], s4 = a.S4[e];
  s3.z = 0.f;  // prev_cart_vel_error, V5:799
  s4.w = 0.f;  // aggregated_rew_buf, V5:810
  if (!p.stale) {
    Dyn d; rel_to_abs(q, qd, d);
    float vy, vz; tip_fk(d, s4.x, s4.y, vy, vz);
    s4.z = 0.f; s3.w = 0.f; s3.y = 0.f;
  }
  a.S0[e] = make_float4(q[0], q[1], q[2], q[3]);
  a.S1[e] = make_float4(q[4], q[5], 0.f, 0.f);
  a.S2[e] = make_float4(0.f, 0.f, 0.f, 0.f);
  a.S3[e] = s3; a.S4[e] = s4;
  a.S5[e] = make_float4(target[1], target[2], obj[0], obj[1]);
  if (a.reset) a.reset[e] = 0;
  if (a.progress) a.progress[e] = 0;
  if (a.rew) a.rew[e] = 0.f;
}

__global__ void vine_state_kernel(const __grid_constant__ VineParams p, const StepArgs a, const VineStateView v, int set) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= a.n) return;
  float4 s0 = a.S0[e], s1 = a.S1[e], s2 = a.S2[e], s3 = a.S3[e], s4 = a.S4[e], s5 = a.S5[e];
  uint32_t ctr = a.ctr[e];
  if (set) {
    if (v.dof_pos) { const float* q = v.dof_pos + 6 * e; s0 = make_float4(q[0], q[1], q[2], q[3]); s1.x = q[4]; s1.y = q[5]; }
    if (v.dof_vel) { const float* q = v.dof_vel + 6 * e; s1.z = q[0]; s1.w = q[1]; s2 = make_float4(q[2], q[3], q[4], q[5]); }
    if (v.tip_positions) { s4.x = v.tip_positions[3 * e + 1]; s4.y = v.tip_positions[3 * e + 2]; }
    if (v.cart_body_vel_y) s4.z = v.cart_body_vel_y[e];
    if (v.target_positions) { s5.x = v.target_positions[3 * e + 1]; s5.y = v.target_positions[3 * e + 2]; }
    if (v.object_info) { s5.z = v.object_info[2 * e]; s5.w = v.object_info[2 * e + 1]; }
    if (v.smoothed_u_fpam) s3.x = v.smoothed_u_fpam[e];
    if (v.prev_cart_vel) s3.y = v.prev_cart_vel[e];
    if (v.prev_cart_vel_error) s3.z = v.prev_cart_vel_error[e];
    if (v.shelf_contact_force) s3.w = v.shelf_contact_force[e];
    if (v.aggregated_rew_buf) s4.w = v.aggregated_rew_buf[e];
    if (v.step_count) ctr = (uint32_t)v.step_count[e];
    if (v.actions_history)
      for (int k = 0; k < p.D; ++k) {
        const float* h = v.actions_history + (e * p.D + k) * 2;
        a.ring[(int64_t)((ctr + (uint32_t)k) % (uint32_t)p.D) * a.n + e] = make_float2(h[0], h[1]);
      }
    a.S0[e] = s0; a.S1[e] = s1; a.S2[e] = s2; a.S3[e] = s3; a.S4[e] = s4; a.S5[e] = s5; a.ctr[e] = ctr;
    return;
  }
  if (v.dof_pos) { float* q = v.dof_pos + 6 * e; q[0] = s0.x; q[1] = s0.y; q[2] = s0.z; q[3] = s0.w; q[4] = s1.x; q[5] = s1.y; }
  if (v.dof_vel) { float* q = v.dof_vel + 6 * e; q[0] = s1.z; q[1] = s1.w; q[2] = s2.x; q[3] = s2.y; q[4] = s2.z; q[5] = s2.w; }
  if (v.tip_positions) { v.tip_positions[3 * e] = 0.f; v.tip_positions[3 * e + 1] = s4.x; v.tip_positions[3 * e + 2] = s4.y; }
  if (v.cart_body_vel_y) v.cart_body_vel_y[e] = s4.z;
  if (v.target_positions) { v.target_positions[3 * e] = 0.f; v.target_positions[3 * e + 1] = s5.x; v.target_positions[3 * e + 2] = s5.y; }
  if (v.object_info) { v.object_info[2 * e] = s5.z; v.object_info[2 * e + 1] = s5.w; }
  if (v.smoothed_u_fpam) v.smoothed_u_fpam[e] = s3.x;
  if (v.prev_cart_vel) v.prev_cart_vel[e] = s3.y;
  if (v.prev_cart_vel_error) v.prev_cart_vel_error[e] = s3.z;
  if (v.shelf_contact_force) v.shelf_contact_force[e] = s3.w;
  if (v.aggregated_rew_buf) v.aggregated_rew_buf[e] = s4.w;
  if (v.step_count) v.step_count[e] = (int64_t)ctr;
  if (v.actions_history)
    for (int k = 0; k < p.D; ++k) {
      const float2 h = a.ring[(int64_t)((ctr + (uint32_t)k) % (uint32_t)p.D) * a.n + e];
      v.actions_history[(e * p.D + k) * 2] = h.x; v.actions_history[(e * p.D + k) * 2 + 1] = h.y;
    }
  if (a.dbg) {
    const float* dbg = a.dbg + e * VINE_DBG_W;
    if (v.u_rail_velocity) v.u_rail_velocity[e] = dbg[0];
    if (v.u_fpam) v.u_fpam[e] = dbg[1];
    if (v.prev_u_rail_velocity) v.prev_u_rail_velocity[e] = dbg[2];
    if (v.rail_force) v.rail_force[e] = dbg[3];
    if (v.tip_velocities) { v.tip_velocities[3 * e] = 0.f; v.tip_velocities[3 * e + 1] = dbg[4]; v.tip_velocities[3 * e + 2] = dbg[5]; }
    if (v.reward_matrix) for (int i = 0; i < VINE_NUM_REWARDS; ++i) v.reward_matrix[VINE_NUM_REWARDS * e + i] = dbg[6 + i];
    if (v.cart_body_pos_y) v.cart_body_pos_y[e] = dbg[19];
    if (v.finite_difference_dof_vel) for (int i = 0; i < 6; ++i) v.finite_difference_dof_vel[6 * e + i] = dbg[20 + i];
    if (v.finite_difference_tip_velocities) {
      v.finite_difference_tip_velocities[3 * e] = 0.f;
      v.finite_difference_tip_velocities[3 * e + 1] = dbg[26]; v.finite_difference_tip_velocities[3 * e + 2] = dbg[27];
    }
  }
}

// ------------------------------------------------------------------------------------------
// function-level kernels (same device functions as the fused step)
// ------------------------------------------------------------------------------------------
__global__ void vine_post_physics_kernel(const __grid_constant__ VineParams p, int64_t n, const VinePostPhysicsIO io) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  PostIn in;
  for (int i = 0; i < 6; ++i) { in.q[i] = io.dof_pos[6 * e + i]; in.qd[i] = io.dof_vel[6 * e + i]; in.prev_q[i] = io.prev_dof_pos[6 * e + i]; }
  for (int i = 0; i < 3; ++i) {
    in.tip[i] = io.tip_positions[3 * e + i]; in.prev_tip[i] = io.prev_tip_positions[3 * e + i];
    in.tipvel[i] = io.tip_velocities[3 * e + i]; in.target[i] = io.target_positions[3 * e + i];
    in.target_vel[i] = io.target_velocities[3 * e + i];
  }
  in.obj[0] = io.object_info[2 * e]; in.obj[1] = io.object_info[2 * e + 1];
  in.cart_y = io.cart_positions_y[e]; in.smoothed = io.smoothed_u_fpam[e]; in.u_fpam = io.u_fpam[e];
  in.u_rail = io.u_rail_velocity[e]; in.prev_u_rail = io.prev_u_rail_velocity[e];
  for (int i = 0; i < VINE_MAX_CFI; ++i) in.contact[i] = (io.contact_force_norms && i < p.C) ? io.contact_force_norms[(int64_t)i * n + e] : 0.f;
  in.reset_in = io.reset_buf_in[e]; in.progress = io.progress_buf[e];
  float noise[VINE_MAX_OBS];
  const bool noisy = p.randomize && io.obs_noise != nullptr;
  if (noisy) for (int i = 0; i < p.O; ++i) noise[i] = io.obs_noise[(int64_t)p.O * e + i];
  PostOut o;
  post_physics(p, in, noisy ? noise : nullptr, o);
  for (int i = 0; i < p.O; ++i) io.obs_buf[(int64_t)p.O * e + i] = o.obs[i];
  io.rew_buf[e] = o.rew;
  if (io.reward_matrix) for (int i = 0; i < VINE_NUM_REWARDS; ++i) io.reward_matrix[VINE_NUM_REWARDS * e + i] = o.r[i];
  io.reset_buf_out[e] = o.reset;
  io.timeout_buf[e] = o.timeout;
}

__global__ void vine_pre_physics_kernel(const __grid_constant__ VineParams p, int64_t n, const VinePrePhysicsIO io) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float a0 = io.actions[2 * e], a1 = io.actions[2 * e + 1];
  if (p.randomize && io.action_noise) {
    a0 = __fadd_rn(a0, __fmul_rn(p.act_noise, io.action_noise[2 * e]));
    a1 = __fadd_rn(a1, __fmul_rn(p.act_noise, io.action_noise[2 * e + 1]));
  }
  float u_rail, u_fpam;
  rescale_actions(p, a0, a1, u_rail, u_fpam);
  if (p.D > 0) {
    const float* hi = io.history_in + (int64_t)2 * p.D * e;
    float* ho = io.history_out + (int64_t)2 * p.D * e;
    const float o_rail = hi[0], o_fpam = hi[1];
    for (int k = 0; k + 1 < p.D; ++k) { ho[2 * k] = hi[2 * k + 2]; ho[2 * k + 1] = hi[2 * k + 3]; }
    ho[2 * (p.D - 1)] = u_rail; ho[2 * (p.D - 1) + 1] = u_fpam;
    u_rail = o_rail; u_fpam = o_fpam;
  }
  float s = io.smoothed_in[e];
  apply_overrides_and_smooth(p, u_rail, u_fpam, s);
  io.u_rail_velocity[e] = u_rail; io.u_fpam[e] = u_fpam; io.smoothed_out[e] = s;
}

__global__ void vine_actuation_kernel(const __grid_constant__ VineParams p, int64_t n, const VineActuationIO io) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  JointLaw law; joint_law_unscaled(law);
  if (io.dynamics_scaling) {
    const float* s = io.dynamics_scaling + 20 * e;
    for (int j = 0; j < VINE_NL; ++j) {
      law.K[j] = __fmul_rn(law.K[j], s[4 * j]); law.Cd[j] = __fmul_rn(law.Cd[j], s[4 * j + 1]);
      law.b[j] = __fmul_rn(law.b[j], s[4 * j + 2]); law.B[j] = __fmul_rn(law.B[j], s[4 * j + 3]);
    }
  }
  float pv = io.prev_cart_vel[e], pe = io.prev_cart_vel_error[e];
  io.dof_efforts[6 * e] = rail_controller(p, io.cart_vel_y[e], io.u_rail_velocity[e],
                                          io.accel_scaling ? io.accel_scaling[e] : 1.f, pv, pe);
  for (int j = 0; j < VINE_NL; ++j)
    io.dof_efforts[6 * e + j + 1] = joint_torque(law, j, io.dof_pos[6 * e + j + 1], io.dof_vel[6 * e + j + 1], io.u_fpam_to_use[e]);
  io.prev_cart_vel_out[e] = pv; io.prev_cart_vel_error_out[e] = pe;
}

template <bool CONTACT>
__global__ void __launch_bounds__(VINE_BLOCK) vine_simulate_kernel(const __grid_constant__ VineParams p, int64_t n, const VineSimulateIO io) {
  __shared__ ContactScratch s_contact[CONTACT ? VINE_BLOCK / 32 : 1];
  ContactScratch* cs = &s_contact[CONTACT ? threadIdx.x >> 5 : 0];
  const int64_t e0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool ghost = e0 >= n;                       // tail lanes run along on a copy of the last env (contact_forces needs whole warps)
  if (ghost && !CONTACT) return;
  const int64_t e = ghost ? n - 1 : e0;
  float q[6], qd[6], efforts[6];
  for (int i = 0; i < 6; ++i) { q[i] = io.dof_pos[6 * e + i]; qd[i] = io.dof_vel[6 * e + i]; efforts[i] = io.dof_efforts[6 * e + i]; }
  JointLaw law; joint_law_unscaled(law);
  if (io.dynamics_scaling) {
    const float* s = io.dynamics_scaling + 20 * e;
    for (int j = 0; j < VINE_NL; ++j) {
      law.K[j] = __fmul_rn(law.K[j], s[4 * j]); law.Cd[j] = __fmul_rn(law.Cd[j], s[4 * j + 1]);
      law.b[j] = __fmul_rn(law.b[j], s[4 * j + 2]); law.B[j] = __fmul_rn(law.B[j], s[4 * j + 3]);
    }
  }
  const float u_use = io.u_fpam_to_use ? io.u_fpam_to_use[e] : 0.f;
  Obstacles ob = {0, -1, 0.f, 0.f, 0.f, 0.f};
  ContactCache cc = {0u, ghost ? -1e30f : 1e30f, 0u};
  if (CONTACT) build_obstacles(p, io.target_positions[3 * e + 1], io.target_positions[3 * e + 2],
                               io.object_info[2 * e], io.object_info[2 * e + 1], cs, ob);
  Dyn d; rel_to_abs(q, qd, d);
  JointImp J; joint_implicit_consts(p, law, u_use, efforts, J);
  float lip = 0.f;
  const float m00 = fmaf(p.h, p.damping, p.mtot), m00inv = rcp_approx(m00);
#pragma unroll 1
  for (int s = 0; s < p.S; ++s) substep<CONTACT, float>(p, J, m00, m00inv, efforts[0], ob, cs, cc, d, lip, ghost);
  if (ghost) return;
  float ty, tz, vy, vz; tip_fk(d, ty, tz, vy, vz);
  abs_to_rel(d, q, qd);
  for (int i = 0; i < 6; ++i) { io.dof_pos[6 * e + i] = q[i]; io.dof_vel[6 * e + i] = qd[i]; }
  if (io.tip_positions) { io.tip_positions[3 * e] = 0.f; io.tip_positions[3 * e + 1] = ty; io.tip_positions[3 * e + 2] = tz; }
  if (io.tip_velocities) { io.tip_velocities[3 * e] = 0.f; io.tip_velocities[3 * e + 1] = vy; io.tip_velocities[3 * e + 2] = vz; }
  if (io.shelf_contact_force) io.shelf_contact_force[e] = lip;
}

__global__ void vine_philox_kernel(uint32_t k0, uint32_t k1, uint32_t gid, uint32_t site, uint32_t step, uint32_t block0,
                                   int64_t n_blocks, uint32_t* out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_blocks) return;
  const uint4 r = philox4x32(k0, k1, gid, site, step, block0 + (uint32_t)i);
  out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
}

// ------------------------------------------------------------------------------------------
// GAE over the horizon (rl_games A2CBase.discount_values; analogue learning/common_agent.py:413-425).
// A_t = delta_t + c_t A_{t+1} is an affine recurrence: each warp owns 32 consecutive envs (coalesced
// [T,N] rows) and walks the horizon backwards; the f32 operation order is the reference's, so the
// result is bit-identical to the sequential Python loop.
// ------------------------------------------------------------------------------------------
__global__ void vine_gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                const float* __restrict__ dones, const float* __restrict__ last_values,
                                const float* __restrict__ last_dones, int64_t T, int64_t N, float gamma, float gt,
                                float* __restrict__ adv, float* __restrict__ ret) {
  vine_launch::grid_dependency_sync();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= N) return;
  float nextv = last_values[e], nonterm = __fsub_rn(1.0f, last_dones[e]), lastgaelam = 0.f;
  // software prefetch: issue the loads of step t-1 before the dependent math of step t
  float r = rewards[(T - 1) * N + e], v = values[(T - 1) * N + e], dn = dones[(T - 1) * N + e];
  for (int64_t t = T - 1; t >= 0; --t) {
    float r2 = 0.f, v2 = 0.f, d2 = 0.f;
    if (t > 0) { r2 = rewards[(t - 1) * N + e]; v2 = values[(t - 1) * N + e]; d2 = dones[(t - 1) * N + e]; }
    const float delta = __fsub_rn(__fadd_rn(r, __fmul_rn(__fmul_rn(gamma, nextv), nonterm)), v);
    lastgaelam = __fadd_rn(delta, __fmul_rn(__fmul_rn(gt, nonterm), lastgaelam));
    adv[t * N + e] = lastgaelam;
    ret[t * N + e] = __fadd_rn(lastgaelam, v);
    nextv = v; nonterm = __fsub_rn(1.0f, dn);
    r = r2; v = v2; dn = d2;
  }
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
static inline unsigned grid_for(int64_t n, int block) { return (unsigned)((n + block - 1) / block); }

extern "C" {

int vine_abi_version(void) { return VINE_ABI_VERSION; }

int vine_set_programmatic_launch(int enabled) {
  const int before = vine_launch::programmatic_launch_enabled();
  vine_launch::programmatic_launch_enabled() = enabled ? 1 : 0;
  return before;
}

int vine_config_defaults(VineConfig* c) {  // YT:7-134
  if (!c) return VINE_ERR_INVALID_ARG;
  memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(*c);
  c->substeps = 10; c->dt = 0.00833; c->gravity_z = -9.81;
  c->control_freq_inv = 4; c->max_episode_length = 500;
  c->clip_observations = 5.0; c->clip_actions = 1.0;
  c->observation_type = VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO; c->scale_observations = 1;
  c->create_shelf = 0; c->create_pipe = 1;
  c->use_smoothed_fpam = 1; c->action_delay = 1;
  c->smoothing_alpha_inflate = 0.81; c->smoothing_alpha_deflate = 0.86;
  c->fpam_min = -0.1; c->fpam_max = 3.0; c->rail_velocity_scale = 1.0;
  c->damping = 2e-2; c->stiffness = 0.0;
  c->rail_soft_limit = 0.3; c->rail_p_gain = 10.0; c->rail_d_gain = 0.0; c->rail_acceleration = 8.0;
  c->randomize_dof_init = 1; c->randomize_targets = 1;
  c->random_init_cart_min_y = -0.1 * 0.3; c->random_init_cart_max_y = 0.3;
  c->success_dist = 0.08;
  c->min_target_depth_in_obstacle = -0.05; c->max_target_depth_in_obstacle = 0.2;
  c->min_target_y = -0.48; c->max_target_y = -0.4; c->min_target_z = 0.58; c->max_target_z = 0.67;
  const double w[VINE_NUM_REWARDS] = {0, 0, 1, 0, 0.1, 0, 0, 0, 0, 1, 0, 0, 0.10};
  memcpy(c->reward_weights, w, sizeof(w));
  c->use_target_reached_reset = 1;
  c->vine_randomize = 1;
  c->dynamics_scaling_min = 0.999; c->dynamics_scaling_max = 1.001;
  c->accel_target_scaling_min = 1.0; c->accel_target_scaling_max = 1.0;
  c->torque_law_integration = VINE_TORQUE_LAW_IMPLICIT;
  c->emulate_stale_body_state = 1;
  c->revolute_lower = -3.4e38; c->revolute_upper = 3.4e38;
  c->prismatic_lower = -3.4e38; c->prismatic_upper = 3.4e38;
  c->contact_stiffness = 2000.0; c->contact_damping = 2.0; c->contact_rest_offset = 0.001;
  c->contact_cull_slack = 0.01; c->contact_binning = 1; c->step_kernel_variant = VINE_STEP_KERNEL_AUTO;
  return VINE_OK;
}

int vine_num_observations(int t) { const int w = vine_obs_width(t); return w < 0 ? VINE_ERR_INVALID_ARG : w; }

const char* vine_last_error(const VineEnv* env) { return env ? env->err : g_create_err; }

void vine_destroy(VineEnv* env) {
  if (!env) return;
  cudaSetDevice(env->device);
  cudaFree(env->a.S0); cudaFree(env->a.S1); cudaFree(env->a.S2); cudaFree(env->a.S3); cudaFree(env->a.S4);
  cudaFree(env->a.S5); cudaFree(env->a.ring); cudaFree(env->a.ctr); cudaFree(env->a.dbg);
  cudaFree(env->a.near); cudaFree(env->a.perm); cudaFree(env->a.bin_cursor); cudaFree(env->a.redo_list);
  if (env->side) cudaStreamDestroy(env->side);
  if (env->ev_fork) cudaEventDestroy(env->ev_fork);
  if (env->ev_join) cudaEventDestroy(env->ev_join);
  delete env;
}

int vine_create(const VineConfig* cfg, int64_t num_envs, int64_t global_env_offset, int device, uint64_t seed,
                VineEnv** out) {
  if (!cfg || !out || num_envs <= 0 || global_env_offset < 0) { snprintf(g_create_err, 256, "invalid argument"); return VINE_ERR_INVALID_ARG; }
  if (global_env_offset + num_envs > 0xFFFFFFFFll) { snprintf(g_create_err, 256, "global env id exceeds 32 bits"); return VINE_ERR_INVALID_ARG; }
  VineParams p; const char* why;
  const int rc = vine_derive_params(cfg, &p, &why);
  if (rc != VINE_OK) { snprintf(g_create_err, 256, "%s", why); return rc; }
  VineEnv* env = new VineEnv();
  memset(env, 0, sizeof(*env));
  // contact variant: re-cull slack in metres (measured on B200: 0.005-0.01 best, 0.04 is 5-10 % slower)
  p.cull_slack = cfg->contact_cull_slack > 0.0 ? (float)cfg->contact_cull_slack : 0.01f;
  if (cfg->step_kernel_variant < VINE_STEP_KERNEL_AUTO || cfg->step_kernel_variant > VINE_STEP_KERNEL_TWO_ENVS_PACKED) {
    snprintf(g_create_err, 256, "unknown step_kernel_variant"); return VINE_ERR_INVALID_ARG;
  }
  env->p = p; env->cfg = *cfg; env->device = device;
  StepArgs& a = env->a;
  a.n = num_envs; a.first = 0; a.end = num_envs; a.gid0 = global_env_offset; a.k0 = (uint32_t)seed; a.k1 = (uint32_t)(seed >> 32);
  cudaError_t e = cudaSetDevice(device);
  const size_t n = (size_t)num_envs;
  if (e == cudaSuccess) e = cudaMalloc(&a.S0, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.S1, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.S2, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.S3, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.S4, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.S5, n * sizeof(float4));
  if (e == cudaSuccess) e = cudaMalloc(&a.ring, n * sizeof(float2) * (size_t)(p.D > 0 ? p.D : 1));
  if (e == cudaSuccess) e = cudaMalloc(&a.ctr, n * sizeof(uint32_t));
  // contact variant: bin the envs by "had contact candidates" before every full step
  if ((p.shelf || p.pipe) && cfg->contact_binning) {
    if (e == cudaSuccess) e = cudaMalloc(&a.near, n);
    if (e == cudaSuccess) e = cudaMemset(a.near, 0, n);
    if (e == cudaSuccess) e = cudaMalloc(&a.perm, n * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc(&a.redo_list, n * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc(&a.bin_cursor, 4 * sizeof(int32_t));   // near cursor, far cursor, redo count, pad
    if (e == cudaSuccess) {   // the near pass (few, slow warps) gets its blocks placed ahead of the far pass's: it then runs beside it
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);
      env->prio_hi = hi;
      e = cudaStreamCreateWithPriority(&env->side, cudaStreamNonBlocking, hi);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&env->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&env->ev_join, cudaEventDisableTiming);
  }
  if (e == cudaSuccess) {
    vine_init_kernel<<<grid_for(num_envs, 256), 256>>>(env->p, env->a);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    snprintf(g_create_err, 256, "vine_create: %s", cudaGetErrorString(e));
    vine_destroy(env);
    return VINE_ERR_CUDA;
  }
  *out = env;
  return VINE_OK;
}

int vine_bind_io(VineEnv* env, const float* actions, float* obs_buf, float* rew_buf, int64_t* reset_buf,
                 int64_t* progress_buf, uint8_t* timeout_buf, float* obs_clamped) {
  if (!env) return VINE_ERR_INVALID_ARG;
  if (!actions || !obs_buf || !rew_buf || !reset_buf || !progress_buf || !timeout_buf) {
    snprintf(env->err, 256, "vine_bind_io: null buffer"); return VINE_ERR_INVALID_ARG;
  }
  if (((uintptr_t)actions | (uintptr_t)obs_buf | (uintptr_t)obs_clamped) & 15u) {
    snprintf(env->err, 256, "vine_bind_io: actions/obs buffers must be 16-byte aligned"); return VINE_ERR_INVALID_ARG;
  }
  env->a.actions = reinterpret_cast<const float2*>(actions);
  env->a.obs = obs_buf; env->a.obs_clamped = obs_clamped; env->a.rew = rew_buf;
  env->a.reset = reset_buf; env->a.progress = progress_buf; env->a.timeout = timeout_buf;
  env->bound = 1;
  return VINE_OK;
}

int vine_set_debug_outputs(VineEnv* env, int enabled) {
  if (!env) return VINE_ERR_INVALID_ARG;
  if (enabled && !env->a.dbg) {
    CUDA_TRY(env, cudaSetDevice(env->device));
    CUDA_TRY(env, cudaMalloc(&env->a.dbg, (size_t)env->a.n * VINE_DBG_W * sizeof(float)));
    CUDA_TRY(env, cudaMemset(env->a.dbg, 0, (size_t)env->a.n * VINE_DBG_W * sizeof(float)));
  } else if (!enabled && env->a.dbg) {
    CUDA_TRY(env, cudaFree(env->a.dbg));
    env->a.dbg = nullptr;
  }
  return VINE_OK;
}

// ------------------------------------------------------------------------------------------
// Metrics of the reference's per-step wandb dict (V5:1250-1322) as ONE reduction launch over the
// debug plane + state planes (the reference issues ~100 `.item()` syncs per step for the same numbers).
// sums f64[VINE_METRIC_SUMS], maxes f32[VINE_METRIC_MAXES]; layouts: include/vine_b200.h.
// ------------------------------------------------------------------------------------------
#define MS_SCALARS 16
#define MS_NSUM (MS_SCALARS + 2 * VINE_NUM_REWARDS + 1 + 2)      /* = VINE_METRIC_SUMS */
#define MS_NMAX (3 + 2 * VINE_NUM_REWARDS + 1)                   /* = VINE_METRIC_MAXES */
static_assert(MS_NSUM == VINE_METRIC_SUMS && MS_NMAX == VINE_METRIC_MAXES, "metric layout");

__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  v = __fadd_rn(v, 0.f);   // -0.0 -> +0.0 (its bit pattern would order below every negative number)
  if (v >= 0.f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__global__ void vine_metrics_init_kernel(double* sums, float* maxes) {
  const int i = threadIdx.x;
  if (i < MS_NSUM) sums[i] = 0.0;
  if (i < MS_NMAX) maxes[i] = __int_as_float(0xff800000);   // -inf
}

__global__ void __launch_bounds__(256) vine_metrics_kernel(const __grid_constant__ VineParams p, const StepArgs a, double* sums,
                                                           float* maxes) {
  float s[MS_NSUM], m[MS_NMAX];
#pragma unroll
  for (int i = 0; i < MS_NSUM; ++i) s[i] = 0.f;
#pragma unroll
  for (int i = 0; i < MS_NMAX; ++i) m[i] = __int_as_float(0xff800000);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < a.n; e += (int64_t)gridDim.x * blockDim.x) {
    const float* d = a.dbg + e * VINE_DBG_W;
    const float4 s3 = a.S3[e], s4 = a.S4[e];
    const float* r = d + 6;
    const float tipvel = sqrtf(d[4] * d[4] + d[5] * d[5]);
    const float v[MS_SCALARS] = {
        -r[0],                                  // dist_tip_to_target (Position reward = -dist, V5:1480)
        r[2] != 0.f ? 1.f : 0.f,                // target_reached
        r[9] != 0.f ? 1.f : 0.f,                // limit_hit
        r[11] != 0.f ? 1.f : 0.f,               // tip_limit_hit
        fabsf(s4.x), s4.y,                      // abs_tip_y, tip_z (rigid-body view)
        tipvel,                                 // tip_velocities
        fabsf(d[0]), fabsf(d[2]), fabsf(d[3]),  // u_rail_velocity, prev_u_rail_velocity, rail_force
        fabsf(d[1]), fabsf(s3.x),               // u_fpam, smoothed_u_fpam
        tipvel,                                 // tip_target_velocity_difference (target velocity == 0, V5:916-918)
        (float)a.progress[e],                   // progress_buf
        -r[12],                                 // contact_forces (Contact Force reward = -contact [contact > 0])
        r[12] != 0.f ? 1.f : 0.f};              // nonzero_contact_force
#pragma unroll
    for (int i = 0; i < MS_SCALARS; ++i) s[i] += v[i];
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < VINE_NUM_REWARDS; ++i) {
      const float wr = r[i] * p.w[i];
      s[MS_SCALARS + i] += r[i];
      s[MS_SCALARS + VINE_NUM_REWARDS + i] += wr;
      m[3 + i] = fmaxf(m[3 + i], r[i]);
      m[3 + VINE_NUM_REWARDS + i] = fmaxf(m[3 + VINE_NUM_REWARDS + i], wr);
    }
    tot = a.rew[e];
    s[MS_SCALARS + 2 * VINE_NUM_REWARDS] += tot;
    s[MS_SCALARS + 2 * VINE_NUM_REWARDS + 1] += s4.w;            // aggregated reward
    s[MS_SCALARS + 2 * VINE_NUM_REWARDS + 2] += s4.w * s4.w;
    m[0] = fmaxf(m[0], fabsf(s4.x)); m[1] = fmaxf(m[1], s4.y); m[2] = fmaxf(m[2], tipvel);
    m[3 + 2 * VINE_NUM_REWARDS] = fmaxf(m[3 + 2 * VINE_NUM_REWARDS], tot);
  }
  __shared__ double rs[8][MS_NSUM];
  __shared__ float rm[8][MS_NMAX];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < MS_NSUM; ++i) {
    double t = (double)s[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) rs[warp][i] = t;
  }
#pragma unroll
  for (int i = 0; i < MS_NMAX; ++i) {
    float t = m[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = fmaxf(t, __shfl_xor_sync(0xffffffffu, t, o));
    if (lane == 0) rm[warp][i] = t;
  }
  __syncthreads();
  if (threadIdx.x < MS_NSUM) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += rs[w][threadIdx.x];
    atomicAdd(sums + threadIdx.x, t);
  }
  if (threadIdx.x < MS_NMAX) {
    float t = rm[0][threadIdx.x];
    for (int w = 1; w < 8; ++w) t = fmaxf(t, rm[w][threadIdx.x]);
    atomic_max_float(maxes + threadIdx.x, t);
  }
}

int vine_metrics(VineEnv* env, double* sums, float* maxes, void* stream) {
  if (!env || !sums || !maxes) return VINE_ERR_INVALID_ARG;
  if (!env->bound) { snprintf(env->err, 256, "vine_metrics: call vine_bind_io first"); return VINE_ERR_NOT_BOUND; }
  if (!env->a.dbg) { snprintf(env->err, 256, "vine_metrics: enable vine_set_debug_outputs first"); return VINE_ERR_INVALID_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  vine_metrics_init_kernel<<<1, 64, 0, st>>>(sums, maxes);
  int64_t blocks = (env->a.n + 255) / 256;
  if (blocks > 592) blocks = 592;
  vine_metrics_kernel<<<(unsigned)blocks, 256, 0, st>>>(env->p, env->a, sums, maxes);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

// free space: one env per thread (AUTO: as fast at 1 M envs and 1.5x faster at 4096, see DESIGN.md) unless the config asks for
// the packed two-envs-per-thread kernel
static void launch_free_step(const VineEnv* env, const StepArgs& a, cudaStream_t st) {
  const int64_t count = a.end - a.first;
  if (env->cfg.step_kernel_variant == VINE_STEP_KERNEL_TWO_ENVS_PACKED)
    vine_step2_kernel<<<grid_for(count, 2 * VINE_BLOCK2), VINE_BLOCK2, 0, st>>>(env->p, a);
  else
    vine_launch::launch(vine_step_kernel<false>, grid_for(count, VINE_BLOCK), VINE_BLOCK, 0, st, env->p, a);
}

// Routed step of the obstacle variants (contact_binning != 0), per control step:
//   1. vine_bin_kernel          orders the envs: "near" (chain box overlapped the obstacles' box in the last step) first, the
//                               rest from the back; the near count stays on the device
//   2. vine_step_kernel<true>   over the near list, on the side stream           } concurrently: the near pass is a handful
//      vine_step_far_kernel     over the rest (free-space integrator + gap bound)  } of latency-bound warps
//   3. vine_step_kernel<true>   over the envs the far pass gave up (boxes came to overlap during this step)
// Per-env results do not depend on the routing (see vine_step_far_kernel).  contact_binning: 0 = one contact-variant launch
// over all envs in identity order, 1 = routed from VINE_ROUTE_MIN_ENVS envs (measured crossover on B200: 131,072 envs 0.37 vs
// 0.42 ms, 262,144 envs 0.63 vs 0.49 ms; below it the step is bounded by its slowest warp either way and the routed step pays
// that latency twice, near pass + redo pass), 2 = always routed.
#define VINE_ROUTE_MIN_ENVS 196608

static unsigned listed_grid(int64_t n, int max_blocks) {
  const int64_t b = (n + VINE_BLOCK_CONTACT - 1) / VINE_BLOCK_CONTACT;
  return (unsigned)(b < max_blocks ? b : max_blocks);
}

int vine_step(VineEnv* env, void* stream) {
  if (!env) return VINE_ERR_INVALID_ARG;
  if (!env->bound) { snprintf(env->err, 256, "vine_step: call vine_bind_io first"); return VINE_ERR_NOT_BOUND; }
  cudaStream_t st = (cudaStream_t)stream;
  if (env->p.shelf || env->p.pipe) {
    StepArgs a = env->a;
    const bool routed = a.perm && (env->cfg.contact_binning >= 2 || a.n >= VINE_ROUTE_MIN_ENVS);
    if (routed) {
      CUDA_TRY(env, cudaMemsetAsync(a.bin_cursor, 0, 4 * sizeof(int32_t), st));
      vine_bin_kernel<<<grid_for(a.n, 1024), 1024, 0, st>>>(a);
      CUDA_TRY(env, cudaEventRecord(env->ev_fork, st));
      CUDA_TRY(env, cudaStreamWaitEvent(env->side, env->ev_fork, 0));
      StepArgs nr = a;
      nr.list = a.perm; nr.list_count = a.bin_cursor; nr.list_reversed = 0;
      {   // the priority travels as a launch attribute too: a captured graph keeps it on the kernel node (a stream's priority alone
          // is not recorded, and without it the far pass's blocks are placed first and the near pass starts when they drain)
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(listed_grid(a.n, 148 * 12)); lc.blockDim = dim3(VINE_BLOCK_CONTACT); lc.stream = env->side;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributePriority; at[0].val.priority = env->prio_hi;
        lc.attrs = at; lc.numAttrs = 1;
        CUDA_TRY(env, cudaLaunchKernelEx(&lc, vine_step_kernel<true>, env->p, nr));
      }
      CUDA_TRY(env, cudaEventRecord(env->ev_join, env->side));
      StepArgs fr = a;
      fr.list = a.perm; fr.list_count = a.bin_cursor; fr.list_reversed = 1;
      fr.redo_list = a.redo_list; fr.redo_count = a.bin_cursor + 2;
      vine_step_far_kernel<<<grid_for(a.n, VINE_BLOCK), VINE_BLOCK, 0, st>>>(env->p, fr);
      CUDA_TRY(env, cudaStreamWaitEvent(st, env->ev_join, 0));
      StepArgs rd = a;
      rd.list = a.redo_list; rd.list_count = a.bin_cursor + 2; rd.list_reversed = 0;
      vine_step_kernel<true><<<listed_grid(a.n, 148 * 6), VINE_BLOCK_CONTACT, 0, st>>>(env->p, rd);
    } else {
      a.perm = nullptr;
      vine_launch::launch(vine_step_kernel<true>, grid_for(a.n, VINE_BLOCK_CONTACT), VINE_BLOCK_CONTACT, 0, st, env->p, a);
    }
  } else {
    launch_free_step(env, env->a, st);
  }
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

// counts of the last routed step: near and far envs as binned, and how many the far pass gave up (synchronises)
int vine_route_counts(VineEnv* env, int64_t out[4]) {
  if (!env || !out) return VINE_ERR_INVALID_ARG;
  out[0] = out[1] = out[2] = out[3] = 0;
  if (!env->a.bin_cursor) return VINE_OK;
  int32_t c[4];
  CUDA_TRY(env, cudaDeviceSynchronize());
  CUDA_TRY(env, cudaMemcpy(c, env->a.bin_cursor, sizeof(c), cudaMemcpyDeviceToHost));
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2];
  return VINE_OK;
}

int vine_step_range(VineEnv* env, int64_t first, int64_t count, void* stream) {
  if (!env) return VINE_ERR_INVALID_ARG;
  if (!env->bound) { snprintf(env->err, 256, "vine_step_range: call vine_bind_io first"); return VINE_ERR_NOT_BOUND; }
  if (first < 0 || count <= 0 || first + count > env->a.n || (first % VINE_BLOCK) != 0) {
    snprintf(env->err, 256, "vine_step_range: need 0 <= first, first %% %d == 0, first + count <= num_envs", VINE_BLOCK);
    return VINE_ERR_INVALID_ARG;
  }
  StepArgs a = env->a;
  a.first = first; a.end = first + count;
  a.perm = nullptr;   // chunked launches keep the identity order (the near flags are still maintained)
  if (env->p.shelf || env->p.pipe) vine_step_kernel<true><<<grid_for(count, VINE_BLOCK_CONTACT), VINE_BLOCK_CONTACT, 0, (cudaStream_t)stream>>>(env->p, a);
  else launch_free_step(env, a, (cudaStream_t)stream);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_reset_idx(VineEnv* env, const int64_t* env_ids, int64_t n, void* stream) {
  if (!env || (n > 0 && !env_ids) || n < 0) return VINE_ERR_INVALID_ARG;
  if (n == 0) return VINE_OK;
  vine_reset_idx_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(env->p, env->a, env_ids, n);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_get_state(VineEnv* env, const VineStateView* view, void* stream) {
  if (!env || !view) return VINE_ERR_INVALID_ARG;
  vine_state_kernel<<<grid_for(env->a.n, 256), 256, 0, (cudaStream_t)stream>>>(env->p, env->a, *view, 0);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_set_state(VineEnv* env, const VineStateView* view, void* stream) {
  if (!env || !view) return VINE_ERR_INVALID_ARG;
  vine_state_kernel<<<grid_for(env->a.n, 256), 256, 0, (cudaStream_t)stream>>>(env->p, env->a, *view, 1);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_post_physics(VineEnv* env, const VinePostPhysicsIO* io, void* stream) {
  if (!env || !io) return VINE_ERR_INVALID_ARG;
  vine_post_physics_kernel<<<grid_for(env->a.n, 128), 128, 0, (cudaStream_t)stream>>>(env->p, env->a.n, *io);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_pre_physics(VineEnv* env, const VinePrePhysicsIO* io, void* stream) {
  if (!env || !io) return VINE_ERR_INVALID_ARG;
  vine_pre_physics_kernel<<<grid_for(env->a.n, 128), 128, 0, (cudaStream_t)stream>>>(env->p, env->a.n, *io);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_actuation(VineEnv* env, const VineActuationIO* io, void* stream) {
  if (!env || !io) return VINE_ERR_INVALID_ARG;
  vine_actuation_kernel<<<grid_for(env->a.n, 128), 128, 0, (cudaStream_t)stream>>>(env->p, env->a.n, *io);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_simulate(VineEnv* env, const VineSimulateIO* io, void* stream) {
  if (!env || !io) return VINE_ERR_INVALID_ARG;
  const unsigned grid = grid_for(env->a.n, VINE_BLOCK);
  if (env->p.shelf || env->p.pipe) vine_simulate_kernel<true><<<grid, VINE_BLOCK, 0, (cudaStream_t)stream>>>(env->p, env->a.n, *io);
  else vine_simulate_kernel<false><<<grid, VINE_BLOCK, 0, (cudaStream_t)stream>>>(env->p, env->a.n, *io);
  CUDA_TRY(env, cudaGetLastError());
  return VINE_OK;
}

int vine_philox_debug(uint64_t seed, uint32_t gid, uint32_t site, uint32_t step, uint32_t block0, int64_t n_blocks,
                      uint32_t* out, void* stream) {
  if (!out || n_blocks <= 0) return VINE_ERR_INVALID_ARG;
  vine_philox_kernel<<<grid_for(n_blocks, 128), 128, 0, (cudaStream_t)stream>>>((uint32_t)seed, (uint32_t)(seed >> 32), gid, site,
                                                                                 step, block0, n_blocks, out);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

int vine_gae(const float* rewards, const float* values, const float* dones, const float* last_values,
             const float* last_dones, int64_t horizon, int64_t num_envs, double gamma, double tau, float* advantages,
             float* returns, void* stream) {
  if (!rewards || !values || !dones || !last_values || !last_dones || !advantages || !returns || horizon <= 0 || num_envs <= 0)
    return VINE_ERR_INVALID_ARG;
  // Python: `self.gamma * self.tau` is a double product that meets the f32 tensor afterwards
  vine_gae_kernel<<<grid_for(num_envs, 128), 128, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, last_dones,
                                                                             horizon, num_envs, (float)gamma, (float)(gamma * tau),
                                                                             advantages, returns);
  return cudaGetLastError() == cudaSuccess ? VINE_OK : VINE_ERR_CUDA;
}

}  // extern "C"
