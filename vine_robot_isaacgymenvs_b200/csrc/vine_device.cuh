// vine_device.cuh — per-environment device functions of the Vine5LinkMovingBase step.
// One environment per thread; everything below works on registers.
//
// Rounding discipline: the task logic the reference computes with torch f32 kernels (action
// path, controller, observations, reward, resets) is written with explicit __f*_rn intrinsics in
// the reference's operation order so nvcc cannot contract it into FMAs — masks stay bit-exact.
// The dynamics (PhysX in the reference, parity unpinned) uses free-form FMA arithmetic.
#pragma once
#include <cuda_runtime.h>

#include "vine_params.h"

#define VDEV __device__ __forceinline__

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11). ctr = (gid, site, step, block), key = seed.
// ------------------------------------------------------------------------------------------
VDEV uint4 philox4x32(uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

// 1/x as one MUFU.RCP (__fdividef(1, x) adds a range check and a scaling multiply per call; the pivots of the SPD system
// matrix and squared edge lengths are far inside the normal range)
VDEV float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// sin/cos as MUFU.SIN / MUFU.COS on the XU pipe behind one shared FMUL by 1/(2 pi), whatever the compiler flags (absolute
// error <= 2^-20.5 for |x| <= 100 pi, PTX ISA)
VDEV float sin_approx(float x) { float r; asm("sin.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
VDEV float cos_approx(float x) { float r; asm("cos.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// IEEE a / b (round to nearest) for the task logic that must match torch bit for bit. div.rn's fast path (FCHK) sends the whole
// warp through a ~50-instruction subroutine whenever one lane's numerator is zero, and the observation row is full of exact
// zeros (x components, depth and angle without an obstacle): ncu showed 20 such calls per warp and step, 17 % of the stall
// samples. 0 / b = 0 with the sign of a xor b for every finite non-zero b, so those lanes divide 1 by b and select.
VDEV float div_rn(float a, float b) {
  const bool bypass = a == 0.f && fabsf(b) > 0.f && fabsf(b) < __int_as_float(0x7f800000);
  const float q = __fdiv_rn(bypass ? 1.f : a, b);
  return bypass ? __int_as_float(__float_as_int(a) ^ (__float_as_int(b) & (int)0x80000000)) : q;
}
VDEV float u01(uint32_t x) { return __fmul_rn((float)(x >> 8), 5.9604644775390625e-08f); }  // [0,1)
VDEV float uniform_ab(uint32_t x, float lo, float rng) { return __fmaf_rn(u01(x), rng, lo); }
// 16-bit draw h in [0, 65536) -> lo + (h 2^-16) rng with rng16 = rng * 2^-16 (the power-of-two scaling of either factor
// leaves the exact product, hence the fused result, unchanged)
VDEV float uniform_ab16(uint32_t h, float lo, float rng16) { return __fmaf_rn((float)h, rng16, lo); }

// sin/cos for |x| up to a few thousand (Cody-Waite reduction + Cephes minimax kernels)
VDEV void vine_sincos(float x, float& s, float& c) {
  const float j = rintf(x * 0.636619772f);
  const int q = (int)j;
  float r = fmaf(j, -1.57079601e+00f, x);
  r = fmaf(j, -3.13916473e-07f, r);
  r = fmaf(j, -5.39030253e-15f, r);
  const float r2 = r * r;
  const float sp = fmaf(fmaf(fmaf(-1.9515295891e-4f, r2, 8.3321608736e-3f), r2, -1.6666654611e-1f), r2 * r, r);
  const float cp = fmaf(fmaf(fmaf(2.443315711809948e-5f, r2, -1.388731625493765e-3f), r2, 4.166664568298827e-2f),
                        r2 * r2, fmaf(-0.5f, r2, 1.0f));
  const float a = (q & 1) ? cp : sp, b = (q & 1) ? sp : cp;
  s = (q & 2) ? -a : a;
  c = ((q + 1) & 2) ? -b : b;
}

// Box-Muller: 4 u32 -> 4 standard normals
VDEV void normal4(uint4 r, float out[4]) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int p = 0; p < 2; ++p) {
    const float u1 = __fmul_rn((float)((w[2 * p] >> 8) + 1u), 5.9604644775390625e-08f);  // (0,1]
    const float u2 = u01(w[2 * p + 1]);
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    vine_sincos(6.283185307179586f * u2, sn, cs);
    out[2 * p] = rad * cs; out[2 * p + 1] = rad * sn;
  }
}

// ------------------------------------------------------------------------------------------
// Action path: raw_actions_to_actions V5:984-997, rescale_to_u V5:1458-1459,
// manual_intervention V5:1023-1026, u_fpam_to_smoothed_u_fpam V5:999-1005.
// `old_*` is the command popped from the delay ring (== new when ACTION_DELAY = 0).
// ------------------------------------------------------------------------------------------
VDEV void rescale_actions(const VineParams& p, float a0, float a1, float& new_rail, float& new_fpam) {
  new_rail = __fmul_rn(a0, p.rail_scale);
  new_fpam = __fadd_rn(__fmul_rn(__fmul_rn(__fadd_rn(a1, 1.0f), 0.5f), p.fpam_range), p.fpam_min);   // x / 2 == x * 0.5 exactly
}

VDEV void apply_overrides_and_smooth(const VineParams& p, float& u_rail, float& u_fpam, float& smoothed) {
  if (p.force_fpam) u_fpam = 0.0f;
  if (p.force_rail) u_rail = 0.0f;
  const float alpha = (u_fpam > smoothed) ? p.alpha_inf : p.alpha_def;
  smoothed = __fadd_rn(__fmul_rn(alpha, smoothed), __fmul_rn(__fsub_rn(1.0f, alpha), u_fpam));
}

// ------------------------------------------------------------------------------------------
// compute_and_set_dof_actuation_force_tensor, V5:1028-1106
// ------------------------------------------------------------------------------------------
__constant__ float cTL_K[VINE_NL] = {0.8385f, 1.5400f, 1.5109f, 1.2887f, 0.4347f};  // V5:1045
__constant__ float cTL_C[VINE_NL] = {0.0178f, 0.0304f, 0.0528f, 0.0367f, 0.0223f};  // V5:1046
__constant__ float cTL_b[VINE_NL] = {0.0007f, 0.0062f, 0.0402f, 0.0160f, 0.0133f};  // V5:1047
__constant__ float cTL_B[VINE_NL] = {0.0247f, 0.0616f, 0.0779f, 0.0498f, 0.0268f};  // V5:1048

// scaled torque-law coefficients of one sim step: (K,C,b,B) * U(DYNAMICS_SCALING) (V5:1053-1055)
struct JointLaw { float K[VINE_NL], Cd[VINE_NL], b[VINE_NL], B[VINE_NL]; };

VDEV void joint_law_unscaled(JointLaw& L) {
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) { L.K[j] = cTL_K[j]; L.Cd[j] = cTL_C[j]; L.b[j] = cTL_b[j]; L.B[j] = cTL_B[j]; }
}

VDEV float joint_torque(const JointLaw& L, int j, float q, float qd, float u) {  // -(Kq + Cqd + b + Bu)
  float t = __fmul_rn(L.K[j], q);
  t = __fadd_rn(t, __fmul_rn(L.Cd[j], qd));
  t = __fadd_rn(t, L.b[j]);
  t = __fadd_rn(t, __fmul_rn(L.B[j], u));
  return -t;
}

VDEV float rail_controller(const VineParams& p, float cart_vel_y, float u_rail, float acc_scale,
                           float& prev_cart_vel, float& prev_err) {
  const float err = __fsub_rn(u_rail, cart_vel_y);
  float minmax = (err > 0.0f) ? p.rail_force_max : -p.rail_force_max;
  const float accel = div_rn(__fsub_rn(cart_vel_y, prev_cart_vel), p.dt);          // V5:1079
  float accel_target = (err > 0.0f) ? p.rail_accel : -p.rail_accel;
  accel_target = __fmul_rn(accel_target, acc_scale);                                   // README.md:63 knob
  minmax = __fadd_rn(minmax, __fmul_rn(0.30f, __fsub_rn(accel_target, accel)));       // V5:1083-1087
  const float pid = __fadd_rn(__fmul_rn(p.p_gain, err), __fmul_rn(p.d_gain, __fsub_rn(err, prev_err)));
  prev_err = err; prev_cart_vel = cart_vel_y;                                          // V5:1097-1098
  return (fabsf(err) > 0.1f) ? minmax : pid;                                           // V5:1094
}

// ------------------------------------------------------------------------------------------
// Obstacles: rectangles in the (y,z) plane of motion (custom_shelf.urdf:82-93,139-152 placed by
// V5:818-829; pipe tube V5:841-885 with the STL's dimensions).
// ------------------------------------------------------------------------------------------
// Per-warp shared scratch of the contact variant (dynamic indexing by link / rectangle without local memory):
//   rect:  six floats per rectangle and env: centre (cy, cz), unit axis (ay, az), half extents along the axis (ha) and the
//          normal (hn); fixed for the control step
//   chain: joint positions / velocities, sin/cos and spin of the links of an env with candidate contacts, rewritten by
//          that env's lane in the substeps in which it has any
enum { CH_PY = 0, CH_PZ = 6, CH_VY = 12, CH_VZ = 18, CH_S = 24, CH_C = 29, CH_W = 34, CH_FIELDS = 39 };
#define VINE_PAIR_PASS 64                   // (env, pair) work items the warp's narrow phase takes per pass
struct ContactScratch {
  float rect[32][VINE_MAX_RECTS * 6 + 1];   // [lane][6 r + field]; odd row stride keeps the lanes on different banks
  float chain[CH_FIELDS][32];               // [field][lane]
  float res[VINE_PAIR_PASS][3];             // net force (y, z) and torque about the proximal joint of a work item's pair
  unsigned short item[VINE_PAIR_PASS];      // owner lane | pair bit << 5
};
// rectangle count and index of the sensing shelf_link rectangle (-1: none), the same for all envs; bounding box of this env's
struct Obstacles { int n, lip; float lo_y, hi_y, lo_z, hi_z; };
// candidate (link, rectangle) pairs of one env (bit 5 r + j) and a bound on how far any point of the chain has moved since
// they were culled (negative: distance still to go before the chain can reach the obstacles' bounding box); registers
struct ContactCache { unsigned pm; float disp; unsigned seen; };   // seen: OR of every mask of this control step

// the obstacle rectangles of one env: put(index, centre y, centre z, axis y, axis z, half extent along the axis, along the normal)
template <class Put>
VDEV void for_each_obstacle_rect(const VineParams& p, float ty, float tz, float depth, float theta, int& n, int& lip, Put&& put) {
  n = 0; lip = -1;
  if (p.shelf) {
    const float ry = ty + (-0.2f + depth), rz = tz - 0.01f;
    put(0, ry - 0.001f, rz, 1.f, 0.f, 0.1995f, 0.005f);
    put(1, ry, rz + 0.2f, 1.f, 0.f, 0.2f, 0.005f);
    put(2, ry + 0.199f, rz, 1.f, 0.f, 0.001f, 0.005f);
    lip = 2; n = 3;
  }
  if (p.pipe) {
    float st, ct; vine_sincos(theta, st, ct);
    const float off = 0.0735f - 0.0777f;            // PIPE_RADIUS (V5:88) - mesh centre
    const float win = 0.07232816f, wout = 0.07758640f;  // sqrt(R^2 - off^2) for R_in, R_out
    const float ey = ty + depth * ct + off * st, ez = tz + depth * st - off * ct;
    const float ay = -ct, az = -st, ny = -az, nz = ay;
    const float mid = 0.5f * (win + wout), hn = 0.5f * (wout - win), ha = 0.5f * 0.34125f;
    put(n, ey + ay * ha - mid * ny, ez + az * ha - mid * nz, ay, az, ha, hn);
    put(n + 1, ey + ay * ha + mid * ny, ez + az * ha + mid * nz, ay, az, ha, hn);
    n += 2;
  }
}

VDEV void build_obstacles(const VineParams& p, float ty, float tz, float depth, float theta, ContactScratch* cs, Obstacles& ob) {
  float* R = cs->rect[threadIdx.x & 31];
  ob.lo_y = ob.lo_z = 1e30f; ob.hi_y = ob.hi_z = -1e30f;
  for_each_obstacle_rect(p, ty, tz, depth, theta, ob.n, ob.lip, [&](int i, float cy, float cz, float ay, float az, float ha, float hn) {
    R[6 * i] = cy; R[6 * i + 1] = cz; R[6 * i + 2] = ay; R[6 * i + 3] = az; R[6 * i + 4] = ha; R[6 * i + 5] = hn;
    const float ey = fabsf(ay) * ha + fabsf(az) * hn, ez = fabsf(az) * ha + fabsf(ay) * hn;
    ob.lo_y = fminf(ob.lo_y, cy - ey); ob.hi_y = fmaxf(ob.hi_y, cy + ey);
    ob.lo_z = fminf(ob.lo_z, cz - ez); ob.hi_z = fmaxf(ob.hi_z, cz + ez);
  });
}

// bounding box of the obstacles only (the far pass of the obstacle variants keeps nothing else)
VDEV void obstacle_bbox(const VineParams& p, float ty, float tz, float depth, float theta, Obstacles& ob) {
  ob.lo_y = ob.lo_z = 1e30f; ob.hi_y = ob.hi_z = -1e30f;
  for_each_obstacle_rect(p, ty, tz, depth, theta, ob.n, ob.lip, [&](int, float cy, float cz, float ay, float az, float ha, float hn) {
    const float ey = fabsf(ay) * ha + fabsf(az) * hn, ez = fabsf(az) * ha + fabsf(ay) * hn;
    ob.lo_y = fminf(ob.lo_y, cy - ey); ob.hi_y = fmaxf(ob.hi_y, cy + ey);
    ob.lo_z = fminf(ob.lo_z, cz - ez); ob.hi_z = fmaxf(ob.hi_z, cz + ez);
  });
}

// ------------------------------------------------------------------------------------------
// Dynamics state in absolute coordinates: x = (cart y, phi'_0..4), v = d/dt.
// ------------------------------------------------------------------------------------------
// S/C = sin/cos of the absolute link angles phi_k = 3.1415 + phi'_k, always link_trig of the current x: evaluated by
// rel_to_abs and again after the position update of every substep.
struct Dyn { float x[6], v[6], S[VINE_NL], C[VINE_NL]; };

// sin/cos of the absolute angle 3.1415 + x of one link (URDF:289): one FADD, one FMUL and two MUFU. Every kernel takes S/C
// from here, so they are one function of x whichever kernel integrated it (the routed step equals a single launch).
VDEV void link_trig(float x, float& s, float& c) {
  const float a = __fadd_rn(x, VINE_BASE_ANGLE);
  s = sin_approx(a); c = cos_approx(a);
}

VDEV void rel_to_abs(const float q[6], const float qd[6], Dyn& d) {
  d.x[0] = q[0]; d.v[0] = qd[0];
  float a = 0.f, b = 0.f;
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) { a += q[j + 1]; b += qd[j + 1]; d.x[j + 1] = a; d.v[j + 1] = b; }
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) link_trig(d.x[j + 1], d.S[j], d.C[j]);
}

VDEV void abs_to_rel(const Dyn& d, float q[6], float qd[6]) {
  q[0] = d.x[0]; qd[0] = d.v[0]; q[1] = d.x[1]; qd[1] = d.v[1];
#pragma unroll
  for (int j = 1; j < VINE_NL; ++j) { q[j + 1] = d.x[j + 1] - d.x[j]; qd[j + 1] = d.v[j + 1] - d.v[j]; }
}

// tip position / velocity (the rigid-body views V5:357-362)
VDEV void tip_fk(const Dyn& d, float& ty, float& tz, float& tvy, float& tvz) {
  float py = d.x[0], pz = VINE_PIVOT_Z, vy = d.v[0], vz = 0.f;
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) {
    py = fmaf(-VINE_LINK_LEN, d.S[j], py); pz = fmaf(VINE_LINK_LEN, d.C[j], pz);
    const float lw = VINE_LINK_LEN * d.v[j + 1];
    vy = fmaf(-lw, d.C[j], vy); vz = fmaf(-lw, d.S[j], vz);
  }
  ty = py; tz = pz; tvy = vy; tvz = vz;
}

// ---- penalty contact, frictionless (V5:477,491,499) ----
// Contacts are rare per env but common per warp, and everything an env does about them runs with ~1 of 32 lanes active,
// i.e. at the latency of one dependent instruction chain.  So the chain is kept short: each env carries a conservative
// candidate mask of (link, rectangle) pairs that is re-culled only after the chain has moved p.cull_slack since the
// last cull (a substep without candidates costs 12 instructions), and there is ONE copy of the narrow phase, entered per
// candidate pair with the link picked by a run-time index into shared memory, its 2 capsules x (2 end points + 4 rectangle
// corners) unrolled so the twelve independent point tests overlap.

struct PairLoad { float fy, fz, t; };  // net force and torque about the link's proximal joint of one (link, rectangle) pair

VDEV void contact_point(const VineParams& p, float Py, float Pz, float ny, float nz, float dist, float reach,
                        float jy, float jz, float jvy, float jvz, float w, PairLoad& L) {
  const float pen = reach - dist;
  if (!(pen > 0.f)) return;
  const float ry = Py - jy, rz = Pz - jz;
  const float vy = jvy - w * rz, vz = jvz + w * ry;
  const float f = p.kc * pen - p.dc * (vy * ny + vz * nz);
  if (!(f > 0.f)) return;
  const float Fy = f * ny, Fz = f * nz;
  L.fy += Fy; L.fz += Fz; L.t += ry * Fz - rz * Fy;
}

// capsule (core A-B, radius r) of a link whose proximal joint is at (jy,jz) moving with (jvy,jvz), spin w
VDEV void capsule_rect(const VineParams& p, const float* R, float Ay, float Az, float By, float Bz, float radius,
                       bool test_a, bool closed_end, float jy, float jz, float jvy, float jvz, float w, PairLoad& L) {
  const float cy = R[0], cz = R[1], ay = R[2], az = R[3], ha = R[4], hn = R[5];
  const float ny = -az, nz = ay;
  const float reach = radius + p.rest;
  // separating-axis cull in the rectangle's frame (exact: every distance used below is >= the separation along either
  // rectangle axis, and a contact needs distance < radius + rest)
  const float laA = (Ay - cy) * ay + (Az - cz) * az, lnA = (Ay - cy) * ny + (Az - cz) * nz;
  const float laB = (By - cy) * ay + (Bz - cz) * az, lnB = (By - cy) * ny + (Bz - cz) * nz;
  if (fminf(lnA, lnB) >= hn + reach || fmaxf(lnA, lnB) <= -(hn + reach) || fminf(laA, laB) >= ha + reach ||
      fmaxf(laA, laB) <= -(ha + reach))
    return;
  // (i) capsule end points against the rectangle's faces
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    if (e == 0 && !test_a) continue;
    const float Py = e == 0 ? Ay : By, Pz = e == 0 ? Az : Bz;
    const float la = e == 0 ? laA : laB, ln = e == 0 ? lnA : lnB;
    const float qa = fabsf(la) - ha, qn = fabsf(ln) - hn;
    if (qa > 0.f && qn > 0.f) continue;  // corner region: handled by (ii)
    float dist, gy, gz;
    if (qa > qn) { dist = qa; const float sg = la < 0.f ? -1.f : 1.f; gy = sg * ay; gz = sg * az; }
    else { dist = qn; const float sg = ln < 0.f ? -1.f : 1.f; gy = sg * ny; gz = sg * nz; }
    contact_point(p, Py, Pz, gy, gz, dist, reach, jy, jz, jvy, jvz, w, L);
  }
  // (ii) rectangle corners against the capsule segment
  const float ey = By - Ay, ez = Bz - Az;
  const float inv_ee = rcp_approx(ey * ey + ez * ez);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float sa = (c & 1) ? 1.f : -1.f, sn = (c & 2) ? 1.f : -1.f;
    const float Vy = cy + sa * ha * ay + sn * hn * ny, Vz = cz + sa * ha * az + sn * hn * nz;
    float t = ((Vy - Ay) * ey + (Vz - Az) * ez) * inv_ee;
    t = fminf(fmaxf(t, 0.f), 1.f);
    if (t >= 1.f && !closed_end) continue;  // shared joint point belongs to the next link
    const float Py = Ay + t * ey, Pz = Az + t * ez;
    const float dy = Py - Vy, dz = Pz - Vz;
    const float d2 = dy * dy + dz * dz;
    if (!(d2 > 1e-18f)) continue;
    const float inv = rsqrtf(d2);
    contact_point(p, Py, Pz, dy * inv, dz * inv, d2 * inv, reach, jy, jz, jvy, jvz, w, L);
  }
}

// conservative per-env cull: link j (both capsules + rest offset lie within `reach` of its midpoint) against rectangle r
VDEV unsigned cull_pairs(const VineParams& p, const Obstacles& ob, const float* R, const float py[VINE_NL + 1],
                         const float pz[VINE_NL + 1]) {
  const float reach = 0.09f + p.rest + p.cull_slack;   // sqrt(0.04425^2 + 0.055^2) + 0.0169 = 0.0875 (FPAM side), 0.0824 (main)
  unsigned pm = 0;
#pragma unroll 1
  for (int r = 0; r < ob.n; ++r) {
    const float cy = R[6 * r], cz = R[6 * r + 1], ay = R[6 * r + 2], az = R[6 * r + 3];
    const float ta = R[6 * r + 4] + reach, tn = R[6 * r + 5] + reach;
    unsigned bits = 0;
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) {
      const float dy = 0.5f * (py[j] + py[j + 1]) - cy, dz = 0.5f * (pz[j] + pz[j + 1]) - cz;
      if (!(fabsf(dy * ay + dz * az) > ta || fabsf(dz * ay - dy * az) > tn)) bits |= 1u << j;
    }
    pm |= bits << (5 * r);
  }
  return pm;
}

// every point of the chain moved at most h (|v_y| + rho sum |w|) in the last substep (rho: farthest point from a joint)
VDEV float chain_displacement_bound(const VineParams& p, const Dyn& d) {
  float ws = 0.f;
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) ws += fabsf(d.v[j + 1]);
  return p.h * fmaf(VINE_LINK_LEN + 0.1f, ws, fabsf(d.v[0]));
}

// Chain inflated by the widest cross-section (FPAM offset + radius) + rest + slack against the obstacles' bounding box: with a
// gap > 0 between the two no contact is possible until some point of the chain has moved `gap`.
VDEV float chain_obstacle_gap(const VineParams& p, const Obstacles& ob, const float py[VINE_NL + 1], const float pz[VINE_NL + 1]) {
  float lo_y = py[0], hi_y = py[0], lo_z = pz[0], hi_z = pz[0];
#pragma unroll
  for (int j = 1; j <= VINE_NL; ++j) {
    lo_y = fminf(lo_y, py[j]); hi_y = fmaxf(hi_y, py[j]); lo_z = fminf(lo_z, pz[j]); hi_z = fmaxf(hi_z, pz[j]);
  }
  const float m = VINE_FPAM_OFFSET + VINE_FPAM_RADIUS + p.rest + 1e-3f + p.cull_slack;
  return fmaxf(fmaxf(lo_y - m - ob.hi_y, ob.lo_y - (hi_y + m)), fmaxf(lo_z - m - ob.hi_z, ob.lo_z - (hi_z + m)));
}

VDEV float chain_obstacle_gap(const VineParams& p, const Obstacles& ob, const Dyn& d) {
  float py[VINE_NL + 1], pz[VINE_NL + 1];
  py[0] = d.x[0]; pz[0] = VINE_PIVOT_Z;
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) {
    py[j + 1] = fmaf(-VINE_LINK_LEN, d.S[j], py[j]); pz[j + 1] = fmaf(VINE_LINK_LEN, d.C[j], pz[j]);
  }
  return chain_obstacle_gap(p, ob, py, pz);
}

// net load of one candidate (link j, rectangle r) pair of the env published in column `owner` of the warp's scratch
VDEV void pair_load(const VineParams& p, const ContactScratch* cs, int owner, int b, PairLoad& L) {
  const int r = b / 5, j = b - 5 * r;
  const float* R = cs->rect[owner] + 6 * r;
  const float* ch = &cs->chain[j][owner];
  const float jy = ch[32 * CH_PY], jz = ch[32 * CH_PZ], ty = ch[32 * (CH_PY + 1)], tz = ch[32 * (CH_PZ + 1)];
  const float jvy = ch[32 * CH_VY], jvz = ch[32 * CH_VZ], S = ch[32 * CH_S], C = ch[32 * CH_C], w = ch[32 * CH_W];
  const bool last = j == VINE_NL - 1;
  L.fy = 0.f; L.fz = 0.f; L.t = 0.f;
  // main cylinder URDF:95-99 as a capsule; the last link's capsules are shortened so that their caps end at the tip
  capsule_rect(p, R, jy, jz, last ? fmaf(VINE_LINK_RADIUS, S, ty) : ty, last ? fmaf(-VINE_LINK_RADIUS, C, tz) : tz,
               VINE_LINK_RADIUS, j == 0, last, jy, jz, jvy, jvz, w, L);
  // FPAM cylinder URDF:110-114, offset along the link's local +y = (cos phi, sin phi)
  const float oy = VINE_FPAM_OFFSET * C, oz = VINE_FPAM_OFFSET * S;
  capsule_rect(p, R, jy + oy, jz + oz, ty + oy + (last ? VINE_FPAM_RADIUS * S : 0.f),
               tz + oz - (last ? VINE_FPAM_RADIUS * C : 0.f), VINE_FPAM_RADIUS, true, true, jy, jz, jvy, jvz, w, L);
}

// All link-vs-obstacle contacts of one substep; adds generalized forces to f[6], returns |F_lip|.
// Called by ALL 32 lanes of the warp together (`ghost` lanes carry no env of their own: tail lanes and, in short listed
// launches, lanes 8..31).  The candidate pairs of the warp's envs are pooled into one work list and dealt out to the 32
// lanes, so a warp does ceil(total pairs / 32) narrow-phase turns instead of max-over-lanes(pairs of one env) with most lanes
// idle.  Every pair is evaluated by the same instruction sequence on the same published values whichever lane runs it, and each
// env adds its pairs' loads in ascending pair order, so the result does not depend on who shares the warp.
VDEV float contact_forces(const VineParams& p, const Obstacles& ob, ContactScratch* cs, ContactCache& cc, const Dyn& d, float f[6],
                          bool ghost) {
  const int lane = threadIdx.x & 31;
  if (!ghost) cc.disp += chain_displacement_bound(p, d);
  const bool stale = !ghost && !(cc.disp <= p.cull_slack);
  float py[VINE_NL + 1], pz[VINE_NL + 1];
  if (stale || cc.pm != 0u) {     // joint positions: for the cull, the published chain and the lever arms of the pairs' loads
    py[0] = d.x[0]; pz[0] = VINE_PIVOT_Z;
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) {
      py[j + 1] = fmaf(-VINE_LINK_LEN, d.S[j], py[j]); pz[j + 1] = fmaf(VINE_LINK_LEN, d.C[j], pz[j]);
    }
  }
  if (stale) {
    const float gap = chain_obstacle_gap(p, ob, py, pz);
    if (gap > 0.f) { cc.pm = 0u; cc.disp = -gap; }
    else { cc.pm = cull_pairs(p, ob, cs->rect[lane], py, pz); cc.disp = 0.f; cc.seen |= cc.pm | 0x80000000u; }   // bit 31: the boxes overlapped
  }
  const unsigned pm = ghost ? 0u : cc.pm;
  if (__ballot_sync(0xffffffffu, pm != 0u) == 0u) return 0.f;   // nobody in the warp has a candidate pair (uniform)
  if (pm) {   // publish this env's chain in its column of the warp's scratch: a pair's link is picked by a run-time index
    float* ch = &cs->chain[0][lane];
    float vy = d.v[0], vz = 0.f;
    ch[32 * CH_PY] = py[0]; ch[32 * CH_PZ] = pz[0]; ch[32 * CH_VY] = vy; ch[32 * CH_VZ] = vz;
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) {
      const float lw = VINE_LINK_LEN * d.v[j + 1];
      vy = fmaf(-lw, d.C[j], vy); vz = fmaf(-lw, d.S[j], vz);
      ch[32 * (CH_PY + j + 1)] = py[j + 1]; ch[32 * (CH_PZ + j + 1)] = pz[j + 1];
      ch[32 * (CH_VY + j + 1)] = vy; ch[32 * (CH_VZ + j + 1)] = vz;
      ch[32 * (CH_S + j)] = d.S[j]; ch[32 * (CH_C + j)] = d.C[j]; ch[32 * (CH_W + j)] = d.v[j + 1];
    }
  }
  // positions of the lanes' pairs in the warp's work list: exclusive prefix sum of the pair counts (< 32 each), bit plane by
  // bit plane with five independent ballots instead of a five-step shuffle scan (a dependent chain of ~150 cycles)
  const int cnt = __popc(pm);
  const unsigned below = (1u << lane) - 1u;
  int next = 0, total = 0;        // next: index of this env's next pair that has not been dealt out / added yet
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    const unsigned plane = __ballot_sync(0xffffffffu, (cnt >> k) & 1);
    next += __popc(plane & below) << k;
    total += __popc(plane) << k;
  }
  unsigned todo = pm, toadd = pm;
  int next_add = next;
  float lfy = 0.f, lfz = 0.f;
#pragma unroll 1
  for (int base = 0; base < total; base += VINE_PAIR_PASS) {
    while (todo && next < base + VINE_PAIR_PASS) {          // this env's pairs that fall into this pass
      const int b = __ffs(todo) - 1;
      todo &= todo - 1;
      cs->item[next - base] = (unsigned short)(lane | (b << 5));
      ++next;
    }
    __syncwarp();
    const int n_pass = min(VINE_PAIR_PASS, total - base);
#pragma unroll 1
    for (int i = lane; i < n_pass; i += 32) {               // the narrow phase, one pair per lane and turn
      const int it = cs->item[i];
      PairLoad L;
      pair_load(p, cs, it & 31, it >> 5, L);
      cs->res[i][0] = L.fy; cs->res[i][1] = L.fz; cs->res[i][2] = L.t;
    }
    __syncwarp();
    while (toadd && next_add < base + VINE_PAIR_PASS) {     // each env adds its own pairs' loads, in ascending pair order
      const int b = __ffs(toadd) - 1;
      toadd &= toadd - 1;
      const float* rs = cs->res[next_add - base];
      ++next_add;
      const float Lfy = rs[0], Lfz = rs[1], Lt = rs[2];
      if (Lfy != 0.f || Lfz != 0.f) {
        const int r = b / 5, j = b - 5 * r;
        // generalized forces: Q_y = F;  Q_j = T_j;  Q_m = (p_{m+1} - p_m) x F for the links m < j below the contact
        f[0] += Lfy;
#pragma unroll
        for (int m = 0; m < VINE_NL; ++m) {
          const float q = m == j ? Lt : (py[m + 1] - py[m]) * Lfz - (pz[m + 1] - pz[m]) * Lfy;
          if (m <= j) f[m + 1] += q;
        }
        if (r == ob.lip) { lfy -= Lfy; lfz -= Lfz; }
      }
    }
    __syncwarp();
  }
  // |F_lip| is zero in almost every substep, and sqrt's zero argument sends the warp through its slow-path subroutine
  const float l2 = lfy * lfy + lfz * lfz;
  const float l = sqrtf(l2 > 0.f ? l2 : 1.f);
  return l2 > 0.f ? l : 0.f;
}

// per-sim-step joint constants for the implicit integrator:
//   t_j = tc_j - kk_j theta_j - ek_j thetadot_j  (ek = dd + h kk),  gam_j = h dd_j + h^2 kk_j + armature,
//   diag_j = alpha_j + gam_j + gam_{j+1} (constant part of the system matrix diagonal)
struct JointImp { float kk[VINE_NL], ek[VINE_NL], tc[VINE_NL], gam[VINE_NL], diag[VINE_NL]; };

VDEV void joint_implicit_consts(const VineParams& p, const JointLaw& law, float u_use, const float efforts[6], JointImp& J) {
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) {
    float dd;
    if (p.implicit_law) {
      J.kk[j] = p.stiffness + law.K[j]; dd = p.damping + law.Cd[j];
      J.tc[j] = -fmaf(law.B[j], u_use, law.b[j]);
    } else {
      J.kk[j] = p.stiffness; dd = p.damping; J.tc[j] = efforts[j + 1];
    }
    J.ek[j] = fmaf(p.h, J.kk[j], dd);
    J.gam[j] = fmaf(p.h, dd, p.h * p.h * J.kk[j]) + p.armature;
  }
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) J.diag[j] = p.alpha[j] + J.gam[j] + (j + 1 < VINE_NL ? J.gam[j + 1] : 0.f);
}

// One substep of the semi-implicit integrator (equations of motion: DESIGN.md §4):
//   (A + h D + h^2 K + armature) dv = h [ f - D v - K (x - x0) - h K v ],  v += dv,  x += h v
// Velocity-product terms in O(n): with a_m = C_m w_m^2, b_m = S_m w_m^2,
//   P_j = sum_{m>j} L beta_m a_m + L beta_j sum_{m<j} a_m  (Q_j likewise with b):
//   f_j = S_j (g beta_j - P_j) + C_j Q_j ,   f_y = F - D v_y - (1/L) sum_m L beta_m b_m
// m00inv = 1 / (M_tot + h D), the reciprocal pivot of the cart row of the system matrix: the same for every env and substep.
// Every operation is an explicit round-to-nearest intrinsic, which nvcc can neither contract nor re-associate: the far pass
// and the contact variant therefore compute the same bits for an env without contact, and the routing changes no result.
template <bool CONTACT>
VDEV void substep(const VineParams& p, const JointImp& J, float m00inv, float rail_force, const Obstacles& ob,
                  ContactScratch* cs, ContactCache& cc, Dyn& d, float& lip, bool ghost = false) {
  float a[VINE_NL], b[VINE_NL], As[VINE_NL], Bs[VINE_NL];
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) { const float w2 = __fmul_rn(d.v[j + 1], d.v[j + 1]); a[j] = __fmul_rn(d.C[j], w2); b[j] = __fmul_rn(d.S[j], w2); }
  As[VINE_NL - 2] = __fmul_rn(p.Lbeta[VINE_NL - 1], a[VINE_NL - 1]);
  Bs[VINE_NL - 2] = __fmul_rn(p.Lbeta[VINE_NL - 1], b[VINE_NL - 1]);
#pragma unroll
  for (int j = VINE_NL - 3; j >= 0; --j) {
    As[j] = __fmaf_rn(p.Lbeta[j + 1], a[j + 1], As[j + 1]);
    Bs[j] = __fmaf_rn(p.Lbeta[j + 1], b[j + 1], Bs[j + 1]);
  }
  float f[6];
  f[0] = __fmaf_rn(-p.inv_L, __fmaf_rn(p.Lbeta[0], b[0], Bs[0]), __fmaf_rn(-p.damping, d.v[0], rail_force));
  {
    float Ap = a[0], Bp = b[0];
    f[1] = __fmaf_rn(d.C[0], Bs[0], __fmul_rn(d.S[0], __fsub_rn(p.gbeta[0], As[0])));
#pragma unroll
    for (int j = 1; j < VINE_NL; ++j) {
      const float P = j == VINE_NL - 1 ? __fmul_rn(p.Lbeta[j], Ap) : __fmaf_rn(p.Lbeta[j], Ap, As[j]);
      const float Q = j == VINE_NL - 1 ? __fmul_rn(p.Lbeta[j], Bp) : __fmaf_rn(p.Lbeta[j], Bp, Bs[j]);
      f[j + 1] = __fmaf_rn(d.C[j], Q, __fmul_rn(d.S[j], __fsub_rn(p.gbeta[j], P)));
      if (j + 1 < VINE_NL) { Ap = __fadd_rn(Ap, a[j]); Bp = __fadd_rn(Bp, b[j]); }
    }
  }
  // joint torques (relative coordinates) -> absolute: Q_j = t_j - t_{j+1}
  {
    float tn = 0.f;
#pragma unroll
    for (int j = VINE_NL - 1; j >= 0; --j) {
      const float th = j == 0 ? d.x[1] : __fsub_rn(d.x[j + 1], d.x[j]);
      const float thd = j == 0 ? d.v[1] : __fsub_rn(d.v[j + 1], d.v[j]);
      const float t = __fmaf_rn(-J.ek[j], thd, __fmaf_rn(-J.kk[j], th, J.tc[j]));
      f[j + 1] = __fadd_rn(f[j + 1], j == VINE_NL - 1 ? t : __fsub_rn(t, tn));
      tn = t;
    }
  }
  if constexpr (CONTACT) lip = contact_forces(p, ob, cs, cc, d, f, ghost);   // ghost: a lane without an env of its own (see there)
  // lower triangle of the SPD system matrix; rows/cols: 0 = cart, 1..5 = links
  float M[6][6];
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) {
    M[j + 1][0] = __fmul_rn(-p.beta[j], d.C[j]);
    M[j + 1][j + 1] = J.diag[j];
#pragma unroll
    for (int m = 0; m < j; ++m) {
      const float c = __fmaf_rn(d.C[j], d.C[m], __fmul_rn(d.S[j], d.S[m]));
      M[j + 1][m + 1] = (m == j - 1) ? __fmaf_rn(p.Lbeta[j], c, -J.gam[j]) : __fmul_rn(p.Lbeta[j], c);
    }
  }
  // LDL^T (row-wise): u_q = A_jq - sum_{r<q} u_r L_qr ; L_jq = u_q / d_q ; d_j = A_jj - sum_q u_q L_jq
  float dinv[6];
  dinv[0] = m00inv;
#pragma unroll
  for (int j = 1; j < 6; ++j) {
    float u[5];
    float dj = M[j][j];
#pragma unroll
    for (int q = 0; q < j; ++q) {
      float uq = M[j][q];
#pragma unroll
      for (int r = 0; r < q; ++r) uq = __fmaf_rn(-u[r], M[q][r], uq);
      u[q] = uq;
      const float l = __fmul_rn(uq, dinv[q]);
      M[j][q] = l;
      dj = __fmaf_rn(-uq, l, dj);
    }
    dinv[j] = rcp_approx(dj);
  }
  // solve M a = f (dv = h a is folded into the velocity update)
#pragma unroll
  for (int i = 1; i < 6; ++i)
#pragma unroll
    for (int q = 0; q < i; ++q) f[i] = __fmaf_rn(-M[i][q], f[q], f[i]);
#pragma unroll
  for (int i = 0; i < 6; ++i) f[i] = __fmul_rn(f[i], dinv[i]);
#pragma unroll
  for (int i = 4; i >= 0; --i)
#pragma unroll
    for (int q = i + 1; q < 6; ++q) f[i] = __fmaf_rn(-M[q][i], f[q], f[i]);
  d.v[0] = __fmaf_rn(p.h, f[0], d.v[0]); d.x[0] = __fmaf_rn(p.h, d.v[0], d.x[0]);
#pragma unroll
  for (int j = 0; j < VINE_NL; ++j) {
    d.v[j + 1] = __fmaf_rn(p.h, f[j + 1], d.v[j + 1]);
    d.x[j + 1] = __fmaf_rn(p.h, d.v[j + 1], d.x[j + 1]);
    link_trig(d.x[j + 1], d.S[j], d.C[j]);   // evaluated afresh: no drift and no bound on the link rate
  }
}

// ------------------------------------------------------------------------------------------
// compute_observations V5:1339-1390, compute_reward V5:1218-1248 + compute_reward_jit
// V5:1470-1537, compute_reset_jit V5:1540-1558, timeout VT:366.
// ------------------------------------------------------------------------------------------
VDEV float norm3_torch(float x, float y, float z) {  // torch linalg.norm (CPU): nested fma, IEEE sqrt
  return __fsqrt_rn(__fmaf_rn(z, z, __fmaf_rn(y, y, __fmul_rn(x, x))));
}

struct PostIn {
  float q[6], qd[6], prev_q[6];
  float tip[3], prev_tip[3], tipvel[3], target[3], target_vel[3], obj[2];
  float cart_y, smoothed, u_fpam, u_rail, prev_u_rail;
  float contact[VINE_MAX_CFI];
  int64_t reset_in, progress;
};

struct PostOut { float obs[VINE_MAX_OBS]; float rew; float r[VINE_NUM_REWARDS]; int64_t reset; unsigned char timeout; };

// raw (unscaled, noise-free) observation row in the order of V5:1354-1378
VDEV void observation_row(const VineParams& p, const PostIn& in, float raw[VINE_MAX_OBS]) {
  float fdq[6], fdt[3];
#pragma unroll
  for (int i = 0; i < 6; ++i) fdq[i] = div_rn(__fsub_rn(in.q[i], in.prev_q[i]), p.control_dt);      // V5:1347
#pragma unroll
  for (int i = 0; i < 3; ++i) fdt[i] = div_rn(__fsub_rn(in.tip[i], in.prev_tip[i]), p.control_dt);  // V5:1348
  const int t = p.obs_type;
#pragma unroll
  for (int i = 0; i < VINE_MAX_OBS; ++i) raw[i] = 0.f;
  if (t == VINE_OBS_TIP_AND_CART_AND_OBJ_INFO) {
    raw[0] = in.q[0]; raw[1] = fdq[0];
#pragma unroll
    for (int i = 0; i < 3; ++i) { raw[2 + i] = in.tip[i]; raw[5 + i] = fdt[i]; raw[8 + i] = in.target[i]; raw[11 + i] = in.target_vel[i]; }
    raw[14] = in.smoothed; raw[15] = in.prev_u_rail; raw[16] = in.obj[0]; raw[17] = in.obj[1];
    return;
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) raw[i] = in.q[i];
  if (t != VINE_OBS_POS_ONLY) {
#pragma unroll
    for (int i = 0; i < 6; ++i) raw[6 + i] = t == VINE_OBS_POS_AND_VEL ? in.qd[i] : (t == VINE_OBS_POS_AND_PREV_POS ? in.prev_q[i] : fdq[i]);
  }
  if (t == VINE_OBS_POS_ONLY) {
#pragma unroll
    for (int i = 0; i < 3; ++i) { raw[6 + i] = in.tip[i]; raw[9 + i] = in.target[i]; }
    raw[12] = in.smoothed; raw[13] = in.prev_u_rail;
    return;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    raw[12 + i] = in.tip[i];
    raw[15 + i] = t == VINE_OBS_POS_AND_VEL ? in.tipvel[i] : (t == VINE_OBS_POS_AND_PREV_POS ? in.prev_tip[i] : fdt[i]);
    raw[18 + i] = in.target[i]; raw[21 + i] = in.target_vel[i];
  }
  raw[24] = in.smoothed; raw[25] = in.prev_u_rail;
  if (t == VINE_OBS_POS_AND_FD_VEL_AND_OBJ_INFO) { raw[26] = in.obj[0]; raw[27] = in.obj[1]; }
}

// noise: [O] standard normals or nullptr
VDEV void post_physics(const VineParams& p, const PostIn& in, const float* noise, PostOut& o) {
  float raw[VINE_MAX_OBS];
  observation_row(p, in, raw);
#pragma unroll
  for (int i = 0; i < VINE_MAX_OBS; ++i) {
    float v = div_rn(raw[i], p.obs_scale[i]);                            // V5:1385
    if (noise != nullptr && i < p.O) v = __fadd_rn(v, __fmul_rn(p.obs_noise, noise[i]));  // V5:1388-1390
    o.obs[i] = v;
  }
  const float dist = norm3_torch(__fsub_rn(in.tip[0], in.target[0]), __fsub_rn(in.tip[1], in.target[1]),
                                 __fsub_rn(in.tip[2], in.target[2]));       // V5:1219
  const bool reached = dist < p.success_dist;                               // V5:1228
  const bool limit_hit = (in.cart_y > p.soft_limit) || (in.cart_y < -p.soft_limit);  // V5:1232-1233
  const bool tip_limit_hit = in.tip[1] < in.target[1];                      // V5:1237
  float contact = 0.f; bool nonzero = false;
  if (p.shelf) {                                                            // V5:1240-1244 mean over the sim steps
    float s = in.contact[0];
#pragma unroll
    for (int i = 1; i < VINE_MAX_CFI; ++i) if (i < p.C) s = __fadd_rn(s, in.contact[i]);
    contact = div_rn(s, (float)p.C);
    nonzero = contact > 0.f;
  }
  float* r = o.r;
  r[0] = __fsub_rn(0.f, dist);
  r[1] = -1.f;
  r[2] = reached ? 1000.f : 0.f;
  const float vs = norm3_torch(__fsub_rn(in.tipvel[0], in.target_vel[0]), __fsub_rn(in.tipvel[1], in.target_vel[1]),
                               __fsub_rn(in.tipvel[2], in.target_vel[2]));
  r[3] = __fsub_rn(0.f, reached ? vs : 0.f);
  r[4] = norm3_torch(in.tipvel[0], in.tipvel[1], in.tipvel[2]);
  r[5] = __fsub_rn(0.f, fabsf(in.u_rail));
  r[6] = __fsub_rn(0.f, fabsf(in.u_fpam));
  r[7] = __fsub_rn(0.f, fabsf(__fsub_rn(in.u_rail, in.prev_u_rail)));
  r[8] = __fsub_rn(0.f, fabsf(__fsub_rn(in.u_fpam, in.smoothed)));
  r[9] = limit_hit ? -100.f : 0.f;
  r[10] = __fsub_rn(0.f, fabsf(in.cart_y));
  r[11] = tip_limit_hit ? -100.f : 0.f;
  r[12] = __fsub_rn(0.f, (contact > 0.f) ? contact : 0.f);
  // torch.sum(dim=-1) over 13 contiguous f32 (CPU kernel): tail 8..12 first, then lanes 0..7
  float acc = 0.f;
#pragma unroll
  for (int i = 8; i < 13; ++i) acc = __fadd_rn(acc, __fmul_rn(r[i], p.w[i]));
#pragma unroll
  for (int i = 0; i < 8; ++i) acc = __fadd_rn(acc, __fmul_rn(r[i], p.w[i]));
  o.rew = acc;
  int64_t reset = (in.progress >= p.max_len_m1) ? 1 : in.reset_in;          // V5:1544
  if (reached && p.reach_reset) reset = 1;
  if (tip_limit_hit && p.tip_reset) reset = 1;
  if (limit_hit) reset = 1;
  if (nonzero && p.contact_reset) reset = 1;
  o.reset = reset;
  o.timeout = (unsigned char)((in.progress >= p.max_len_m1) && (reset != 0));  // VT:366
}

// ------------------------------------------------------------------------------------------
// reset_idx V5:774-885 + sample_target_positions V5:887-914.  Draw k of the reference's call
// order = Philox block k/4, lane k%4: joints 1..5, cart, target x,y,z, shelf depth, pipe depth.
// ------------------------------------------------------------------------------------------
VDEV void sample_targets(const VineParams& p, const uint32_t u[12], float target[3]) {
  if (p.rand_targets) {
    target[0] = uniform_ab(u[6], 0.f, 0.f);
    target[1] = uniform_ab(u[7], p.ty_lo, p.ty_rng);
    target[2] = uniform_ab(u[8], p.tz_lo, p.tz_rng);
  } else { target[0] = 0.f; target[1] = p.ty_hi; target[2] = p.tz_lo_fixed; }
}

VDEV void reset_env(const VineParams& p, uint32_t k0, uint32_t k1, uint32_t gid, uint32_t step,
                    float q[6], float qd[6], float target[3], float obj[2]) {
  uint32_t u[12];
#pragma unroll
  for (uint32_t b = 0; b < 3; ++b) {
    const uint4 r = philox4x32(k0, k1, gid, VINE_SITE_RESET, step, b);
    u[4 * b] = r.x; u[4 * b + 1] = r.y; u[4 * b + 2] = r.z; u[4 * b + 3] = r.w;
  }
  if (p.rand_dof_init) {
#pragma unroll
    for (int j = 0; j < VINE_NL; ++j) q[j + 1] = uniform_ab(u[j], p.rev_lo, p.rev_rng);
    q[0] = uniform_ab(u[5], p.cart_lo, p.cart_rng);
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) q[j] = 0.f;
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) qd[j] = 0.f;
  sample_targets(p, u, target);
  if (p.shelf) obj[0] = uniform_ab(u[9], p.dep_lo, p.dep_rng);              // V5:822-839
  if (p.pipe) {                                                             // V5:854-885
    const float ez = __fsub_rn(1.0f, target[2]);
    // np.polyval with float64 coefficients evaluated on the f32 effective_z (Horner), then f32
    const double x = (double)ez;
    double y = 1.0e4 * 1.3199;
    y = __dadd_rn(__dmul_rn(y, x), 1.0e4 * -1.2276);
    y = __dadd_rn(__dmul_rn(y, x), 1.0e4 * 0.4045);
    y = __dadd_rn(__dmul_rn(y, x), 1.0e4 * -0.0447);
    obj[1] = __fmul_rn((float)y, 0.017453292519943295f);                    // torch.deg2rad
    obj[0] = uniform_ab(u[p.shelf ? 10 : 9], p.dep_lo, p.dep_rng);          // V5:863
  }
}
