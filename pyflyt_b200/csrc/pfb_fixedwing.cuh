// pfb_fixedwing.cuh — per-env body of the Fixedwing stepper (one thread = one aircraft = one env).
//
// Replaces (paths under /root/reference/PyFlyt/):
//   core/drones/fixedwing.py:229-291                 update_control / update_physics / update_state
//   core/abstractions/lifting_surfaces.py:73-110,266-498   Khan & Nahon flat-plate / stall aero per surface
//   core/abstractions/motors.py:110-195              one propeller motor
//   PyBullet stepSimulation (SURVEY §A.3)            composite rigid body with COM offset + products of inertia
//   gym_envs/fixedwing_envs/fixedwing_waypoints_env.py:121-190, fixedwing_base_env.py:226-278,
//   gym_envs/utils/waypoint_handler.py:53-213        Fixedwing-Waypoints epilogue
//
// The lifting-surface model and the general rigid-body step are shared with the rocket (pfb_rocket.cuh).
#pragma once

#include "pfb_quadx.cuh"

namespace pfb {

constexpr int kMaxSurfaces = 5;
constexpr int kMaxTargets = 8;

// one lifting surface, host-precomputed (lifting_surfaces.py:217-262); axis vectors in the base frame
struct SurfaceParams {
  float r[3];          // point of application (link COM)
  float lift[3];       // lifting_unit
  float fwd[3];        // forward_unit (drag_unit)
  float tq[3];         // torque_unit = lift x fwd
  float lag;           // physics_period / tau
  float Cl_alpha_3D;
  float inv_pi_aspect; // 1 / (pi * aspect)
  float dCl;           // Cl_alpha_3D * aero_tau * eta * deg2rad(deflection_limit): delta_Cl per unit actuation
  float flap_to_chord;
  float alpha_0_base, alpha_stall_P_base, alpha_stall_N_base;
  float Cd_0;
  float defl_rad;      // deg2rad(deflection_limit)
  float stall_k;       // 0.41 * (1 - exp(-17 / aspect))
  float q_area;        // half_rho * area
  float chord;
};

// general rigid body about the base origin O (base axes): mass M, first moment M c, inertia I_O and
// the inverse of the 6x6 Newton-Euler matrix [[M E, -M c^x], [M c^x, I_O]]
struct RigidParams {
  float mass;
  float mc[3];
  float I[9];
  float Ainv[36];
};

constexpr int kMaxShapes = 12;
struct ContactParams {
  int n_shapes;
  int kind[kMaxShapes];
  float dims[kMaxShapes][3];
  float at[kMaxShapes][3];
  float rot[kMaxShapes][9];  // primitive axes in the base frame (row-major)
  float thr[kMaxShapes];
  float zmax;
};

struct FixedwingParams {
  float dt, gravity, vmax;
  int ratio;
  RigidParams rb;
  int n_surfaces;
  SurfaceParams surf[kMaxSurfaces];
  // motor (fixedwing.py:145-166): thrust along +x at r_m
  float motor_r[3];
  float thrust_k, torque_k, motor_lag, noise_ratio, noise_loc;
  float start_vel[3];
  ContactParams contact;
  WindParams wind;  // analytic wind field; kind 0 = still air
};

struct WaypointParams {
  int env_step_ratio, max_steps, angle_representation, sparse_reward, warmup_steps, flight_mode;
  int num_targets;
  float dome2, dome, goal_reach_distance, min_height;
};

// MAFixedwingDogfight constants (pz_envs/fixedwing_envs/ma_fixedwing_dogfight_env.py:42-62)
struct DogfightParams {
  int team_size, env_step_ratio, max_steps, sparse_reward, warmup_steps;
  float dome, damage_per_hit, lethal_distance, lethal_angle, aggressiveness, cooperativeness;
  float spawn_min_radius, spawn_max_radius;
};

// state tensor rows [F][N] for Fixedwing
enum {
  FW_POS = 0, FW_QUAT = 3, FW_VEL = 7, FW_ANGVEL = 10, FW_ACT = 13 /*5*/, FW_THR = 18, FW_POS_LO = 19, FW_QUAT_LO = 22,
  FW_VEL_LO = 26, FW_DIST = 29 /* waypoint handler new_distance */, FW_TARGETS = 30 /* 3 * kMaxTargets */, FW_ROWS = 30 + 3 * kMaxTargets
};
enum { FI_STEP = 0, FI_FLAGS = 1, FI_NTARGETS = 2 /* targets reached so far */, FI_ROWS = 3 };
enum { FLAG_ENV_COMPLETE = 64 };

struct FixedwingRegs {
  xreal px, py, pz;
  qreal qx, qy, qz, qw;
  vreal vx, vy, vz;
  float wx, wy, wz;
  float act[kMaxSurfaces];
  float thr;
  float sp[6];
  Rot<rreal> R;
  Vec3 vb;
  uint32_t flags;
};

// sin and cos for |x| <= ~6.5 (alpha_eff): quadrant reduction + minimax on [-pi/4, pi/4]; |error| < 2e-7
PFB_HD void sincos_f(float x, float& s, float& c) {
  float k = rintf(x * 0.63661977236758134308f);
  float r = fmaf(k, -1.57079637050628662109f, x);   // pi/2 split in two fp32 words
  r = fmaf(k, 4.37113900018624283e-8f, r);
  float r2 = r * r;
  float sp = fmaf(r2, fmaf(r2, fmaf(r2, -1.9515295891e-4f, 8.3321608736e-3f), -1.6666654611e-1f), 1.0f) * r;
  float cp = fmaf(r2, fmaf(r2, fmaf(r2, fmaf(r2, 2.443315711809948e-5f, -1.388731625493765e-3f), 4.166664568298827e-2f), -0.5f), 1.0f);
  int q = (int)k & 3;
  float ss = (q & 1) ? cp : sp, cc = (q & 1) ? sp : cp;
  s = (q & 2) ? -ss : ss;
  c = ((q + 1) & 2) ? -cc : cc;
}

// LiftingSurface.physics_update (lifting_surfaces.py:266-324): actuation lag, AoA, (Cl, Cd, CM) with the
// pre-/post-stall branches evaluated as selects, force + torque in the base frame.
// `wind` / `wc`: optional analytic wind (lifting_surfaces.py:88-93): the surface sees the velocity through the air
PFB_HD void surface_force(const SurfaceParams& sf, float& act, float cmd, Vec3 vb, Vec3 w, Vec3& F, Vec3& T, const WindParams* wind = nullptr,
                          const WindCtx* wc = nullptr) {
  act = fmaf(sf.lag, cmd - act, act);
  // link COM velocity in the body frame: v_b + w_b x r
  Vec3 r = Vec3{sf.r[0], sf.r[1], sf.r[2]};
  Vec3 v = vb + cross(w, r);
  if (wind) v = v - wind_body_at(*wind, *wc, sf.r[0], sf.r[1], sf.r[2]);
  float lifting = v.x * sf.lift[0] + v.y * sf.lift[1] + v.z * sf.lift[2];
  float forward = v.x * sf.fwd[0] + v.y * sf.fwd[1] + v.z * sf.fwd[2];
  float speed2 = v.x * v.x + v.y * v.y + v.z * v.z;
  float alpha = atan2_f(-lifting, forward);
  // _jitted_compute_aero_data (lifting_surfaces.py:349-448)
  float deflection = act * sf.defl_rad;
  float delta_Cl = sf.dCl * act;
  float delta_Cl_max = sf.flap_to_chord * delta_Cl;
  float inv_cl3d = fast_rcp(sf.Cl_alpha_3D);
  float Cl_max_P = fmaf(sf.Cl_alpha_3D, sf.alpha_stall_P_base - sf.alpha_0_base, delta_Cl_max);
  float Cl_max_N = fmaf(sf.Cl_alpha_3D, sf.alpha_stall_N_base - sf.alpha_0_base, delta_Cl_max);
  float alpha_0 = sf.alpha_0_base - delta_Cl * inv_cl3d;
  float alpha_stall_P = alpha_0 + Cl_max_P * inv_cl3d;
  float alpha_stall_N = alpha_0 + Cl_max_N * inv_cl3d;
  bool attached = (alpha_stall_N < alpha) && (alpha < alpha_stall_P);
  const float half_pi = 1.57079632679489661923f;
  float Cl_lin = sf.Cl_alpha_3D * (alpha - alpha_0);
  // induced angle: linear regime Cl / (pi AR); post-stall np.interp from the stall value down to 0 at +-90 deg
  bool pos = alpha > 0.0f;
  float a_st = pos ? alpha_stall_P : alpha_stall_N;
  float ai_stall = sf.Cl_alpha_3D * (a_st - alpha_0) * sf.inv_pi_aspect;
  float edge = pos ? half_pi : -half_pi;
  float frac = fast_div(alpha - a_st, edge - a_st);   // 0 at the stall angle, 1 at +-90 deg
  frac = fminf(fmaxf(frac, 0.0f), 1.0f);              // np.interp clamps outside the interval
  float ai_post = ai_stall * (1.0f - frac);
  float alpha_i = attached ? Cl_lin * sf.inv_pi_aspect : ai_post;
  float alpha_eff = alpha - alpha_0 - alpha_i;
  float se, ce;
  sincos_f(alpha_eff, se, ce);
  float Cd_90 = fmaf(deflection, fmaf(deflection, -4.26e-2f, 2.1e-1f), 1.98f);
  float CN_post = Cd_90 * se * (fast_rcp(fmaf(0.44f, fabsf(se), 0.56f)) - sf.stall_k);
  float CT = (attached ? 1.0f : 0.5f) * sf.Cd_0 * ce;
  float CN = attached ? (Cl_lin + CT * se) * fast_rcp(ce) : CN_post;
  float Cl = attached ? Cl_lin : (CN * ce - CT * se);
  float Cd = CN * se + CT * ce;
  float aeff_m = attached ? alpha_eff : fabsf(alpha_eff);
  float CM = -CN * (0.25f - 0.175f * (1.0f - aeff_m * 0.63661977236758134308f));
  // _jitted_compute_force_torque (lifting_surfaces.py:450-498); sin/cos(alpha) straight from the components
  float Q_area = sf.q_area * speed2;
  float h2 = lifting * lifting + forward * forward;
  float inv_h = h2 > 0.0f ? fast_rsqrt(h2) : 0.0f;
  float sa = -lifting * inv_h, ca = h2 > 0.0f ? forward * inv_h : 1.0f;
  float lift = Cl * Q_area, drag = Cd * Q_area;
  float fn = lift * ca + drag * sa;
  float fp = lift * sa - drag * ca;
  Vec3 Fi = Vec3{sf.lift[0] * fn + sf.fwd[0] * fp, sf.lift[1] * fn + sf.fwd[1] * fp, sf.lift[2] * fn + sf.fwd[2] * fp};
  float tm = Q_area * CM * sf.chord;
  F = F + Fi;
  T = T + cross(r, Fi) + Vec3{tm * sf.tq[0], tm * sf.tq[1], tm * sf.tq[2]};
}

// ground-contact flag over a list of axis-aligned primitives (shared helper)
// `top` = height of the surface tested (0 for the ground plane, 0.15 for the landing pad)
PFB_HD bool ground_contact(const ContactParams& cp, float pz, float r20, float r21, float r22, float top = 0.0f) {
  if (pz - top > cp.zmax) return false;
  bool hit = false;
#pragma unroll 1
  for (int k = 0; k < cp.n_shapes; ++k) {
    float cz = pz + r20 * cp.at[k][0] + r21 * cp.at[k][1] + r22 * cp.at[k][2];
    // world-z components of the primitive's own axes: third row of (R * rot)
    const float* q = cp.rot[k];
    float z0 = r20 * q[0] + r21 * q[3] + r22 * q[6];
    float z1 = r20 * q[1] + r21 * q[4] + r22 * q[7];
    float z2 = r20 * q[2] + r21 * q[5] + r22 * q[8];
    float extent;
    if (cp.kind[k] == 0) extent = fabsf(z0) * cp.dims[k][0] + fabsf(z1) * cp.dims[k][1] + fabsf(z2) * cp.dims[k][2];
    else if (cp.kind[k] == 1) extent = cp.dims[k][1] * fabsf(z2) + cp.dims[k][0] * fast_sqrt(fmaxf(0.0f, 1.0f - z2 * z2));
    else extent = cp.dims[k][0];
    hit = hit || (cz - extent - top < cp.thr[k]);
  }
  return hit;
}

// Bullet free-body step for a composite body with COM offset c and full inertia I_O (SURVEY §A.3):
//   F = M (a_O + wdot x c + w x (w x c)),   T_O = I_O wdot + w x I_O w + M c x a_O
// F_b / T_b: external force / torque about O in the body frame (without gravity).  State update is the
// same semi-implicit Euler + body-frame exp-map as the quad.
template <typename Regs>
PFB_HD void rigid_step(const RigidParams& rb, float gravity, float dt_f, float vmax_f, Regs& s, Vec3 F, Vec3 T) {
  const Rot<rreal>& R = s.R;
  const float r20 = (float)R.m20, r21 = (float)R.m21, r22 = (float)R.m22;
  // gravity on every link: M g at the COM; world z seen from the body is the third row of R
  Vec3 gb = Vec3{gravity * r20, gravity * r21, gravity * r22};
  Vec3 mc = Vec3{rb.mc[0], rb.mc[1], rb.mc[2]};
  F = F + rb.mass * gb;
  T = T + cross(mc, gb);
  Vec3 w = Vec3{s.wx, s.wy, s.wz};
  Vec3 Iw = Vec3{rb.I[0] * w.x + rb.I[1] * w.y + rb.I[2] * w.z, rb.I[3] * w.x + rb.I[4] * w.y + rb.I[5] * w.z,
                 rb.I[6] * w.x + rb.I[7] * w.y + rb.I[8] * w.z};
  Vec3 rf = F - cross(w, cross(w, mc));
  Vec3 rt = T - cross(w, Iw);
  const float rhs[6] = {rf.x, rf.y, rf.z, rt.x, rt.y, rt.z};
  float sol[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    float acc = 0.0f;
#pragma unroll
    for (int j = 0; j < 6; ++j) acc = fmaf(rb.Ainv[6 * i + j], rhs[j], acc);
    sol[i] = acc;
  }
  // world acceleration of the base origin, velocities first, then positions
  rreal ax = R.m00 * (rreal)sol[0] + R.m01 * (rreal)sol[1] + R.m02 * (rreal)sol[2];
  rreal ay = R.m10 * (rreal)sol[0] + R.m11 * (rreal)sol[1] + R.m12 * (rreal)sol[2];
  rreal az = R.m20 * (rreal)sol[0] + R.m21 * (rreal)sol[1] + R.m22 * (rreal)sol[2];
  const vreal dt = (vreal)dt_f;
  s.vx += (vreal)ax * dt;
  s.vy += (vreal)ay * dt;
  s.vz += (vreal)az * dt;
  if (fmaxf(fmaxf(fabsf((float)s.vx), fabsf((float)s.vy)), fabsf((float)s.vz)) >= vmax_f) {
    const vreal vmax = (vreal)vmax_f;
    s.vx = fmin(fmax(s.vx, -vmax), vmax);
    s.vy = fmin(fmax(s.vy, -vmax), vmax);
    s.vz = fmin(fmax(s.vz, -vmax), vmax);
  }
  s.px += (xreal)(s.vx * dt);
  s.py += (xreal)(s.vy * dt);
  s.pz += (xreal)(s.vz * dt);
  s.wx = fmaf(sol[3], dt_f, s.wx);
  s.wy = fmaf(sol[4], dt_f, s.wy);
  s.wz = fmaf(sol[5], dt_f, s.wz);
  if (fmaxf(fmaxf(fabsf(s.wx), fabsf(s.wy)), fabsf(s.wz)) > vmax_f * 0.57735f) {
    Mat3 Rf{(float)R.m00, (float)R.m01, (float)R.m02, (float)R.m10, (float)R.m11, (float)R.m12, (float)R.m20, (float)R.m21, (float)R.m22};
    Vec3 wc = quadx_clamp_world_rates(vmax_f, Rf, Vec3{s.wx, s.wy, s.wz});
    s.wx = wc.x; s.wy = wc.y; s.wz = wc.z;
  }
  float h2 = (s.wx * s.wx + s.wy * s.wy + s.wz * s.wz) * (0.25f * dt_f * dt_f);
  float sinc = fmaf(h2, fmaf(h2, fmaf(h2, fmaf(h2, 2.7557319e-6f, -1.9841270e-4f), 8.3333333e-3f), -1.6666667e-1f), 1.0f);
  float scale = 0.5f * dt_f * sinc;
  float cw = fmaf(h2, fmaf(h2, fmaf(h2, fmaf(h2, fmaf(h2, -2.7557319e-7f, 2.4801587e-5f), -1.3888889e-3f), 4.1666667e-2f), -0.5f), 1.0f);
  qreal dx = (qreal)(s.wx * scale), dy = (qreal)(s.wy * scale), dz = (qreal)(s.wz * scale), dw = (qreal)cw;
  qreal nx = s.qw * dx + s.qx * dw + s.qy * dz - s.qz * dy;
  qreal ny = s.qw * dy + s.qy * dw + s.qz * dx - s.qx * dz;
  qreal nz = s.qw * dz + s.qz * dw + s.qx * dy - s.qy * dx;
  qreal nw = s.qw * dw - s.qx * dx - s.qy * dy - s.qz * dz;
  qreal n2 = nx * nx + ny * ny + nz * nz + nw * nw;
#if PFB_Q_DOUBLE
  qreal e = n2 - 1.0;
  qreal inv = 1.0 - 0.5 * e + 0.375 * e * e;
#else
  qreal inv = 1.0f / sqrtf(n2);
#endif
  s.qx = nx * inv; s.qy = ny * inv; s.qz = nz * inv; s.qw = nw * inv;
}

// first half of update_state (fixedwing.py:271-283): rotation matrix + body-frame linear velocity
template <typename Regs>
PFB_HD void body_update_state(Regs& s) {
  rot_from_quat<rreal>(s.qx, s.qy, s.qz, s.qw, s.R);
  const Rot<rreal>& R = s.R;
  rreal vx = (rreal)s.vx, vy = (rreal)s.vy, vz = (rreal)s.vz;
  s.vb.x = (float)(R.m00 * vx + R.m10 * vy + R.m20 * vz);
  s.vb.y = (float)(R.m01 * vx + R.m11 * vy + R.m21 * vz);
  s.vb.z = (float)(R.m02 * vx + R.m12 * vy + R.m22 * vz);
}

// fixedwing.py:229-259: mode 0 = RPYT mixing onto [left ail, right ail, h-tail, v-tail, main wing, motor]
template <int MODE>
PFB_HD void fixedwing_command(const FixedwingRegs& s, float* cmd) {
  if (MODE == -1) {
#pragma unroll
    for (int k = 0; k < 6; ++k) cmd[k] = s.sp[k];
  } else {
    cmd[0] = s.sp[0]; cmd[1] = -s.sp[0]; cmd[2] = s.sp[1]; cmd[3] = -s.sp[2]; cmd[4] = -s.sp[1]; cmd[5] = s.sp[3];
  }
}

// one physics substep: update_physics (fixedwing.py:261-264) + stepSimulation + update_state
// FULL = the caller has checked (launch-uniform) that the model has all kMaxSurfaces surfaces and no wind.  The generic path
// tests `i < n_surfaces` and `windy` per surface: uniform branches, but branches — every surface becomes its own chain of basic
// blocks and ptxas schedules inside a block only, so the five ~230-instruction surfaces run one after the other, each at the
// pace of its own dependency chain (atan2 -> stall selects -> sincos -> coefficients -> force).  With < 1 warp per scheduler
// at the batch sizes these vehicles run at (16 384 envs) instruction-level parallelism is the only latency hiding there is:
// FULL removes the tests at compile time, the surfaces land in ONE basic block and their chains interleave.
template <bool FULL = false>
PFB_HD void fixedwing_substep(const FixedwingParams& p, FixedwingRegs& s, const float* cmd, float xi) {
  Vec3 F = Vec3{0.f, 0.f, 0.f}, T = Vec3{0.f, 0.f, 0.f};
  const Vec3 w = Vec3{s.wx, s.wy, s.wz};
  // fully unrolled: the surface tables become immediate constant-bank operands instead of indexed loads
  const bool windy = FULL ? false : p.wind.kind != 0;  // uniform: the parameter block is launch-constant
  WindCtx wc = WindCtx{Vec3{0.f, 0.f, 0.f}, 0.f, 0.f, 0.f, 0.f};
  if (windy) wc = wind_ctx(p.wind, (float)s.pz, (float)s.R.m00, (float)s.R.m01, (float)s.R.m02, (float)s.R.m10, (float)s.R.m11, (float)s.R.m12,
                           (float)s.R.m20, (float)s.R.m21, (float)s.R.m22);
#pragma unroll
  for (int i = 0; i < kMaxSurfaces; ++i) {
    if (FULL) surface_force(p.surf[i], s.act[i], cmd[i], s.vb, w, F, T);
    else if (i < p.n_surfaces) surface_force(p.surf[i], s.act[i], cmd[i], s.vb, w, F, T, windy ? &p.wind : nullptr, &wc);
  }
  // motor (motors.py:130-155): thrust + reaction torque along +x at motor_r
  {
    float t = s.thr;
    t = fmaf(p.motor_lag, cmd[5] - t, t);
    t = fmaf(xi * p.noise_ratio, t, t);
    s.thr = t;
    float a = t * fabsf(t);
    Vec3 Fm = Vec3{p.thrust_k * a, 0.0f, 0.0f};
    F = F + Fm;
    T = T + cross(Vec3{p.motor_r[0], p.motor_r[1], p.motor_r[2]}, Fm) + Vec3{p.torque_k * a, 0.0f, 0.0f};
  }
  const bool c = ground_contact(p.contact, (float)s.pz, (float)s.R.m20, (float)s.R.m21, (float)s.R.m22);
  s.flags = (s.flags & ~(uint32_t)FLAG_CONTACT_PREV) | (c ? (FLAG_CONTACT_PREV | FLAG_CONTACT_ARRAY) : 0u);
  rigid_step(p.rb, p.gravity, p.dt, p.vmax, s, F, T);
  body_update_state(s);
}

template <int MODE, bool FULL = false, typename NoiseFn>
PFB_HD void fixedwing_aviary_step(const FixedwingParams& p, FixedwingRegs& s, NoiseFn& noise) {
  s.flags &= ~(uint32_t)FLAG_CONTACT_ARRAY;
  noise.begin_step();
  float cmd[6];
  fixedwing_command<MODE>(s, cmd);
#pragma unroll 1
  for (int u = 0; u < p.ratio; ++u) fixedwing_substep<FULL>(p, s, cmd, noise.get(u));
}
// launch-uniform test for the FULL instantiation
#ifdef PFB_NO_FULL  // A/B knob: always the generic (branch per surface) substep
PFB_HD bool fixedwing_full_model(const FixedwingParams&) { return false; }
#else
PFB_HD bool fixedwing_full_model(const FixedwingParams& p) { return p.n_surfaces == kMaxSurfaces && p.wind.kind == 0; }
#endif

// fixedwing.py:194-204 + aviary.py:310-311
PFB_HD void fixedwing_reset(const FixedwingParams& p, FixedwingRegs& s, float sx, float sy, float sz, float roll, float pitch, float yaw) {
  s.px = (xreal)sx; s.py = (xreal)sy; s.pz = (xreal)sz;
  {
    qreal hr = (qreal)roll * (qreal)0.5, hp = (qreal)pitch * (qreal)0.5, hy = (qreal)yaw * (qreal)0.5;
    qreal sr = sin(hr), cr = cos(hr), sp = sin(hp), cp = cos(hp), sy_ = sin(hy), cy = cos(hy);
    s.qx = sr * cp * cy - cr * sp * sy_;
    s.qy = cr * sp * cy + sr * cp * sy_;
    s.qz = cr * cp * sy_ - sr * sp * cy;
    s.qw = cr * cp * cy + sr * sp * sy_;
  }
  s.vx = (vreal)p.start_vel[0]; s.vy = (vreal)p.start_vel[1]; s.vz = (vreal)p.start_vel[2];  // resetBaseVelocity, world frame
  s.wx = s.wy = s.wz = 0.0f;
#pragma unroll
  for (int k = 0; k < kMaxSurfaces; ++k) s.act[k] = 0.0f;
  s.thr = 0.0f;
#pragma unroll
  for (int k = 0; k < 6; ++k) s.sp[k] = 0.0f;
  s.flags = 0u;
  body_update_state(s);
}

// `st` is field-major [F][N] by default; `rs` / `ci` select an env-major record instead (row stride 1, base already at the
// env's record): the spare post-reset states of the Waypoints env (pfb_fixedwing.cu)
PFB_HD void fixedwing_load(const float* __restrict__ st, const int32_t* __restrict__ ist, int64_t N, int64_t i, FixedwingRegs& s,
                           int64_t rs = -1, int64_t ci = -1) {
  if (rs < 0) { rs = N; ci = i; }
  auto F = [&](int row) { return st[(int64_t)row * rs + ci]; };
  s.px = join_hi_lo(F(FW_POS + 0), F(FW_POS_LO + 0));
  s.py = join_hi_lo(F(FW_POS + 1), F(FW_POS_LO + 1));
  s.pz = join_hi_lo(F(FW_POS + 2), F(FW_POS_LO + 2));
  s.qx = join_hi_lo(F(FW_QUAT + 0), F(FW_QUAT_LO + 0));
  s.qy = join_hi_lo(F(FW_QUAT + 1), F(FW_QUAT_LO + 1));
  s.qz = join_hi_lo(F(FW_QUAT + 2), F(FW_QUAT_LO + 2));
  s.qw = join_hi_lo(F(FW_QUAT + 3), F(FW_QUAT_LO + 3));
  s.vx = join_hi_lo(F(FW_VEL + 0), F(FW_VEL_LO + 0));
  s.vy = join_hi_lo(F(FW_VEL + 1), F(FW_VEL_LO + 1));
  s.vz = join_hi_lo(F(FW_VEL + 2), F(FW_VEL_LO + 2));
  s.wx = F(FW_ANGVEL + 0); s.wy = F(FW_ANGVEL + 1); s.wz = F(FW_ANGVEL + 2);
#pragma unroll
  for (int k = 0; k < kMaxSurfaces; ++k) s.act[k] = F(FW_ACT + k);
  s.thr = F(FW_THR);
  s.flags = (uint32_t)ist[(int64_t)FI_FLAGS * N + i];
  body_update_state(s);
}

PFB_HD void fixedwing_store(float* __restrict__ st, int32_t* __restrict__ ist, int64_t N, int64_t i, const FixedwingRegs& s,
                            bool with_flags = true, int64_t rs = -1, int64_t ci = -1) {
  if (rs < 0) { rs = N; ci = i; }
  auto S = [&](int row, float v) { st[(int64_t)row * rs + ci] = v; };
  float hi, lo;
  split_hi_lo(s.px, hi, lo); S(FW_POS + 0, hi); S(FW_POS_LO + 0, lo);
  split_hi_lo(s.py, hi, lo); S(FW_POS + 1, hi); S(FW_POS_LO + 1, lo);
  split_hi_lo(s.pz, hi, lo); S(FW_POS + 2, hi); S(FW_POS_LO + 2, lo);
  split_hi_lo(s.qx, hi, lo); S(FW_QUAT + 0, hi); S(FW_QUAT_LO + 0, lo);
  split_hi_lo(s.qy, hi, lo); S(FW_QUAT + 1, hi); S(FW_QUAT_LO + 1, lo);
  split_hi_lo(s.qz, hi, lo); S(FW_QUAT + 2, hi); S(FW_QUAT_LO + 2, lo);
  split_hi_lo(s.qw, hi, lo); S(FW_QUAT + 3, hi); S(FW_QUAT_LO + 3, lo);
  split_hi_lo(s.vx, hi, lo); S(FW_VEL + 0, hi); S(FW_VEL_LO + 0, lo);
  split_hi_lo(s.vy, hi, lo); S(FW_VEL + 1, hi); S(FW_VEL_LO + 1, lo);
  split_hi_lo(s.vz, hi, lo); S(FW_VEL + 2, hi); S(FW_VEL_LO + 2, lo);
  S(FW_ANGVEL + 0, s.wx); S(FW_ANGVEL + 1, s.wy); S(FW_ANGVEL + 2, s.wz);
#pragma unroll
  for (int k = 0; k < kMaxSurfaces; ++k) S(FW_ACT + k, s.act[k]);
  S(FW_THR, s.thr);
  if (with_flags) ist[(int64_t)FI_FLAGS * N + i] = (int32_t)s.flags;
}

// Round the fp64-carried fields to what the state tensor holds (hi + lo fp32 words) and re-derive the body-frame state
PFB_HD void fixedwing_requantize(FixedwingRegs& s) {
  float hi, lo;
  split_hi_lo(s.px, hi, lo); s.px = join_hi_lo(hi, lo);
  split_hi_lo(s.py, hi, lo); s.py = join_hi_lo(hi, lo);
  split_hi_lo(s.pz, hi, lo); s.pz = join_hi_lo(hi, lo);
  split_hi_lo(s.qx, hi, lo); s.qx = join_hi_lo(hi, lo);
  split_hi_lo(s.qy, hi, lo); s.qy = join_hi_lo(hi, lo);
  split_hi_lo(s.qz, hi, lo); s.qz = join_hi_lo(hi, lo);
  split_hi_lo(s.qw, hi, lo); s.qw = join_hi_lo(hi, lo);
  split_hi_lo(s.vx, hi, lo); s.vx = join_hi_lo(hi, lo);
  split_hi_lo(s.vy, hi, lo); s.vy = join_hi_lo(hi, lo);
  split_hi_lo(s.vz, hi, lo); s.vz = join_hi_lo(hi, lo);
  body_update_state(s);
}

// Aviary.state(i) (4,3) + aux_state (5 surface actuations + motor throttle): fixedwing.py:285-291
PFB_HD void fixedwing_drone_state(const FixedwingRegs& s, float* out12, float* aux6) {
  float roll, pitch, yaw;
  euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
  out12[0] = s.wx; out12[1] = s.wy; out12[2] = s.wz;
  out12[3] = roll; out12[4] = pitch; out12[5] = yaw;
  out12[6] = s.vb.x; out12[7] = s.vb.y; out12[8] = s.vb.z;
  out12[9] = (float)s.px; out12[10] = (float)s.py; out12[11] = (float)s.pz;
#pragma unroll
  for (int k = 0; k < kMaxSurfaces; ++k) aux6[k] = s.act[k];
  aux6[5] = s.thr;
}

}  // namespace pfb
