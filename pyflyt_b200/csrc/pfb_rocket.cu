// pfb_rocket.cu — Rocket kernels (Aviary surface + Rocket-Landing env) and their launchers.
#include <cmath>
#include <cstring>

#include "pfb_context.h"
#include "pfb_noise.cuh"
#include "pfb_tail_reset.cuh"
#include "pfb_rocket_host.h"

using namespace pfb;

int rk_build_params(const PfbModel& m, const PfbEnvConfig* env, RocketParams& p, LandingParams& l) { return rk_build_params_impl(m, env, p, l); }
int rk_state_rows() { return RK_ROWS; }
int rk_istate_rows() { return RI_ROWS; }
int rk_obs_dim(const PfbContext* h) { return (h->land.angle_representation == 0 ? 12 : 13) + 7 + 9 + 1; }

// ---------------------------------------------------------------------------------------------------
// kernels — Aviary surface
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_rk_reset(const __grid_constant__ RocketParams p, float* __restrict__ st,
                                                     int32_t* __restrict__ ist, float* __restrict__ setpoint,
                                                     const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                                                     const uint8_t* __restrict__ mask, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  RocketRegs s;
  rocket_reset(p, s, start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1], start_orn[3 * i + 2]);
  rocket_store(st, ist, N, i, s);
  ist[(int64_t)RI_STEP * N + i] = 0;
  if (setpoint)
    for (int k = 0; k < 7; ++k) setpoint[7 * i + k] = 0.0f;
}

// p.resetBaseVelocity(id, lin, ang) (rocket_base_env.py:228): world-frame velocities -> state rows
__global__ void __launch_bounds__(kBlock) k_rk_set_velocity(float* __restrict__ st, int32_t* __restrict__ ist, const float* __restrict__ lin,
                                                            const float* __restrict__ ang, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  RocketRegs s;
  rocket_load(st, ist, N, i, s);
  s.vx = (vreal)lin[3 * i]; s.vy = (vreal)lin[3 * i + 1]; s.vz = (vreal)lin[3 * i + 2];
  // the state carries the BODY rate: w_b = R^T w_world
  float ox = ang[3 * i], oy = ang[3 * i + 1], oz = ang[3 * i + 2];
  const Rot<rreal>& R = s.R;
  s.wx = (float)R.m00 * ox + (float)R.m10 * oy + (float)R.m20 * oz;
  s.wy = (float)R.m01 * ox + (float)R.m11 * oy + (float)R.m21 * oz;
  s.wz = (float)R.m02 * ox + (float)R.m12 * oy + (float)R.m22 * oz;
  rocket_store(st, ist, N, i, s);
}

template <bool INJECT>
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_rk_aviary_step(const __grid_constant__ RocketParams p, const __grid_constant__ RngParams rng, float* __restrict__ st,
                     int32_t* __restrict__ ist, const float* __restrict__ setpoint, const float* __restrict__ noise, int n_steps,
                     uint32_t seq, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  RocketRegs s;
  rocket_load(st, ist, N, i, s);
#pragma unroll
  for (int k = 0; k < 7; ++k) s.sp[k] = __ldg(setpoint + 7 * i + k);
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_AVIARY, p.noise_loc, p.ratio);
  for (int k = 0; k < n_steps; ++k) rocket_aviary_step(p, s, nz, false);
  rocket_store(st, ist, N, i, s);
}

__global__ void __launch_bounds__(kBlock) k_rk_observe(const float* __restrict__ st, const int32_t* __restrict__ ist,
                                                       float* __restrict__ drone_state, float* __restrict__ aux,
                                                       uint8_t* __restrict__ contact, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  RocketRegs s;
  rocket_load(st, ist, N, i, s);
  float o[12], a[9];
  rocket_drone_state(s, o, a);
  if (drone_state)
    for (int k = 0; k < 12; ++k) drone_state[12 * i + k] = o[k];
  if (aux)
    for (int k = 0; k < 9; ++k) aux[9 * i + k] = a[k];
  if (contact) contact[i] = (s.flags & FLAG_CONTACT_ARRAY) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------------
// Rocket-Landing epilogue
// ---------------------------------------------------------------------------------------------------
constexpr int kLandObsMax = 30;
constexpr int kLandObsStride = 31;

// values of the previous compute_state (rocket_landing_env.py:140-144)
struct LandingPrev {
  float lat, z, gvz;     // |lin_pos[:2]|, lin_pos[2], ground_lin_vel[2]
  float ang_n, lin_n;    // |ang_vel|, |lin_vel|
};

__device__ __forceinline__ void landing_snapshot(const RocketRegs& s, LandingPrev& c) {
  float px = (float)s.px, py = (float)s.py;
  c.lat = sqrtf(px * px + py * py);
  c.z = (float)s.pz;
  c.gvz = (float)s.vz;  // ground_lin_vel = lin_vel @ rotation.T = the world-frame velocity
  c.ang_n = sqrtf(s.wx * s.wx + s.wy * s.wy + s.wz * s.wz);
  c.lin_n = sqrtf(s.vb.x * s.vb.x + s.vb.y * s.vb.y + s.vb.z * s.vb.z);
}

// compute_term_trunc_reward (rocket_landing_env.py:192-263 + rocket_base_env.py:295-325)
__device__ __forceinline__ void landing_term_trunc_reward(const LandingParams& l, RocketRegs& s, const LandingPrev& prev,
                                                          const LandingPrev& cur, int step_count, float& reward) {
  if (step_count > l.max_steps) s.flags |= FLAG_TRUNC;
  if ((s.flags & FLAG_CONTACT_GROUND) || cur.z < 0.0f) s.flags |= FLAG_COLLISION | FLAG_TERM;  // fatal_collision
  if (cur.lat > l.max_displacement || cur.z > l.ceiling) s.flags |= FLAG_OOB | FLAG_TERM;
  float roll, pitch;
  roll_pitch_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch);
  float tilt = sqrtf(roll * roll + pitch * pitch);
  if (!l.sparse_reward) {
    float lateral_progress = prev.lat - cur.lat;
    float vertical_progress = prev.z - cur.z;
    float lateral_distance = cur.lat + 0.1f;
    float decel = (cur.gvz - prev.gvz + 1.0f) * expf(-cur.z) * (cur.gvz < 0.0f ? 1.0f : -1.0f);
    reward += -0.3f + 0.3f / lateral_distance + 10.0f * lateral_progress + 0.2f * vertical_progress + 4.0f * decel - fabsf(s.wz) - tilt;
  }
  if (s.flags & FLAG_CONTACT_PAD) {
    s.flags |= FLAG_PAD_OBS;
    reward += 5.0f - 0.3f * fabsf(cur.gvz);
  } else {
    s.flags &= ~(uint32_t)FLAG_PAD_OBS;
    return;
  }
  if (prev.ang_n > 0.35f || prev.lin_n > 1.0f) { s.flags |= FLAG_TERM | FLAG_COLLISION; return; }
  if (prev.ang_n < 0.02f && prev.lin_n < 0.02f && tilt < 0.1f) { s.flags |= FLAG_TRUNC | FLAG_ENV_COMPLETE; reward += 3.0f; }
}

// compute_state (rocket_landing_env.py:129-190): attitude + action + aux + landing_pad_contact
__device__ __forceinline__ void landing_observation(const LandingParams& l, const RocketRegs& s, const float* action, bool pad_obs, float* obs) {
  float roll, pitch, yaw;
  euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
  int o = 0;
  obs[o++] = s.wx; obs[o++] = s.wy; obs[o++] = s.wz;
  if (l.angle_representation == 0) {
    obs[o++] = roll; obs[o++] = pitch; obs[o++] = yaw;
  } else {
    float ox, oy, oz, ow;
    quat_from_euler(roll, pitch, yaw, ox, oy, oz, ow);
    obs[o++] = ox; obs[o++] = oy; obs[o++] = oz; obs[o++] = ow;
  }
  obs[o++] = s.vb.x; obs[o++] = s.vb.y; obs[o++] = s.vb.z;
  obs[o++] = (float)s.px; obs[o++] = (float)s.py; obs[o++] = (float)s.pz;
  for (int k = 0; k < 7; ++k) obs[o++] = action[k];
  for (int k = 0; k < 4; ++k) obs[o++] = s.act[k];
  obs[o++] = s.ign; obs[o++] = s.fuel; obs[o++] = s.thr; obs[o++] = s.gim[0]; obs[o++] = s.gim[1];
  obs[o++] = pad_obs ? 1.0f : 0.0f;
}

// env.reset() for one env (rocket_landing_env.py:87-127, rocket_base_env.py:166-261)
// `pose` = the 6 start-pose words the caller read from start_pos / start_orn (ignored with randomize_drop)
template <bool INJECT>
__device__ __forceinline__ void landing_reset_env_inline(const RocketParams& p, const LandingParams& l, const RngParams& rng, const float* pose,
                                                  const float* __restrict__ noise, uint32_t seq, bool randomize, int64_t N, int64_t i,
                                                  RocketRegs& s) {
  float sx = pose[0], sy = pose[1], sz = pose[2];
  float r0 = pose[3], r1 = pose[4], r2 = pose[5];
  if (randomize) {  // options["randomize_drop"] (rocket_base_env.py:192-199), drawn from this env's Philox stream
    uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
    U4 a = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), seq, 5u << 24}, rng.k0, rng.k1);
    U4 b = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), seq, (5u << 24) | 1u}, rng.k0, rng.k1);
    float range = l.max_displacement * 0.1f;
    sx = range * (2.0f * u32_to_unit_open(a.x) - 1.0f);
    sy = range * (2.0f * u32_to_unit_open(a.y) - 1.0f);
    sz = l.ceiling * (0.8f + 0.1f * u32_to_unit_open(a.z));
    r0 = 0.3f * (2.0f * u32_to_unit_open(b.x) - 1.0f);
    r1 = 0.3f * (2.0f * u32_to_unit_open(b.y) - 1.0f);
    r2 = 0.3f * (2.0f * u32_to_unit_open(b.z) - 1.0f);
  }
  rocket_reset(p, s, sx, sy, sz, r0, r1, r2);
  // rocket_base_env.py:224-228: resetBaseVelocity is NOT followed by an update_state in the reference, so the
  // first warm-up substep evaluates drag / finlet forces with the stale (zero) body velocity; s.vb stays 0 here
  if (l.accelerate_drop) s.vz += (vreal)(-100.0);
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
  for (int k = 0; k < l.warmup_steps; ++k) rocket_aviary_step(p, s, nz, true);
  rocket_requantize(s);  // exactly what the state tensor / a spare record will hold
}

// The warm-up of the AUTORESET paths (spare build, inline fallback) is ONE out-of-line copy shared by every instantiation of
// k_land_step: a spare built by the <RANDACT = false> build launch must equal the warm-up a <RANDACT = true> step launch runs
// inline BIT FOR BIT, and two inlined copies of the same source are free to contract their multiply-adds differently.  State in
// and out by value (the caller's registers never have their address taken); the parameter blocks are the kernel's
// __grid_constant__ parameters, read through their address.
static __device__ __noinline__ RocketRegs landing_reset_env_shared(const RocketParams* p, const LandingParams* l, const RngParams* rng, float p0,
                                                                   float p1, float p2, float p3, float p4, float p5, uint32_t seq, int randomize,
                                                                   int64_t N, int64_t i) {
  RocketRegs s;
  const float pose[6] = {p0, p1, p2, p3, p4, p5};
  landing_reset_env_inline<false>(*p, *l, *rng, pose, nullptr, seq, randomize != 0, N, i, s);
  return s;
}

// 8 CTAs of one warp per SM are plenty at the batch sizes this env runs at (16 384 envs = 4.5 CTAs per SM): give the step the
// whole register file instead of spilling (contact response + wind + variable-mass composite: ~170 live registers)
constexpr int kLandBlocks = 8;

// spare post-reset states (pfb_tail_reset.cuh): an env-major record of 64 floats, the RK_* state words, then the spare header
enum { LSP_ROWS = 64 };
static_assert(SpareHdr<RK_ROWS>::END <= LSP_ROWS, "spare record too small");

template <bool INJECT, bool RANDACT, bool AUTORESET>
__global__ void __launch_bounds__(kBlock, kLandBlocks)
    k_land_step(const __grid_constant__ RocketParams p, const __grid_constant__ LandingParams l, const __grid_constant__ RngParams rng,
                float* __restrict__ st, int32_t* __restrict__ ist, float* __restrict__ actions, const float* __restrict__ noise,
                float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ term, uint8_t* __restrict__ trunc,
                uint8_t* __restrict__ info, const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                float* __restrict__ spare, const __grid_constant__ TailArgs a, int64_t N) {
  __shared__ float smem[kBlock * kLandObsStride];
  __shared__ uint8_t row_skip[kBlock];
  const int O = (l.angle_representation == 0 ? 12 : 13) + 17;
  const uint32_t step_seq = a.step_seq;
  TailWork sch = tail_schedule<1, AUTORESET>(a, N, threadIdx.x);
  const bool tail = sch.tail;
  bool skip = true;
  float* row = smem + threadIdx.x * kLandObsStride;
#pragma unroll 1
  for (; sch.t < sch.t_end; sch.t += sch.t_stride) {
    const int64_t i = tail_env<1>(a, sch, 0);
    RocketRegs s;
    float act[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    int step_count = 0;
    float rew = 0.0f;
    bool pad_obs = false;
    if (tail) {
      // env.reset(): normally a copy of the env's spare; build mode computes that spare; without a usable spare the
      // warm-up runs inline with the same episode number (which also keys a randomised drop)
      float* rec = spare ? spare + i * LSP_ROWS : nullptr;
      float pose[6];
#pragma unroll
      for (int k = 0; k < 3; ++k) { pose[k] = start_pos[3 * i + k]; pose[3 + k] = start_orn[3 * i + k]; }
      const SpareProbe sp = spare_probe<RK_ROWS>(a, rec, pose, !l.randomize_drop);  // a randomised drop does not read the start pose
      if (sp.hit) {
        rocket_load(rec, ist, N, i, s, 1, 0);
        s.flags = __float_as_uint(rec[SpareHdr<RK_ROWS>::FLAGS]);
      } else {
        if (a.build) spare_open<RK_ROWS>(rec, pose);
        s = landing_reset_env_shared(&p, &l, &rng, pose[0], pose[1], pose[2], pose[3], pose[4], pose[5], sp.episode, l.randomize_drop, N, i);
      }
      if (a.build) {
        rocket_store(rec, ist, N, i, s, false, 1, 0);
        spare_seal<RK_ROWS>(rec, s.flags, sp.episode);
        continue;
      }
      s.flags |= fresh_tag(step_seq);
    } else {
      rocket_load(st, ist, N, i, s);
      if (AUTORESET && tail_owns(s.flags, FLAG_TERM | FLAG_TRUNC, step_seq)) continue;
      s.flags &= ~(uint32_t)FLAG_FRESH_ANY;
      if (RANDACT) {  // rocket_base_env.py:82-107: [-1,1]^3, ignition {0..1}, throttle [0,1], gimbal [-1,1]^2
        uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
        U4 a = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), step_seq, (uint32_t)TAG_ACTION << 24}, rng.k0, rng.k1);
        U4 b = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), step_seq, ((uint32_t)TAG_ACTION << 24) | 1u}, rng.k0, rng.k1);
        act[0] = 2.0f * u32_to_unit_open(a.x) - 1.0f; act[1] = 2.0f * u32_to_unit_open(a.y) - 1.0f; act[2] = 2.0f * u32_to_unit_open(a.z) - 1.0f;
        act[3] = u32_to_unit_open(a.w); act[4] = u32_to_unit_open(b.x);
        act[5] = 2.0f * u32_to_unit_open(b.y) - 1.0f; act[6] = 2.0f * u32_to_unit_open(b.z) - 1.0f;
        for (int k = 0; k < 7; ++k) actions[7 * i + k] = act[k];
      } else {
#pragma unroll
        for (int k = 0; k < 7; ++k) act[k] = __ldg(actions + 7 * i + k);
      }
#pragma unroll
      for (int k = 0; k < 7; ++k) s.sp[k] = act[k];
      step_count = ist[(int64_t)RI_STEP * N + i];
      auto nz = make_noise<INJECT>(noise, N, i, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
      LandingPrev prev, cur;
      landing_snapshot(s, cur);  // the values of the last compute_state are the state we just loaded
      pad_obs = (s.flags & FLAG_PAD_OBS) != 0;
#pragma unroll 1
      for (int k = 0; k < l.env_step_ratio; ++k) {
        if (s.flags & (FLAG_TERM | FLAG_TRUNC)) break;
        rocket_aviary_step(p, s, nz, true);
        prev = cur;
        landing_snapshot(s, cur);
        // compute_state runs BEFORE compute_term_trunc_reward: the observation carries landing_pad_contact
        // as it stood after the previous Aviary step
        pad_obs = (s.flags & FLAG_PAD_OBS) != 0;
        landing_term_trunc_reward(l, s, prev, cur, step_count, rew);
      }
      step_count += 1;
    }
    landing_observation(l, s, act, pad_obs, row);
    rocket_store(st, ist, N, i, s);
    ist[(int64_t)RI_STEP * N + i] = step_count;
    reward[i] = rew;
    term[i] = (s.flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (s.flags & FLAG_TRUNC) ? 1 : 0;
    if (info) info[i] = (uint8_t)(((s.flags & FLAG_OOB) ? 1 : 0) | ((s.flags & FLAG_COLLISION) ? 2 : 0) | ((s.flags & FLAG_ENV_COMPLETE) ? 4 : 0));
    if (tail) {
      float* dst = obs + i * O;
      for (int k = 0; k < O; ++k) dst[k] = row[k];
    } else {
      skip = false;
      if (AUTORESET) append_done(a, sch, __activemask(), (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0, i);
    }
  }
  if (tail) return;
  flush_obs_tile<kLandObsStride>(smem, row_skip, skip, obs, sch, O, N);
}

template <bool INJECT>
__global__ void __launch_bounds__(kBlock)
    k_land_reset(const __grid_constant__ RocketParams p, const __grid_constant__ LandingParams l, const __grid_constant__ RngParams rng,
                 float* __restrict__ st, int32_t* __restrict__ ist, const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                 const uint8_t* __restrict__ mask, const float* __restrict__ noise, float* __restrict__ obs, uint32_t seq, int randomize,
                 int64_t N) {
  __shared__ float smem[kBlock * kLandObsStride];
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  const int O = (l.angle_representation == 0 ? 12 : 13) + 17;
  RocketRegs s;
  const float pose[6] = {start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1], start_orn[3 * i + 2]};
  landing_reset_env_inline<INJECT>(p, l, rng, pose, noise, seq, randomize != 0, N, i, s);
  const float zero[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float* row = smem + threadIdx.x * kLandObsStride;
  landing_observation(l, s, zero, false, row);
  rocket_store(st, ist, N, i, s);
  ist[(int64_t)RI_STEP * N + i] = 0;
  if (obs)
    for (int k = 0; k < O; ++k) obs[i * O + k] = row[k];
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
int rk_reset(PfbContext* h, const uint8_t* mask, cudaStream_t s) {
  k_rk_reset<<<grid_for(h->n), kBlock, 0, s>>>(h->rk, h->buf.state, h->buf.istate, h->buf.setpoint, h->buf.start_pos, h->buf.start_orn, mask, h->n);
  LAUNCH_CHECK(h);
  if (!mask) h->mode = 0;
  return 0;
}

int rk_set_mode(PfbContext* h, int mode, cudaStream_t s) {
  (void)s;
  if (mode != 0)  // base_drone.py:252-255
    return fail("`mode` must be either 0 or be registered in self.registered_controllers.keys()=dict_keys([]), got %d.", mode);
  h->mode = 0;
  return 0;
}

int rk_set_velocity(PfbContext* h, const float* lin, const float* ang, cudaStream_t s) {
  k_rk_set_velocity<<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, lin, ang, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

int rk_aviary_step(PfbContext* h, int n_steps, const float* noise, cudaStream_t s) {
  const uint32_t seq = (uint32_t)h->aviary_seq++;
  const int g = grid_for(h->n);
  if (noise) k_rk_aviary_step<true><<<g, kBlock, 0, s>>>(h->rk, h->rng, h->buf.state, h->buf.istate, h->buf.setpoint, noise, n_steps, seq, h->n);
  else k_rk_aviary_step<false><<<g, kBlock, 0, s>>>(h->rk, h->rng, h->buf.state, h->buf.istate, h->buf.setpoint, nullptr, n_steps, seq, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

int rk_observe(PfbContext* h, cudaStream_t s) {
  k_rk_observe<<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, h->buf.drone_state, h->buf.aux_state, h->buf.contact, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

// k_land_step for tail_env_step / tail_env_reset
static auto rk_step_launch(PfbContext* h, float* actions, const float* noise) {
  return [=](auto inject, auto randact, auto autoreset, int grid, cudaStream_t s, float* spare, const TailArgs& a) -> int {
    k_land_step<decltype(inject)::value, decltype(randact)::value, decltype(autoreset)::value><<<grid, kBlock, 0, s>>>(
        h->rk, h->land, h->rng, h->buf.state, h->buf.istate, actions, noise, h->buf.obs, h->buf.reward, h->buf.term, h->buf.trunc, h->buf.info,
        h->buf.start_pos, h->buf.start_orn, spare, a, h->n);
    return 0;
  };
}

int rk_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s) {
  // an explicit env.reset() honours the bound start_pos / start_orn unless randomize_drop is configured
  const int randomize = h->land.randomize_drop;
  auto reset = [&](uint32_t seq, int g) -> int {
    if (noise)
      k_land_reset<true><<<g, kBlock, 0, s>>>(h->rk, h->land, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn, mask, noise,
                                              h->buf.obs, seq, randomize, h->n);
    else
      k_land_reset<false><<<g, kBlock, 0, s>>>(h->rk, h->land, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn, mask,
                                               nullptr, h->buf.obs, seq, randomize, h->n);
    return 0;
  };
  return tail_env_reset(h, mask, s, reset, rk_step_launch(h, h->buf.setpoint, nullptr));
}

int rk_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s) {
  return tail_env_step(h, noise, randact, s, rk_step_launch(h, actions, noise));
}
