// pfb_fixedwing.cu — Fixedwing kernels (Aviary surface + Fixedwing-Waypoints env) and their launchers.
// Same structure as the QuadX kernels in pfb_lib.cu: one thread = one env, state in registers between a
// coalesced SoA load and store, obs staged through shared memory, NEXT_STEP autoreset by tail CTAs.
#include <cmath>
#include <cstring>

#include "pfb_context.h"
#include "pfb_noise.cuh"
#include "pfb_tail_reset.cuh"

using namespace pfb;

#include "pfb_fixedwing_host.h"

int fw_build_params(const PfbModel& m, const PfbEnvConfig* env, FixedwingParams& p, WaypointParams& w) {
  return fw_build_params_impl(m, env, p, w);
}

static inline int fw_setpoint_dim(const PfbContext* h) { return h->env.env_kind == PFB_ENV_NONE ? 6 : 4; }
int fw_state_rows() { return FW_ROWS; }
int fw_istate_rows() { return FI_ROWS; }
int fw_obs_dim(const PfbContext* h) { return (h->wp.angle_representation == 0 ? 22 : 23) + 3 * h->wp.num_targets; }

// ---------------------------------------------------------------------------------------------------
// kernels — Aviary surface
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock) k_fw_reset(const __grid_constant__ FixedwingParams p, float* __restrict__ st,
                                                     int32_t* __restrict__ ist, float* __restrict__ setpoint,
                                                     const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                                                     const uint8_t* __restrict__ mask, int sp_dim, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  FixedwingRegs s;
  fixedwing_reset(p, s, start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1],
                  start_orn[3 * i + 2]);
  fixedwing_store(st, ist, N, i, s);
  ist[(int64_t)FI_STEP * N + i] = 0;
  if (setpoint)  // the caller's buffer is [N][sp_dim]: 6 on the Aviary surface, 4 behind an env
    for (int k = 0; k < sp_dim; ++k) setpoint[(int64_t)sp_dim * i + k] = 0.0f;
}

template <int MODE, bool INJECT>
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_fw_aviary_step(const __grid_constant__ FixedwingParams p, const __grid_constant__ RngParams rng, float* __restrict__ st,
                     int32_t* __restrict__ ist, const float* __restrict__ setpoint, const float* __restrict__ noise,
                     int n_steps, uint32_t seq, int sp_dim, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  FixedwingRegs s;
  fixedwing_load(st, ist, N, i, s);
#pragma unroll
  for (int k = 0; k < 6; ++k) s.sp[k] = k < sp_dim ? __ldg(setpoint + (int64_t)sp_dim * i + k) : 0.0f;
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_AVIARY, p.noise_loc, p.ratio);
  if (fixedwing_full_model(p)) {  // launch-uniform: all surfaces, no wind -> the one-basic-block substep (pfb_fixedwing.cuh)
    for (int k = 0; k < n_steps; ++k) fixedwing_aviary_step<MODE, true>(p, s, nz);
  } else {
    for (int k = 0; k < n_steps; ++k) fixedwing_aviary_step<MODE>(p, s, nz);
  }
  fixedwing_store(st, ist, N, i, s);
}

__global__ void __launch_bounds__(kBlock) k_fw_observe(const float* __restrict__ st, const int32_t* __restrict__ ist,
                                                       float* __restrict__ drone_state, float* __restrict__ aux,
                                                       uint8_t* __restrict__ contact, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  FixedwingRegs s;
  fixedwing_load(st, ist, N, i, s);
  float o[12], a[6];
  fixedwing_drone_state(s, o, a);
  if (drone_state)
    for (int k = 0; k < 12; ++k) drone_state[12 * i + k] = o[k];
  if (aux)
    for (int k = 0; k < 6; ++k) aux[6 * i + k] = a[k];
  if (contact) contact[i] = (s.flags & FLAG_CONTACT_ARRAY) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------------
// Fixedwing-Waypoints epilogue
// ---------------------------------------------------------------------------------------------------
constexpr int kWpObsMax = 23 + 3 * kMaxTargets;
constexpr int kWpObsStride = kWpObsMax | 1;

// WaypointHandler.reset (waypoint_handler.py:53-83): polar sampling of the targets, on-device Philox stream
// Target words are addressed as tb[row * ts]: tb = st + i, ts = N for the field-major state tensor, tb = the env's spare
// record, ts = 1 while a spare is being built.
__device__ __forceinline__ void wp_sample_targets(const WaypointParams& w, const RngParams& rng, int64_t i, uint32_t seq,
                                                  float* __restrict__ tb, int64_t ts) {
  uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
  for (int k = 0; k < w.num_targets; ++k) {
    U4 r = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), seq, (4u << 24) | (uint32_t)k}, rng.k0, rng.k1);
    float theta = 6.28318530717958647692f * u32_to_unit_open(r.x);
    float phi = 6.28318530717958647692f * u32_to_unit_open(r.y);
    float dist = 1.0f + (w.dome * 0.9f - 1.0f) * u32_to_unit_open(r.z);
    float st_, ct, sp, cp;
    sincos_f(theta, st_, ct);
    sincos_f(phi, sp, cp);
    float z = fabsf(dist * cp);
    tb[(int64_t)(FW_TARGETS + 3 * k + 0) * ts] = dist * sp * ct;
    tb[(int64_t)(FW_TARGETS + 3 * k + 1) * ts] = dist * sp * st_;
    tb[(int64_t)(FW_TARGETS + 3 * k + 2) * ts] = z > w.min_height ? z : w.min_height;
  }
}

struct WpState {
  float t0x, t0y, t0z;  // next target
  float new_dist;       // WaypointHandler.new_distance
  int first;            // targets reached so far == index of the next target (the list is never shifted)
  bool reached_now;     // a target was reached on the most recent Aviary step
};

__device__ __forceinline__ void wp_load_target0(const float* __restrict__ tb, int64_t ts, WpState& wp) {
  wp.t0x = tb[(int64_t)(FW_TARGETS + 3 * wp.first + 0) * ts];
  wp.t0y = tb[(int64_t)(FW_TARGETS + 3 * wp.first + 1) * ts];
  wp.t0z = tb[(int64_t)(FW_TARGETS + 3 * wp.first + 2) * ts];
}

// compute_state's waypoint part (waypoint_handler.py:120-157): old <- new, new <- |target0 - pos|
__device__ __forceinline__ float wp_update_distance(const FixedwingRegs& s, WpState& wp) {
  float old = wp.new_dist;
  float dx = wp.t0x - (float)s.px, dy = wp.t0y - (float)s.py, dz = wp.t0z - (float)s.pz;
  wp.new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
  return old;
}

// fixedwing_base_env.py:226-244 + fixedwing_waypoints_env.py:169-190
__device__ __forceinline__ void wp_term_trunc_reward(const WaypointParams& w, FixedwingRegs& s, WpState& wp, float old_dist,
                                                     int step_count, float& reward, const float* __restrict__ tb, int64_t ts) {
  if (step_count > w.max_steps) s.flags |= FLAG_TRUNC;
  if (s.flags & FLAG_CONTACT_ARRAY) { reward = -100.0f; s.flags |= FLAG_COLLISION | FLAG_TERM; }
  float px = (float)s.px, py = (float)s.py, pz = (float)s.pz;
  if (px * px + py * py + pz * pz > w.dome2) { reward = -100.0f; s.flags |= FLAG_OOB | FLAG_TERM; }
  if (!w.sparse_reward) {
    float progress = (isinf(old_dist) || isinf(wp.new_dist)) ? 0.0f : old_dist - wp.new_dist;
    reward += fmaxf(3.0f * progress, 0.0f);
    reward += 1.0f / wp.new_dist;
  }
  wp.reached_now = false;
  if (wp.new_dist < w.goal_reach_distance) {  // target_reached (no yaw targets for the fixedwing)
    reward = 100.0f;
    wp.first += 1;  // advance_targets (waypoint_handler.py:176-185): the list head moves, nothing is copied
    wp.reached_now = true;
    if (wp.first == w.num_targets) s.flags |= FLAG_TRUNC | FLAG_ENV_COMPLETE;
    else wp_load_target0(tb, ts, wp);
  }
}

// compute_state (fixedwing_waypoints_env.py:121-167): attitude + action + aux + body-frame target deltas
__device__ __forceinline__ void wp_observation(const WaypointParams& w, const FixedwingRegs& s, const float* action, int first,
                                               const float* __restrict__ tb, int64_t ts, float* obs) {
  const float x = (float)s.qx, y = (float)s.qy, z = (float)s.qz, qw = (float)s.qw;
  float roll, pitch, yaw;
  euler_from_quat(x, y, z, qw, roll, pitch, yaw);
  int o = 0;
  obs[o++] = s.wx; obs[o++] = s.wy; obs[o++] = s.wz;
  if (w.angle_representation == 0) {
    obs[o++] = roll; obs[o++] = pitch; obs[o++] = yaw;
  } else {
    float ox, oy, oz, ow;
    quat_from_euler(roll, pitch, yaw, ox, oy, oz, ow);
    obs[o++] = ox; obs[o++] = oy; obs[o++] = oz; obs[o++] = ow;
  }
  obs[o++] = s.vb.x; obs[o++] = s.vb.y; obs[o++] = s.vb.z;
  obs[o++] = (float)s.px; obs[o++] = (float)s.py; obs[o++] = (float)s.pz;
  for (int k = 0; k < 4; ++k) obs[o++] = action[k];
  for (int k = 0; k < kMaxSurfaces; ++k) obs[o++] = s.act[k];
  obs[o++] = s.thr;
  // target_deltas = (targets - lin_pos) @ R  (waypoint_handler.py:139-142): body-frame deltas
  const Rot<rreal>& R = s.R;
  for (int k = 0; k < w.num_targets; ++k) {
    float bx = 0.f, by = 0.f, bz = 0.f;
    if (first + k < w.num_targets) {  // remaining targets first, zero padding after
      float dx = tb[(int64_t)(FW_TARGETS + 3 * (first + k) + 0) * ts] - (float)s.px;
      float dy = tb[(int64_t)(FW_TARGETS + 3 * (first + k) + 1) * ts] - (float)s.py;
      float dz = tb[(int64_t)(FW_TARGETS + 3 * (first + k) + 2) * ts] - (float)s.pz;
      bx = (float)R.m00 * dx + (float)R.m10 * dy + (float)R.m20 * dz;
      by = (float)R.m01 * dx + (float)R.m11 * dy + (float)R.m21 * dz;
      bz = (float)R.m02 * dx + (float)R.m12 * dy + (float)R.m22 * dz;
    }
    obs[o++] = bx; obs[o++] = by; obs[o++] = bz;
  }
}

// env.reset() for one env (fixedwing_waypoints_env.py:102-119, fixedwing_base_env.py:126-192); `pose` = the 6 start-pose
// words the caller read (and, when building a spare, recorded), targets go to tb / ts
template <bool INJECT>
__device__ __forceinline__ void wp_reset_env(const FixedwingParams& p, const WaypointParams& w, const RngParams& rng, const float* pose,
                                             const float* __restrict__ reset_targets, const float* __restrict__ noise, uint32_t seq,
                                             int64_t N, int64_t i, float* __restrict__ tb, int64_t ts, FixedwingRegs& s, WpState& wp) {
  fixedwing_reset(p, s, pose[0], pose[1], pose[2], pose[3], pose[4], pose[5]);
  if (reset_targets) {
    for (int k = 0; k < 3 * w.num_targets; ++k) tb[(int64_t)(FW_TARGETS + k) * ts] = reset_targets[(int64_t)i * 3 * w.num_targets + k];
  } else {
    wp_sample_targets(w, rng, i, seq, tb, ts);
  }
  wp.first = 0;
  wp.reached_now = false;
  wp.new_dist = INFINITY;
  wp_load_target0(tb, ts, wp);
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
  for (int k = 0; k < w.warmup_steps; ++k) fixedwing_aviary_step<0>(p, s, nz);
  fixedwing_requantize(s);             // exactly what the state tensor / a spare record will hold
  (void)wp_update_distance(s, wp);     // end_reset -> compute_state
}

// spare post-reset states (pfb_tail_reset.cuh): an env-major record of 64 floats, the FW_* state words INCLUDING the
// episode's targets and new_distance, then the spare header
enum { WSP_ROWS = 64 };
static_assert(SpareHdr<FW_ROWS>::END <= WSP_ROWS, "spare record too small");

// One thread per aircraft.  Splitting the five lifting surfaces over L lanes per aircraft was measured slower on B200 (16 384
// envs, L2 flushed, us per env step: L = 1: 37.5, L = 2: 39.3, L = 4: 41.8, L = 8: 58.6): the surfaces are only ~55 % of a
// substep's instructions, the rest is replicated in every lane of a group (DESIGN.md §9).

template <bool INJECT, bool RANDACT, bool AUTORESET>
__global__ void __launch_bounds__(kBlock, kAeroBlocks)
    k_fwwp_step(const __grid_constant__ FixedwingParams p, const __grid_constant__ WaypointParams w,
                const __grid_constant__ RngParams rng, float* __restrict__ st, int32_t* __restrict__ ist,
                float* __restrict__ actions, const float* __restrict__ noise, float* __restrict__ obs, float* __restrict__ reward,
                uint8_t* __restrict__ term, uint8_t* __restrict__ trunc, uint8_t* __restrict__ info,
                const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ spare, const __grid_constant__ TailArgs a, int64_t N) {
  __shared__ float smem[kBlock * kWpObsStride];
  __shared__ uint8_t row_skip[kBlock];
  const int O = (w.angle_representation == 0 ? 22 : 23) + 3 * w.num_targets;
  const uint32_t step_seq = a.step_seq;
  TailWork sch = tail_schedule<1, AUTORESET>(a, N, threadIdx.x);
  const bool tail = sch.tail;
  bool skip = true;
  float* row = smem + threadIdx.x * kWpObsStride;
#pragma unroll 1
  for (; sch.t < sch.t_end; sch.t += sch.t_stride) {
    const int64_t i = tail_env<1>(a, sch, 0);
    FixedwingRegs s;
    WpState wp;
    float act[4] = {0.f, 0.f, 0.f, 0.f};
    int step_count = 0;
    float rew = 0.0f;
    float* tb = st + i;  // where this env's targets live (field-major state rows, or the spare record being built)
    int64_t ts = N;
    if (tail) {
      // env.reset(): normally a copy of the env's spare (state, targets, new_distance of the NEXT episode); build mode
      // computes that spare; without a usable spare the warm-up runs inline with the same episode number
      float* rec = spare ? spare + i * WSP_ROWS : nullptr;
      float pose[6];
#pragma unroll
      for (int k = 0; k < 3; ++k) { pose[k] = start_pos[3 * i + k]; pose[3 + k] = start_orn[3 * i + k]; }
      const SpareProbe sp = spare_probe<FW_ROWS>(a, rec, pose, true);
      if (sp.hit) {
        fixedwing_load(rec, ist, N, i, s, 1, 0);
        s.flags = __float_as_uint(rec[SpareHdr<FW_ROWS>::FLAGS]);
        for (int k = 0; k < 3 * w.num_targets; ++k) tb[(int64_t)(FW_TARGETS + k) * ts] = rec[FW_TARGETS + k];
        wp.first = 0;
        wp.reached_now = false;
        wp.new_dist = rec[FW_DIST];
      } else {
        if (a.build) {
          spare_open<FW_ROWS>(rec, pose);
          tb = rec;
          ts = 1;
        }
        wp_reset_env<false>(p, w, rng, pose, nullptr, nullptr, sp.episode, N, i, tb, ts, s, wp);
      }
      if (a.build) {
        fixedwing_store(rec, ist, N, i, s, false, 1, 0);
        rec[FW_DIST] = wp.new_dist;
        spare_seal<FW_ROWS>(rec, s.flags, sp.episode);
        continue;
      }
      s.flags |= fresh_tag(step_seq);
    } else {
      fixedwing_load(st, ist, N, i, s);
      if (AUTORESET && tail_owns(s.flags, FLAG_TERM | FLAG_TRUNC, step_seq)) continue;
      s.flags &= ~(uint32_t)FLAG_FRESH_ANY;
      if (RANDACT) {
        uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
        U4 r = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), step_seq, (uint32_t)TAG_ACTION << 24}, rng.k0, rng.k1);
        act[0] = 2.0f * u32_to_unit_open(r.x) - 1.0f; act[1] = 2.0f * u32_to_unit_open(r.y) - 1.0f;
        act[2] = 2.0f * u32_to_unit_open(r.z) - 1.0f; act[3] = 2.0f * u32_to_unit_open(r.w) - 1.0f;
        reinterpret_cast<float4*>(actions)[i] = make_float4(act[0], act[1], act[2], act[3]);
      } else {
        float4 a4 = __ldg(reinterpret_cast<const float4*>(actions) + i);
        act[0] = a4.x; act[1] = a4.y; act[2] = a4.z; act[3] = a4.w;
      }
      // fixedwing_base_env.py:257-261: the throttle channel is remapped from [-1, 1] to [0, 1]
      s.sp[0] = act[0]; s.sp[1] = act[1]; s.sp[2] = act[2]; s.sp[3] = act[3] * 0.5f + 0.5f;
      step_count = ist[(int64_t)FI_STEP * N + i];
      wp.first = ist[(int64_t)FI_NTARGETS * N + i];
      wp.reached_now = false;
      wp.new_dist = st[(int64_t)FW_DIST * N + i];
      wp_load_target0(tb, ts, wp);
      rew = -0.1f;
      auto nz = make_noise<INJECT>(noise, N, i, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
      const bool full = fixedwing_full_model(p);
#pragma unroll 1
      for (int k = 0; k < w.env_step_ratio; ++k) {
        if (s.flags & (FLAG_TERM | FLAG_TRUNC)) break;
        if (full) fixedwing_aviary_step<0, true>(p, s, nz);
        else fixedwing_aviary_step<0>(p, s, nz);
        float old = wp_update_distance(s, wp);
        wp_term_trunc_reward(w, s, wp, old, step_count, rew, tb, ts);
      }
      step_count += 1;
    }
    // the reference builds the observation in compute_state, BEFORE compute_term_trunc_reward advances the
    // target list: a target reached on the last Aviary step is still the head of the reported list
    wp_observation(w, s, act, wp.first - (wp.reached_now ? 1 : 0), tb, ts, row);
    fixedwing_store(st, ist, N, i, s);
    st[(int64_t)FW_DIST * N + i] = wp.new_dist;
    ist[(int64_t)FI_STEP * N + i] = step_count;
    ist[(int64_t)FI_NTARGETS * N + i] = wp.first;
    reward[i] = rew;
    term[i] = (s.flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (s.flags & FLAG_TRUNC) ? 1 : 0;
    if (info)
      info[i] = (uint8_t)(((s.flags & FLAG_OOB) ? 1 : 0) | ((s.flags & FLAG_COLLISION) ? 2 : 0) | ((s.flags & FLAG_ENV_COMPLETE) ? 4 : 0) |
                          (wp.first << 3));
    if (tail) {
      float* dst = obs + i * O;
      for (int k = 0; k < O; ++k) dst[k] = row[k];
    } else {
      skip = false;
      if (AUTORESET) append_done(a, sch, __activemask(), (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0, i);
    }
  }
  if (tail) return;
  flush_obs_tile<kWpObsStride>(smem, row_skip, skip, obs, sch, O, N);
}

template <bool INJECT>
__global__ void __launch_bounds__(kBlock)
    k_fwwp_reset(const __grid_constant__ FixedwingParams p, const __grid_constant__ WaypointParams w,
                 const __grid_constant__ RngParams rng, float* __restrict__ st, int32_t* __restrict__ ist,
                 const float* __restrict__ start_pos, const float* __restrict__ start_orn, const float* __restrict__ reset_targets,
                 const uint8_t* __restrict__ mask, const float* __restrict__ noise, float* __restrict__ obs, uint32_t seq, int64_t N) {
  __shared__ float smem[kBlock * kWpObsStride];
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  const int O = (w.angle_representation == 0 ? 22 : 23) + 3 * w.num_targets;
  FixedwingRegs s;
  WpState wp;
  const float pose[6] = {start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1], start_orn[3 * i + 2]};
  wp_reset_env<INJECT>(p, w, rng, pose, reset_targets, noise, seq, N, i, st + i, N, s, wp);
  const float zero[4] = {0.f, 0.f, 0.f, 0.f};
  float* row = smem + threadIdx.x * kWpObsStride;
  wp_observation(w, s, zero, wp.first, st + i, N, row);
  fixedwing_store(st, ist, N, i, s);
  st[(int64_t)FW_DIST * N + i] = wp.new_dist;
  ist[(int64_t)FI_STEP * N + i] = 0;
  ist[(int64_t)FI_NTARGETS * N + i] = wp.first;
  if (obs)
    for (int k = 0; k < O; ++k) obs[i * O + k] = row[k];
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
int fw_reset(PfbContext* h, const uint8_t* mask, cudaStream_t s) {
  k_fw_reset<<<grid_for(h->n), kBlock, 0, s>>>(h->fw, h->buf.state, h->buf.istate, h->buf.setpoint, h->buf.start_pos,
                                               h->buf.start_orn, mask, fw_setpoint_dim(h), h->n);
  LAUNCH_CHECK(h);
  if (!mask) h->mode = 0;
  return 0;
}

int fw_set_mode(PfbContext* h, int mode, cudaStream_t s) {
  if (mode < -1 || mode > 0)  // fixedwing.py:216-219
    return fail("`mode` must be between -1 and 0 or be registered in self.registered_controllers.keys()=dict_keys([]), got %d.", mode);
  if (mode == -1 && fw_setpoint_dim(h) < 6) return fail("mode -1 needs the 6-wide setpoint buffer of the Aviary surface");
  CUDA_OK(cudaMemsetAsync(h->buf.setpoint, 0, (size_t)h->n * fw_setpoint_dim(h) * sizeof(float), s));  // fixedwing.py:224-227
  h->mode = mode;
  return 0;
}

int fw_aviary_step(PfbContext* h, int n_steps, const float* noise, cudaStream_t s) {
  const uint32_t seq = (uint32_t)h->aviary_seq++;
  const int g = grid_for(h->n);
#define FW_ARGS h->fw, h->rng, h->buf.state, h->buf.istate, h->buf.setpoint, noise, n_steps, seq, fw_setpoint_dim(h), h->n
  if (h->mode == 0) {
    if (noise) k_fw_aviary_step<0, true><<<g, kBlock, 0, s>>>(FW_ARGS);
    else k_fw_aviary_step<0, false><<<g, kBlock, 0, s>>>(FW_ARGS);
  } else {
    if (noise) k_fw_aviary_step<-1, true><<<g, kBlock, 0, s>>>(FW_ARGS);
    else k_fw_aviary_step<-1, false><<<g, kBlock, 0, s>>>(FW_ARGS);
  }
#undef FW_ARGS
  LAUNCH_CHECK(h);
  return 0;
}

int fw_observe(PfbContext* h, cudaStream_t s) {
  k_fw_observe<<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, h->buf.drone_state, h->buf.aux_state, h->buf.contact, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

// k_fwwp_step for tail_env_step / tail_env_reset
static auto fw_step_launch(PfbContext* h, float* actions, const float* noise) {
  return [=](auto inject, auto randact, auto autoreset, int grid, cudaStream_t s, float* spare, const TailArgs& a) -> int {
    k_fwwp_step<decltype(inject)::value, decltype(randact)::value, decltype(autoreset)::value><<<grid, kBlock, 0, s>>>(
        h->fw, h->wp, h->rng, h->buf.state, h->buf.istate, actions, noise, h->buf.obs, h->buf.reward, h->buf.term, h->buf.trunc, h->buf.info,
        h->buf.start_pos, h->buf.start_orn, spare, a, h->n);
    return 0;
  };
}

int fw_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s) {
  auto reset = [&](uint32_t seq, int g) -> int {
    if (noise)
      k_fwwp_reset<true><<<g, kBlock, 0, s>>>(h->fw, h->wp, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn,
                                              h->buf.reset_targets, mask, noise, h->buf.obs, seq, h->n);
    else
      k_fwwp_reset<false><<<g, kBlock, 0, s>>>(h->fw, h->wp, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn,
                                               h->buf.reset_targets, mask, nullptr, h->buf.obs, seq, h->n);
    return 0;
  };
  return tail_env_reset(h, mask, s, reset, fw_step_launch(h, h->buf.setpoint, nullptr));
}

int fw_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s) {
  return tail_env_step(h, noise, randact, s, fw_step_launch(h, actions, noise));
}
