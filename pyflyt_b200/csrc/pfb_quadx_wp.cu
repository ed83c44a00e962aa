// pfb_quadx_wp.cu — QuadX-Waypoints: QuadXWaypointsEnv.step / reset for every env, one launch.
//
// Reference (under /root/reference/PyFlyt/):
//   gym_envs/quadx_envs/quadx_waypoints_env.py:105-212  reset, compute_state, compute_term_trunc_reward
//   gym_envs/quadx_envs/quadx_base_env.py:149-301       begin_reset / end_reset / step / base termination rules
//   gym_envs/utils/waypoint_handler.py:53-213           target sampling, body-frame deltas, yaw targets, reached / advance
// The vehicle part is pfb_quadx.cuh (all nine flight modes); this file adds the waypoint epilogue.  Same launch
// structure as k_hover_step before its reset pipeline: regular CTAs own one env per thread, "tail" CTAs at the front of
// the grid reset the envs that finished on the previous launch (NEXT_STEP autoreset, inline warm-up).
#include "pfb_noise.cuh"
#include "pfb_quadx.cuh"
#include "pfb_tail_reset.cuh"

using namespace pfb;

// extra state rows behind the QuadX rows: WaypointHandler.new_distance, yaw_error_scalar, targets (x, y, z, yaw)
enum { QW_DIST = QX_ROWS, QW_YAWERR = QX_ROWS + 1, QW_TARGETS = QX_ROWS + 2, QW_ROWS = QX_ROWS + 2 + 4 * kMaxTargets };
enum { QWI_NTARGETS = QI_ROWS, QWI_ROWS = QI_ROWS + 1 };
enum { FLAG_QW_COMPLETE = 64 };
constexpr int kQwObsMax = 21 + 4 * kMaxTargets;
constexpr int kQwObsStride = kQwObsMax | 1;

int qwp_state_rows() { return QW_ROWS; }
int qwp_istate_rows() { return QWI_ROWS; }
int qwp_obs_dim(const PfbContext* h) { return (h->hover.angle_representation == 0 ? 20 : 21) + (h->qwp.use_yaw_targets ? 4 : 3) * h->qwp.num_targets; }

struct QwState {
  float t0x, t0y, t0z, t0yaw;  // next target
  float new_dist, yaw_err;     // WaypointHandler.new_distance / yaw_error_scalar
  int first;                   // targets reached so far == index of the next target (the list is never shifted)
  bool reached_now;            // a target was reached on the most recent Aviary step
};

// Target words are addressed as tb[row * ts]: tb = st + i, ts = N for the field-major state tensor, tb = the env's spare
// record, ts = 1 while a spare is being built.
__device__ __forceinline__ void qw_load_target0(const float* __restrict__ tb, int64_t ts, QwState& wp) {
  wp.t0x = tb[(int64_t)(QW_TARGETS + 4 * wp.first + 0) * ts];
  wp.t0y = tb[(int64_t)(QW_TARGETS + 4 * wp.first + 1) * ts];
  wp.t0z = tb[(int64_t)(QW_TARGETS + 4 * wp.first + 2) * ts];
  wp.t0yaw = tb[(int64_t)(QW_TARGETS + 4 * wp.first + 3) * ts];
}

__device__ __forceinline__ float wrap_pi(float e) {  // waypoint_handler.py:147-149
  const float pi = 3.14159265358979323846f;
  if (e > pi) e -= 2.0f * pi;
  if (e < -pi) e += 2.0f * pi;
  return e;
}

// WaypointHandler.reset (waypoint_handler.py:65-90): polar sampling of the targets, on-device Philox stream
__device__ __forceinline__ void qw_sample_targets(const QxWaypointParams& w, const RngParams& rng, int64_t i, uint32_t seq,
                                                  float* __restrict__ tb, int64_t ts) {
  uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
  for (int k = 0; k < w.num_targets; ++k) {
    U4 r = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), seq, (4u << 24) | (uint32_t)k}, rng.k0, rng.k1);
    const float two_pi = 6.28318530717958647692f;
    float theta = two_pi * u32_to_unit_open(r.x), phi = two_pi * u32_to_unit_open(r.y);
    float dist = 1.0f + (w.dome * 0.9f - 1.0f) * u32_to_unit_open(r.z);
    float st_, ct, sp, cp;
    sincos_f(theta, st_, ct);
    sincos_f(phi, sp, cp);
    float z = fabsf(dist * cp);
    tb[(int64_t)(QW_TARGETS + 4 * k + 0) * ts] = dist * sp * ct;
    tb[(int64_t)(QW_TARGETS + 4 * k + 1) * ts] = dist * sp * st_;
    tb[(int64_t)(QW_TARGETS + 4 * k + 2) * ts] = z > w.min_height ? z : w.min_height;
    tb[(int64_t)(QW_TARGETS + 4 * k + 3) * ts] = -3.14159265358979323846f + two_pi * u32_to_unit_open(r.w);
  }
}

// compute_state's waypoint part (waypoint_handler.py:120-157): old <- new, new <- |target0 - pos|, yaw error
__device__ __forceinline__ float qw_update_distance(const QxWaypointParams& w, const QuadXRegs& s, QwState& wp) {
  float old = wp.new_dist;
  float dx = wp.t0x - (float)s.px, dy = wp.t0y - (float)s.py, dz = wp.t0z - (float)s.pz;
  wp.new_dist = sqrtf(dx * dx + dy * dy + dz * dz);
  if (w.use_yaw_targets) {
    float roll, pitch, yaw;
    euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
    wp.yaw_err = fabsf(wrap_pi(wp.t0yaw - yaw));
  }
  return old;
}

// quadx_base_env.py:251-266 + quadx_waypoints_env.py:183-212
__device__ __forceinline__ void qw_term_trunc_reward(const QxWaypointParams& w, QuadXRegs& s, QwState& wp, float old_dist, int step_count,
                                                     float& reward, const float* __restrict__ tb, int64_t ts) {
  if (step_count > w.max_steps) s.flags |= FLAG_TRUNC;
  if (s.flags & FLAG_CONTACT_ARRAY) { reward = -100.0f; s.flags |= FLAG_COLLISION | FLAG_TERM; }
  float px = (float)s.px, py = (float)s.py, pz = (float)s.pz;
  if (px * px + py * py + pz * pz > w.dome2) { reward = -100.0f; s.flags |= FLAG_OOB | FLAG_TERM; }
  if (!w.sparse_reward) {
    float progress = (isinf(old_dist) || isinf(wp.new_dist)) ? 0.0f : old_dist - wp.new_dist;
    reward += fmaxf(3.0f * progress, 0.0f);
    reward += 0.1f / wp.new_dist;
    reward -= 0.01f * s.wz * s.wz;  // yaw-rate penalty on env.state(0)[0][2]
  }
  wp.reached_now = false;
  bool reached = wp.new_dist < w.goal_reach_distance;
  if (reached && w.use_yaw_targets) reached = wp.yaw_err < w.goal_reach_angle;
  if (reached) {
    reward = 100.0f;
    wp.first += 1;  // advance_targets: the list head moves, nothing is copied
    wp.reached_now = true;
    if (wp.first == w.num_targets) s.flags |= FLAG_TRUNC | FLAG_QW_COMPLETE;
    else qw_load_target0(tb, ts, wp);
  }
}

// compute_state (quadx_waypoints_env.py:130-181): the Hover attitude block + body-frame target deltas (+ yaw errors)
__device__ __forceinline__ void qw_observation(const HoverParams& h, const QxWaypointParams& w, const QuadXRegs& s, const float* action,
                                               int first, const float* __restrict__ tb, int64_t ts, float* obs) {
  hover_observation(h, s, action, obs);
  int o = h.angle_representation == 0 ? 20 : 21;
  float yaw = 0.0f;
  if (w.use_yaw_targets) {
    float roll, pitch;
    euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
  }
  const Rot<rreal>& R = s.R;
  for (int k = 0; k < w.num_targets; ++k) {
    float bx = 0.f, by = 0.f, bz = 0.f, be = 0.f;
    if (first + k < w.num_targets) {  // remaining targets first, zero padding after
      const float* tk = tb + (int64_t)(QW_TARGETS + 4 * (first + k)) * ts;
      float dx = tk[0] - (float)s.px, dy = tk[ts] - (float)s.py, dz = tk[2 * ts] - (float)s.pz;
      bx = (float)R.m00 * dx + (float)R.m10 * dy + (float)R.m20 * dz;  // (targets - lin_pos) @ R
      by = (float)R.m01 * dx + (float)R.m11 * dy + (float)R.m21 * dz;
      bz = (float)R.m02 * dx + (float)R.m12 * dy + (float)R.m22 * dz;
      if (w.use_yaw_targets) be = wrap_pi(tk[3 * ts] - yaw);
    }
    obs[o++] = bx; obs[o++] = by; obs[o++] = bz;
    if (w.use_yaw_targets) obs[o++] = be;
  }
}

// env.reset() for one env (quadx_waypoints_env.py:105-128, quadx_base_env.py:149-212); `pose` = the 6 start-pose words the
// caller read (and, when building a spare, recorded); targets go to tb / ts
template <int MODE, bool INJECT>
__device__ __forceinline__ void qw_reset_env(const QuadXParams& p, const QxWaypointParams& w, const RngParams& rng, const float* pose,
                                             const float* __restrict__ reset_targets, const float* __restrict__ noise, uint32_t seq,
                                             int64_t N, int64_t i, float* __restrict__ tb, int64_t ts, QuadXRegs& s, QwState& wp) {
  quadx_reset(s, pose[0], pose[1], pose[2], pose[3], pose[4], pose[5]);
  if (reset_targets) {
    const int T = w.use_yaw_targets ? 4 : 3;
    for (int k = 0; k < w.num_targets; ++k)
      for (int c = 0; c < 4; ++c)
        tb[(int64_t)(QW_TARGETS + 4 * k + c) * ts] = c < T ? reset_targets[((int64_t)i * w.num_targets + k) * T + c] : 0.0f;
  } else {
    qw_sample_targets(w, rng, i, seq, tb, ts);
  }
  wp.first = 0;
  wp.reached_now = false;
  wp.new_dist = INFINITY;
  wp.yaw_err = 0.0f;
  qw_load_target0(tb, ts, wp);
  quadx_set_mode<MODE>(s);
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
  for (int k = 0; k < w.warmup_steps; ++k) quadx_aviary_step<MODE>(p, s, nz);
  quadx_requantize(s);                  // exactly what the state tensor / a spare record will hold
  (void)qw_update_distance(w, s, wp);  // end_reset -> compute_state
}

// spare post-reset states (pfb_tail_reset.cuh): an env-major record of 128 floats, the QW_* state words INCLUDING the
// episode's targets, new_distance and yaw error, then the spare header
enum { QSP_ROWS = 128 };
static_assert(SpareHdr<QW_ROWS>::END <= QSP_ROWS, "spare record too small");
int qwp_spare_rows() { return QSP_ROWS; }

template <int MODE, bool INJECT, bool RANDACT, bool AUTORESET>
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_qxwp_step(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ QxWaypointParams w,
                const __grid_constant__ RngParams rng, float* __restrict__ st, int32_t* __restrict__ ist, float* __restrict__ actions,
                const float* __restrict__ noise, float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ term,
                uint8_t* __restrict__ trunc, uint8_t* __restrict__ info, const float* __restrict__ start_pos,
                const float* __restrict__ start_orn, float* __restrict__ spare, const __grid_constant__ TailArgs a, int64_t N) {
  __shared__ float smem[kBlock * kQwObsStride];
  __shared__ uint8_t row_skip[kBlock];
  const int O = (h.angle_representation == 0 ? 20 : 21) + (w.use_yaw_targets ? 4 : 3) * w.num_targets;
  const uint32_t step_seq = a.step_seq;
  TailWork sch = tail_schedule<1, AUTORESET>(a, N, threadIdx.x);
  const bool tail = sch.tail;
  bool skip = true;
  float* row = smem + threadIdx.x * kQwObsStride;
#pragma unroll 1
  for (; sch.t < sch.t_end; sch.t += sch.t_stride) {
    const int64_t i = tail_env<1>(a, sch, 0);
    QuadXRegs s;
    QwState wp;
    float act[4] = {0.f, 0.f, 0.f, 0.f};
    int step_count = 0;
    float rew = 0.0f;
    float* tb = st + i;  // where this env's targets live (field-major state rows, or the spare record being built)
    int64_t ts = N;
    if (tail) {
      // env.reset(): normally a copy of the env's spare (state, targets, distances of the NEXT episode); build mode
      // computes that spare; without a usable spare the warm-up runs inline with the same episode number
      float* rec = spare ? spare + i * QSP_ROWS : nullptr;
      float pose[6];
#pragma unroll
      for (int k = 0; k < 3; ++k) { pose[k] = start_pos[3 * i + k]; pose[3 + k] = start_orn[3 * i + k]; }
      const SpareProbe sp = spare_probe<QW_ROWS>(a, rec, pose, true);
      if (sp.hit) {
        quadx_load<MODE>(rec, ist, N, i, s, 1, 0);
        s.flags = __float_as_uint(rec[SpareHdr<QW_ROWS>::FLAGS]);
#pragma unroll
        for (int k = 0; k < 4; ++k) { s.sp[k] = 0.0f; s.pwm[k] = rec[QX_PWM + k]; }
        for (int k = 0; k < 4 * w.num_targets; ++k) tb[(int64_t)(QW_TARGETS + k) * ts] = rec[QW_TARGETS + k];
        wp.first = 0;
        wp.reached_now = false;
        wp.new_dist = rec[QW_DIST];
        wp.yaw_err = rec[QW_YAWERR];
      } else {
        if (a.build) {
          spare_open<QW_ROWS>(rec, pose);
          tb = rec;
          ts = 1;
        }
        qw_reset_env<MODE, false>(p, w, rng, pose, nullptr, nullptr, sp.episode, N, i, tb, ts, s, wp);
      }
      if (a.build) {
        quadx_store<MODE>(rec, ist, N, i, s, false, 1, 0);
        rec[QW_DIST] = wp.new_dist;
        rec[QW_YAWERR] = wp.yaw_err;
        spare_seal<QW_ROWS>(rec, s.flags, sp.episode);
        continue;
      }
      s.flags |= fresh_tag(step_seq);
    } else {
      quadx_load<MODE>(st, ist, N, i, s);
      if (AUTORESET && tail_owns(s.flags, FLAG_TERM | FLAG_TRUNC, step_seq)) continue;
      s.flags &= ~(uint32_t)FLAG_FRESH_ANY;
      if (RANDACT) {  // uniform in the action box (quadx_base_env.py:79-102)
        uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
        U4 r = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), step_seq, (uint32_t)TAG_ACTION << 24}, rng.k0, rng.k1);
        const float pi = 3.14159265358979323846f;
        if (MODE == -1) {
          act[0] = 0.8f * u32_to_unit_open(r.x); act[1] = 0.8f * u32_to_unit_open(r.y);
          act[2] = 0.8f * u32_to_unit_open(r.z); act[3] = 0.8f * u32_to_unit_open(r.w);
        } else {
          act[0] = pi * (2.0f * u32_to_unit_open(r.x) - 1.0f); act[1] = pi * (2.0f * u32_to_unit_open(r.y) - 1.0f);
          act[2] = pi * (2.0f * u32_to_unit_open(r.z) - 1.0f); act[3] = 0.8f * u32_to_unit_open(r.w);
        }
        reinterpret_cast<float4*>(actions)[i] = make_float4(act[0], act[1], act[2], act[3]);
      } else {
        float4 a4 = __ldg(reinterpret_cast<const float4*>(actions) + i);
        act[0] = a4.x; act[1] = a4.y; act[2] = a4.z; act[3] = a4.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) s.sp[k] = act[k];
      step_count = ist[(int64_t)QI_STEP * N + i];
      wp.first = ist[(int64_t)QWI_NTARGETS * N + i];
      wp.reached_now = false;
      wp.new_dist = st[(int64_t)QW_DIST * N + i];
      wp.yaw_err = st[(int64_t)QW_YAWERR * N + i];
      if (wp.first < w.num_targets) qw_load_target0(tb, ts, wp);
      rew = -0.1f;
      auto nz = make_noise<INJECT>(noise, N, i, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
#pragma unroll 1
      for (int k = 0; k < w.env_step_ratio; ++k) {
        if (s.flags & (FLAG_TERM | FLAG_TRUNC)) break;
        quadx_aviary_step<MODE>(p, s, nz);
        float old = qw_update_distance(w, s, wp);
        qw_term_trunc_reward(w, s, wp, old, step_count, rew, tb, ts);
      }
      step_count += 1;
    }
    // the reference builds the observation in compute_state, BEFORE compute_term_trunc_reward advances the target list
    qw_observation(h, w, s, act, wp.first - (wp.reached_now ? 1 : 0), tb, ts, row);
    quadx_store<MODE>(st, ist, N, i, s);
    st[(int64_t)QW_DIST * N + i] = wp.new_dist;
    st[(int64_t)QW_YAWERR * N + i] = wp.yaw_err;
    ist[(int64_t)QI_STEP * N + i] = step_count;
    ist[(int64_t)QWI_NTARGETS * N + i] = wp.first;
    reward[i] = rew;
    term[i] = (s.flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (s.flags & FLAG_TRUNC) ? 1 : 0;
    if (info)
      info[i] = (uint8_t)(((s.flags & FLAG_OOB) ? 1 : 0) | ((s.flags & FLAG_COLLISION) ? 2 : 0) | ((s.flags & FLAG_QW_COMPLETE) ? 4 : 0) |
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
  flush_obs_tile<kQwObsStride>(smem, row_skip, skip, obs, sch, O, N);
}

template <int MODE, bool INJECT>
__global__ void __launch_bounds__(kBlock)
    k_qxwp_reset(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ QxWaypointParams w,
                 const __grid_constant__ RngParams rng, float* __restrict__ st, int32_t* __restrict__ ist,
                 const float* __restrict__ start_pos, const float* __restrict__ start_orn, const float* __restrict__ reset_targets,
                 const uint8_t* __restrict__ mask, const float* __restrict__ noise, float* __restrict__ obs, uint32_t seq, int64_t N) {
  __shared__ float smem[kBlock * kQwObsStride];
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  const int O = (h.angle_representation == 0 ? 20 : 21) + (w.use_yaw_targets ? 4 : 3) * w.num_targets;
  QuadXRegs s;
  QwState wp;
  const float pose[6] = {start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1], start_orn[3 * i + 2]};
  qw_reset_env<MODE, INJECT>(p, w, rng, pose, reset_targets, noise, seq, N, i, st + i, N, s, wp);
  const float zero[4] = {0.f, 0.f, 0.f, 0.f};
  float* row = smem + threadIdx.x * kQwObsStride;
  qw_observation(h, w, s, zero, wp.first, st + i, N, row);
  quadx_store<7>(st, ist, N, i, s);
  st[(int64_t)QW_DIST * N + i] = wp.new_dist;
  st[(int64_t)QW_YAWERR * N + i] = wp.yaw_err;
  ist[(int64_t)QI_STEP * N + i] = 0;
  ist[(int64_t)QWI_NTARGETS * N + i] = 0;
  if (obs)
    for (int k = 0; k < O; ++k) obs[i * O + k] = row[k];
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
// k_qxwp_step for tail_env_step / tail_env_reset
static auto qwp_step_launch(PfbContext* h, float* actions, const float* noise) {
  return [=](auto inject, auto randact, auto autoreset, int grid, cudaStream_t s, float* spare, const TailArgs& a) -> int {
    PFB_MODE_SWITCH(h->hover.flight_mode,
                    (k_qxwp_step<MODE, decltype(inject)::value, decltype(randact)::value, decltype(autoreset)::value><<<grid, kBlock, 0, s>>>(
                        h->qx, h->hover, h->qwp, h->rng, h->buf.state, h->buf.istate, actions, noise, h->buf.obs, h->buf.reward, h->buf.term,
                        h->buf.trunc, h->buf.info, h->buf.start_pos, h->buf.start_orn, spare, a, h->n)));
    return 0;
  };
}

int qwp_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s) {
  const int mode = h->hover.flight_mode;
  auto reset = [&](uint32_t seq, int g) -> int {
#define QR_ARGS h->qx, h->hover, h->qwp, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn, h->buf.reset_targets, mask, noise, \
                h->buf.obs, seq, h->n
    if (noise) { PFB_MODE_SWITCH(mode, (k_qxwp_reset<MODE, true><<<g, kBlock, 0, s>>>(QR_ARGS))); }
    else { PFB_MODE_SWITCH(mode, (k_qxwp_reset<MODE, false><<<g, kBlock, 0, s>>>(QR_ARGS))); }
#undef QR_ARGS
    return 0;
  };
  if (tail_env_reset(h, mask, s, reset, qwp_step_launch(h, h->buf.setpoint, nullptr))) return -1;
  h->mode = mode;  // the env's flight mode, not the Aviary default
  return 0;
}

int qwp_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s) {
  return tail_env_step(h, noise, randact, s, qwp_step_launch(h, actions, noise));
}
