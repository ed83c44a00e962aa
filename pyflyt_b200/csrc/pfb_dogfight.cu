// pfb_dogfight.cu — MAFixedwingDogfight on the batched stepper (BASELINE.json configs[4]).
//
// Replaces /root/reference/PyFlyt/pz_envs/fixedwing_envs/ma_fixedwing_dogfight_env.py:346-721 and
// ma_fixedwing_base_env.py:166-338 for many arenas at once.  One thread = one aircraft; an arena is
// A = 2*team_size ADJACENT lanes of a warp (A in {2, 4}), so the pairwise combat state — separation,
// engagement angle, hits, healths — is exchanged with warp shuffles inside the same launch that integrates
// the aircraft: no shared memory, no second kernel, no collective.  (The cross-rank variant, where an arena's
// agents live on different GPUs, exchanges the same 16-float payload through an NCCL all-gather between two
// kernels: see DESIGN.md §7; it is not built yet.)
#include <cmath>
#include <cstring>

#include "pfb_context.h"
#include "pfb_noise.cuh"
#include "pfb_tail_reset.cuh"

using namespace pfb;

// per-agent dogfight rows alias the (unused) waypoint-target rows of the fixedwing state tensor
enum {
  DF_HEALTH = FW_TARGETS + 0, DF_REWARD = FW_TARGETS + 1, DF_PAST = FW_TARGETS + 2 /*4*/, DF_CUR = FW_TARGETS + 6 /*4*/,
  DF_DIST = FW_TARGETS + 10 /*7*/, DF_ANG = FW_TARGETS + 17 /*7*/
};
enum { FLAG_AGENT_DONE = 1024 /* popped out of self.agents */, FLAG_DF_DEAD = 2048, FLAG_DF_WIN = 4096 };
enum { DI_STEP = 0, DI_FLAGS = 1, DI_HITS = 2 };

constexpr int kDfObsMax = 23 + 14 * 3;   // A = 4
constexpr int kDfObsStride = kDfObsMax | 1;

int df_build_params(const PfbEnvConfig* env, DogfightParams& d) {
  memset(&d, 0, sizeof(d));
  if (!env) return 0;
  d.team_size = env->team_size;
  if (env->env_kind == PFB_ENV_DOGFIGHT && d.team_size != 1 && d.team_size != 2)
    return fail("the fused dogfight kernel supports team_size 1 or 2 (arenas of 2 or 4 adjacent lanes), got %d", d.team_size);
  d.env_step_ratio = env->env_step_ratio;
  d.max_steps = env->max_steps;
  d.sparse_reward = env->sparse_reward;
  d.warmup_steps = env->warmup_steps;
  d.dome = (float)env->flight_dome_size;
  d.damage_per_hit = (float)env->damage_per_hit;
  d.lethal_distance = (float)env->lethal_distance;
  d.lethal_angle = (float)env->lethal_angle;
  d.aggressiveness = (float)env->aggressiveness;
  d.cooperativeness = (float)env->cooperativeness;
  d.spawn_min_radius = (float)env->spawn_min_radius;
  d.spawn_max_radius = (float)env->spawn_max_radius;
  return 0;
}
int df_obs_dim(const PfbContext* h) { return 23 + 14 * (2 * h->df.team_size - 1); }

// spare post-reset states (pfb_tail_reset.cuh): one env-major record of 160 floats per AGENT — the FW_* / DF_* state words,
// the spare header, the received-hits counter and the agent's first observation (its past-action slots are patched when the
// spare is used: the action history survives resets)
enum { DSP_HITS = SpareHdr<FW_ROWS>::END, DSP_OBS = 64, DSP_ROWS = 160 };
static_assert(DSP_HITS < DSP_OBS && DSP_OBS + 23 + 14 * 3 <= DSP_ROWS, "spare record too small");
constexpr int kDfObsPast = 19;  // index of past_actions inside the observation (3 + 3 + 3 + 3 + 5 + 1 + 1)
int df_spare_rows() { return DSP_ROWS; }

struct DfAgent {
  float health, acc_reward;
  float past[4], cur[4];
  float dist[3], ang[3];   // current_distances / current_angles towards partner slot k (other agents in index order)
  int hits;                // received_hits
};

// update_states for the calling agent: _compute_observation + _compute_term_trunc_rew_info.
// `li` = index inside the arena, `base` = lane of agent 0, `full` = lanes taking part (whole arenas only).
// Partners are addressed RELATIVELY (r = 1 .. A-1 -> agent (li + r) mod A) so that every per-partner array is
// indexed by a compile-time constant and stays in registers; slot r-1 is this agent's persistent slot for it.
template <int A>
__device__ __forceinline__ void df_update_states(const DogfightParams& d, FixedwingRegs& s, DfAgent& ag, int li, int base, int step_count,
                                                 bool write_obs, float* obs, unsigned full) {
  constexpr int ts = A / 2;
  const Rot<rreal>& R = s.R;
  // forward vector = first column of R; the reported position is shifted 0.35 m back along it (:390)
  const float fx = (float)R.m00, fy = (float)R.m10, fz = (float)R.m20;
  const float px = (float)s.px - 0.35f * fx, py = (float)s.py - 0.35f * fy, pz = (float)s.pz - 0.35f * fz;
  const float gvx = (float)s.vx, gvy = (float)s.vy, gvz = (float)s.vz;  // rotation @ lin_vel == world velocity
  float roll = 0.f, pitch = 0.f, yaw = 0.f;
  if (write_obs) euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
  const bool my_team = li >= ts;
  const float dorigin = sqrtf(px * px + py * py + pz * pz);

  int hits_made = 0, received = 0, team_hits_others = 0;
  float er = 0.0f, close_pen = 0.0f;
  int pj[A - 1];
  float p_sep[A - 1][3], p_gv[A - 1][3], p_speed2[A - 1], p_z[A - 1];
  bool p_hit_ij[A - 1];
#pragma unroll
  for (int r = 1; r < A; ++r) {
    const int k = r - 1;
    const int j = (li + r) & (A - 1);
    const int src = base + j;
    pj[k] = j;
    const float jx = __shfl_sync(full, px, src), jy = __shfl_sync(full, py, src), jz = __shfl_sync(full, pz, src);
    const float jfx = __shfl_sync(full, fx, src), jfy = __shfl_sync(full, fy, src), jfz = __shfl_sync(full, fz, src);
    p_gv[k][0] = __shfl_sync(full, gvx, src); p_gv[k][1] = __shfl_sync(full, gvy, src); p_gv[k][2] = __shfl_sync(full, gvz, src);
    p_speed2[k] = p_gv[k][0] * p_gv[k][0] + p_gv[k][1] * p_gv[k][1] + p_gv[k][2] * p_gv[k][2];
    p_z[k] = jz;
    // pairwise combat state, my row (i -> j) and my column (j -> i); :393-415
    const float sx = jx - px, sy = jy - py, sz = jz - pz;
    p_sep[k][0] = sx; p_sep[k][1] = sy; p_sep[k][2] = sz;
    const float dist = sqrtf(sx * sx + sy * sy + sz * sz);
    // arccos(sep . fwd / |sep|) evaluated as atan2(|sep x fwd|, sep . fwd): accurate near 0 where the cone test lives
    const float cx = sy * fz - sz * fy, cy = sz * fx - sx * fz, cz = sx * fy - sy * fx;
    const float ang = atan2_f(sqrtf(cx * cx + cy * cy + cz * cz), sx * fx + sy * fy + sz * fz);
    const float dx = sy * jfz - sz * jfy, dy = sz * jfx - sx * jfz, dz = sx * jfy - sy * jfx;
    const float ang_ji = atan2_f(sqrtf(dx * dx + dy * dy + dz * dz), -(sx * jfx + sy * jfy + sz * jfz));
    const bool ffm = (j >= ts) != my_team;  // friendly-fire mask: only opponents can be hit
    const bool rng = dist < d.lethal_distance;
    const bool ch_ij = fabsf(ang) < 1.57079632679f, ch_ji = fabsf(ang_ji) < 1.57079632679f;
    const bool h_ij = (ang < d.lethal_angle) && rng && ch_ij && ffm;
    const bool h_ji = (ang_ji < d.lethal_angle) && rng && ch_ji && ffm;
    p_hit_ij[k] = h_ij;
    hits_made += h_ij ? 1 : 0;
    received += h_ji ? 1 : 0;
    // engagement rewards, row i (:552-600)
    if (!d.sparse_reward) {
      const float dd = fmaxf(ag.dist[k] - dist, 0.0f);  // previous - current
      er += (!rng && ch_ij && ffm) ? 4.0f * dd : 0.0f;
      float da = (rng && ffm) ? (ag.ang[k] - ang) : 0.0f;
      if (da < 0.0f) da *= d.aggressiveness;
      er += 30.0f * da;
      const float inv_ij = (ffm && rng && ch_ij) ? fast_rcp(ang + 0.1f) : 0.0f;
      const float inv_ji = (ffm && rng && ch_ji) ? fast_rcp(ang_ji + 0.1f) : 0.0f;
      er += 3.0f * (inv_ij - (1.0f - d.aggressiveness) * inv_ji);
      close_pen += dist < 5.0f ? 10.0f * (5.0f - dist) : 0.0f;
    }
    er += 20.0f * ((h_ij ? 1.0f : 0.0f) - (1.0f - d.aggressiveness) * (h_ji ? 1.0f : 0.0f));
    ag.dist[k] = dist;
    ag.ang[k] = ang;
  }
  // healths (:486-489)
  ag.hits += received;
  ag.health = fmaxf(ag.health - d.damage_per_hit * (float)received, 0.0f);
  const bool collided = (s.flags & FLAG_CONTACT_ARRAY) != 0;
  const bool oob = dorigin > d.dome;
  const float h_final = (collided || oob) ? 0.0f : ag.health;
  // second exchange: post-damage health (observation), final health (team wins), hits made (team bonus)
  float n_h[A - 1];
  bool own_alive = h_final > 0.0f;
#pragma unroll
  for (int r = 1; r < A; ++r) {
    const int k = r - 1;
    const int src = base + pj[k];
    n_h[k] = __shfl_sync(full, ag.health, src);
    const float hf = __shfl_sync(full, h_final, src);
    const int hm = __shfl_sync(full, hits_made, src);
    const bool same_team = (pj[k] >= ts) == my_team;
    team_hits_others += same_team ? hm : 0;
    own_alive = own_alive || (same_team && hf > 0.0f);
  }
  // the opponent paired with me by the reference's elementwise team_wins (:684-691)
  const int opp = (my_team ? 0 : ts) + (li - (my_team ? ts : 0));
  const float opp_h = __shfl_sync(full, h_final, base + opp);

  if (write_obs) {  // :503-529: "self", then every other ACTIVE agent in ascending index order, zero padding
    int n = 0;
    obs[n++] = s.wx; obs[n++] = s.wy; obs[n++] = s.wz;
    obs[n++] = roll; obs[n++] = pitch; obs[n++] = yaw;
    obs[n++] = s.vb.x; obs[n++] = s.vb.y; obs[n++] = s.vb.z;
    obs[n++] = px; obs[n++] = py; obs[n++] = pz;
#pragma unroll
    for (int k = 0; k < kMaxSurfaces; ++k) obs[n++] = s.act[k];
    obs[n++] = s.thr;
    obs[n++] = ag.health;
#pragma unroll
    for (int k = 0; k < 4; ++k) obs[n++] = ag.past[k];
    constexpr int O = 23 + 14 * (A - 1);
    for (int k = n; k < O; ++k) obs[k] = 0.0f;  // the row lives in shared memory: dynamic indexing is free
    bool inactive[A - 1];
#pragma unroll
    for (int k = 0; k < A - 1; ++k) inactive[k] = (n_h[k] <= 0.0f) && (p_z[k] < 2.0f) && (p_speed2[k] < 0.01f);
#pragma unroll
    for (int r = 1; r < A; ++r) {
      const int k = r - 1;
      const int src = base + pj[k];
      // these shuffles must be executed by every lane of the arena, active partner or not
      const float jwx = __shfl_sync(full, s.wx, src), jwy = __shfl_sync(full, s.wy, src), jwz = __shfl_sync(full, s.wz, src);
      const float jr = __shfl_sync(full, roll, src), jp = __shfl_sync(full, pitch, src), jyw = __shfl_sync(full, yaw, src);
      if (inactive[k]) continue;
      int pos = 0;  // active partners with a smaller index come first
#pragma unroll
      for (int q = 0; q < A - 1; ++q) pos += (q != k && !inactive[q] && pj[q] < pj[k]) ? 1 : 0;
      float* o = obs + 23 + 14 * pos;
      o[0] = jwx; o[1] = jwy; o[2] = jwz;
      o[3] = jr - roll; o[4] = jp - pitch; o[5] = jyw - yaw;
      // partner's world velocity and the separation, both in MY body frame (x @ rotation == R^T x)
      const float vx = p_gv[k][0], vy = p_gv[k][1], vz = p_gv[k][2];
      o[6] = ((float)R.m00 * vx + (float)R.m10 * vy + (float)R.m20 * vz) - s.vb.x;
      o[7] = ((float)R.m01 * vx + (float)R.m11 * vy + (float)R.m21 * vz) - s.vb.y;
      o[8] = ((float)R.m02 * vx + (float)R.m12 * vy + (float)R.m22 * vz) - s.vb.z;
      const float sx = p_sep[k][0], sy = p_sep[k][1], sz = p_sep[k][2];
      o[9] = (float)R.m00 * sx + (float)R.m10 * sy + (float)R.m20 * sz;
      o[10] = (float)R.m01 * sx + (float)R.m11 * sy + (float)R.m21 * sz;
      o[11] = (float)R.m02 * sx + (float)R.m12 * sy + (float)R.m22 * sz;
      o[12] = n_h[k];
      o[13] = ((pj[k] >= ts) == my_team) ? 1.0f : 0.0f;
    }
  }
  // team bonus (:601-610) and boundary rewards (:614-639)
  er += d.cooperativeness * (float)(hits_made + team_hits_others);
  float br = 0.0f;
  if (!d.sparse_reward) br = tanhf(0.1f * pz - 1.0f) - tanhf(0.0025f * dorigin - 1.0f) - close_pen;
  ag.acc_reward += er + br;
  // terminations (:655-692)
  if (step_count > d.max_steps) s.flags |= FLAG_TRUNC;
  if (ag.health <= 1e-3f) s.flags |= FLAG_TERM | FLAG_DF_DEAD;
  if (collided) { s.flags |= FLAG_TERM | FLAG_COLLISION; ag.acc_reward = -1000.0f; }
  if (oob) { s.flags |= FLAG_TERM | FLAG_OOB; ag.acc_reward = -1000.0f; }
  ag.health = h_final;
  if (opp_h <= 0.0f && own_alive) { s.flags |= FLAG_TERM | FLAG_DF_WIN; ag.acc_reward = 300.0f; }
  (void)p_hit_ij;
}

// rs / ci: as for fixedwing_load — field-major state rows by default, an env-major spare record with (1, 0); `hits` then
// comes from the record's own word instead of the int tensor
__device__ __forceinline__ void df_load_agent(const float* __restrict__ st, const int32_t* __restrict__ ist, int64_t N, int64_t i, DfAgent& ag,
                                              int64_t rs = -1, int64_t ci = -1) {
  const bool rec = rs >= 0;
  if (!rec) { rs = N; ci = i; }
  auto F = [&](int row) { return st[(int64_t)row * rs + ci]; };
  ag.health = F(DF_HEALTH); ag.acc_reward = F(DF_REWARD);
#pragma unroll
  for (int k = 0; k < 4; ++k) { ag.past[k] = F(DF_PAST + k); ag.cur[k] = F(DF_CUR + k); }
#pragma unroll
  for (int k = 0; k < 3; ++k) { ag.dist[k] = F(DF_DIST + k); ag.ang[k] = F(DF_ANG + k); }
  ag.hits = rec ? __float_as_int(st[DSP_HITS]) : ist[(int64_t)DI_HITS * N + i];
}
__device__ __forceinline__ void df_store_agent(float* __restrict__ st, int32_t* __restrict__ ist, int64_t N, int64_t i, const DfAgent& ag,
                                               int64_t rs = -1, int64_t ci = -1) {
  const bool rec = rs >= 0;
  if (!rec) { rs = N; ci = i; }
  auto S = [&](int row, float v) { st[(int64_t)row * rs + ci] = v; };
  S(DF_HEALTH, ag.health); S(DF_REWARD, ag.acc_reward);
#pragma unroll
  for (int k = 0; k < 4; ++k) { S(DF_PAST + k, ag.past[k]); S(DF_CUR + k, ag.cur[k]); }
#pragma unroll
  for (int k = 0; k < 3; ++k) { S(DF_DIST + k, ag.dist[k]); S(DF_ANG + k, ag.ang[k]); }
  if (rec) st[DSP_HITS] = __int_as_float(ag.hits);
  else ist[(int64_t)DI_HITS * N + i] = ag.hits;
}

// reset of the calling agent's arena (:219-344): spawn pose from the bound buffers or drawn on device
template <int A, bool INJECT>
__device__ __forceinline__ void df_reset_agent(const FixedwingParams& p, const DogfightParams& d, const RngParams& rng,
                                               const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                                               const float* __restrict__ noise, uint32_t seq, bool random_spawn, int64_t N, int64_t i, int li,
                                               int base, FixedwingRegs& s, DfAgent& ag, float* obs, unsigned lanes) {
  float sx = start_pos[3 * i], sy = start_pos[3 * i + 1], sz = start_pos[3 * i + 2];
  float yaw = start_orn[3 * i + 2], roll = start_orn[3 * i], pitch = start_orn[3 * i + 1];
  if (random_spawn) {  // _get_start_pos_orn (:177-217): one base angle per arena, per-agent radius / height / heading jitter
    const uint64_t g0 = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)(i - li);
    U4 a = philox4x32_10(U4{(uint32_t)g0, (uint32_t)(g0 >> 32), seq, 6u << 24}, rng.k0, rng.k1);
    const uint64_t g = g0 + (uint64_t)li;
    U4 b = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), seq, (6u << 24) | 1u}, rng.k0, rng.k1);
    const float two_pi = 6.28318530717958647692f;
    float rad = (two_pi / (float)A) * (float)li + two_pi * u32_to_unit_open(a.x);  // pi / team_size * index + U(0, 2 pi)
    float radius = d.spawn_min_radius + (d.spawn_max_radius - d.spawn_min_radius) * u32_to_unit_open(b.x);
    float height = d.spawn_min_radius + (d.spawn_max_radius - d.spawn_min_radius) * u32_to_unit_open(b.y);  // (sic) radius range, :199-203
    float sn, cs;
    sincos_f(fmodf(rad, two_pi), sn, cs);
    sx = radius * cs; sy = radius * sn; sz = height;
    roll = 0.0f; pitch = 0.0f;
    yaw = rad + u32_to_unit_open(b.z) * 0.39269908169872414f;
  }
  fixedwing_reset(p, s, sx, sy, sz, roll, pitch, yaw);
  // starting_velocity = 20 m/s along the heading (:235-239)
  s.vx = (vreal)(20.0f * (float)s.R.m00); s.vy = (vreal)(20.0f * (float)s.R.m10); s.vz = (vreal)(20.0f * (float)s.R.m20);
  body_update_state(s);
  ag.health = 1.0f; ag.acc_reward = 0.0f; ag.hits = 0;
#pragma unroll
  for (int k = 0; k < 3; ++k) { ag.dist[k] = 0.0f; ag.ang[k] = 0.0f; }
  // current_actions / past_actions survive a reset in the reference (they are only created in __init__)
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
  for (int k = 0; k < d.warmup_steps; ++k) fixedwing_aviary_step<0>(p, s, nz);
  fixedwing_requantize(s);  // exactly what the state tensor / a spare record will hold
  df_update_states<A>(d, s, ag, li, base, 0, true, obs, lanes);
}

template <int A, bool INJECT, bool RANDACT, bool AUTORESET>
__global__ void __launch_bounds__(kBlock, kAeroBlocks)
    k_df_step(const __grid_constant__ FixedwingParams p, const __grid_constant__ DogfightParams d, const __grid_constant__ RngParams rng,
              float* __restrict__ st, int32_t* __restrict__ ist, float* __restrict__ actions, const float* __restrict__ noise,
              float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ term, uint8_t* __restrict__ trunc,
              uint8_t* __restrict__ info, const float* __restrict__ start_pos, const float* __restrict__ start_orn,
              float* __restrict__ spare, const __grid_constant__ TailArgs a, int64_t N) {
  __shared__ float smem[kBlock * kDfObsStride];
  __shared__ uint8_t row_skip[kBlock];
  constexpr int O = 23 + 14 * (A - 1);
  const uint32_t step_seq = a.step_seq;
  // work items are whole arenas: a regular lane owns one agent; tail lanes stride over the done-arena list
  TailWork sch = tail_schedule<A, AUTORESET>(a, N, threadIdx.x);  // N is a multiple of A: an arena is never cut
  const bool tail = sch.tail;
  const int li = threadIdx.x % A;                 // agent index inside its arena
  const int base = (threadIdx.x & 31) - li;       // lane of the arena's agent 0
  bool skip = true;
  float* row = smem + threadIdx.x * kDfObsStride;
#pragma unroll 1
  for (;; sch.t += sch.t_stride) {
    // whole arenas enter or leave together (t is arena-uniform), so every shuffle below names exactly the
    // lanes that are present
    const bool go = sch.t < sch.t_end;
    unsigned lanes = __ballot_sync(0xffffffffu, go);
    if (lanes == 0u) break;
    if (!go) continue;
    const int64_t i = tail_env<A>(a, sch, li);
    FixedwingRegs s;
    DfAgent ag;
    float rew_out = 0.0f;
    int step_count = 0;
    if (tail) {
      // arena reset: normally every agent copies its spare (state, combat bookkeeping, first observation of the next
      // episode); build mode computes those spares; without usable spares the arena runs its warm-up inline.  The episode
      // number (arena-uniform: agent 0's) keys the spawn and the warm-up noise in all three cases.
      float* rec = spare ? spare + i * DSP_ROWS : nullptr;
      const SpareProbe sp = spare_probe<FW_ROWS>(a, rec, nullptr, false);
      const uint32_t nseq = __shfl_sync(lanes, sp.episode, base);
      const unsigned arena_mask = ((1u << A) - 1u) << base;
      const bool hit = (__ballot_sync(lanes, sp.hit) & arena_mask) == arena_mask;  // all of the arena's spares, or none
      df_load_agent(st, ist, N, i, ag);  // current / past actions survive the reset, like the reference's arrays
      if (hit) {
        const float p0 = ag.past[0], p1 = ag.past[1], p2 = ag.past[2], p3 = ag.past[3];
        const float c0 = ag.cur[0], c1 = ag.cur[1], c2 = ag.cur[2], c3 = ag.cur[3];
        fixedwing_load(rec, ist, N, i, s, 1, 0);
        df_load_agent(rec, ist, N, i, ag, 1, 0);
        ag.past[0] = p0; ag.past[1] = p1; ag.past[2] = p2; ag.past[3] = p3;
        ag.cur[0] = c0; ag.cur[1] = c1; ag.cur[2] = c2; ag.cur[3] = c3;
        s.flags = __float_as_uint(rec[SpareHdr<FW_ROWS>::FLAGS]);
        for (int k = 0; k < O; ++k) row[k] = rec[DSP_OBS + k];
        row[kDfObsPast + 0] = p0; row[kDfObsPast + 1] = p1; row[kDfObsPast + 2] = p2; row[kDfObsPast + 3] = p3;
      }
      const unsigned inl = __ballot_sync(lanes, !hit);  // the arenas that run their warm-up here exchange among themselves
      if (!hit) {
        if (a.build) spare_open<FW_ROWS>(rec, nullptr);
        df_reset_agent<A, false>(p, d, rng, start_pos, start_orn, nullptr, nseq, true, N, i, li, base, s, ag, row, inl);
      }
      if (a.build) {
        fixedwing_store(rec, ist, N, i, s, false, 1, 0);
        df_store_agent(rec, ist, N, i, ag, 1, 0);
        for (int k = 0; k < O; ++k) rec[DSP_OBS + k] = row[k];
        spare_seal<FW_ROWS>(rec, s.flags & ~(uint32_t)FLAG_AGENT_DONE, nseq);
        continue;
      }
      s.flags &= ~(uint32_t)(FLAG_AGENT_DONE);
      s.flags |= fresh_tag(step_seq);
    } else {
      fixedwing_load(st, ist, N, i, s);
      df_load_agent(st, ist, N, i, ag);
      // an arena whose agents are all done is reset by a tail CTA on this call; an agent that CTA has already rewritten
      // carries this launch's fresh tag instead of AGENT_DONE (pfb_quadx.cuh, FLAG_FRESH*)
      const unsigned arena_mask = ((1u << A) - 1u) << base;
      const bool i_done = (s.flags & FLAG_AGENT_DONE) != 0;
      const bool owned = tail_owns(s.flags, FLAG_AGENT_DONE, step_seq);
      s.flags &= ~(uint32_t)FLAG_FRESH_ANY;
      const bool arena_done = (__ballot_sync(lanes, owned) & arena_mask) == arena_mask;
      lanes = __ballot_sync(lanes, !(AUTORESET && arena_done));
      if (AUTORESET && arena_done) continue;
      float act[4];
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
      // ma_fixedwing_base_env.py:299-308: past <- current, current <- action of the agents still in self.agents
#pragma unroll
      for (int k = 0; k < 4; ++k) { ag.past[k] = ag.cur[k]; ag.cur[k] = i_done ? 0.0f : act[k]; }
      s.sp[0] = ag.cur[0]; s.sp[1] = ag.cur[1]; s.sp[2] = ag.cur[2]; s.sp[3] = ag.cur[3] * 0.5f + 0.5f;
      step_count = ist[(int64_t)DI_STEP * N + i];
      auto nz = make_noise<INJECT>(noise, N, i, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
      const bool full = fixedwing_full_model(p);  // launch-uniform
#pragma unroll 1
      for (int k = 0; k < d.env_step_ratio; ++k) {  // parallel envs do not break out of the loop (:312-314)
        if (full) fixedwing_aviary_step<0, true>(p, s, nz);
        else fixedwing_aviary_step<0>(p, s, nz);
        df_update_states<A>(d, s, ag, li, base, step_count, k == d.env_step_ratio - 1, row, lanes);
      }
      rew_out = ag.acc_reward;
      if (!i_done) ag.acc_reward = 0.0f;  // pop_term_trunc_rew_info_by_id only runs for agents still in self.agents
      step_count += 1;
    }
    fixedwing_store(st, ist, N, i, s);
    // fixedwing_store wrote the flags; mark agents that just left self.agents
    uint32_t flags = s.flags;
    if (!tail && (flags & (FLAG_TERM | FLAG_TRUNC))) flags |= FLAG_AGENT_DONE;
    ist[(int64_t)DI_FLAGS * N + i] = (int32_t)flags;
    df_store_agent(st, ist, N, i, ag);
    ist[(int64_t)DI_STEP * N + i] = step_count;
    reward[i] = rew_out;
    term[i] = (flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (flags & FLAG_TRUNC) ? 1 : 0;
    if (info)
      info[i] = (uint8_t)(((flags & FLAG_OOB) ? 1 : 0) | ((flags & FLAG_COLLISION) ? 2 : 0) | ((flags & FLAG_DF_DEAD) ? 4 : 0) | ((flags & FLAG_DF_WIN) ? 8 : 0));
    if (tail) {
      float* dst = obs + i * O;
      for (int k = 0; k < O; ++k) dst[k] = row[k];
    } else {
      skip = false;
      if (AUTORESET) {  // queue arenas whose agents have ALL left self.agents (the arena's first lane speaks for it)
        const unsigned arena_mask = ((1u << A) - 1u) << base;
        const unsigned done_lanes = __ballot_sync(lanes, (flags & FLAG_AGENT_DONE) != 0);
        const bool leader_done = (li == 0) && ((done_lanes & arena_mask) == arena_mask);
        append_done(a, sch, lanes, leader_done, i);
      }
    }
  }
  if (tail) return;
  flush_obs_tile<kDfObsStride>(smem, row_skip, skip, obs, sch, O, N);
}

template <int A, bool INJECT>
__global__ void __launch_bounds__(kBlock)
    k_df_reset(const __grid_constant__ FixedwingParams p, const __grid_constant__ DogfightParams d, const __grid_constant__ RngParams rng,
               float* __restrict__ st, int32_t* __restrict__ ist, const float* __restrict__ start_pos, const float* __restrict__ start_orn,
               const uint8_t* __restrict__ mask, const float* __restrict__ noise, float* __restrict__ obs, uint32_t seq, int random_spawn,
               int64_t N) {
  __shared__ float smem[kBlock * kDfObsStride];
  constexpr int O = 23 + 14 * (A - 1);
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const int li = threadIdx.x % A;
  const int base = (threadIdx.x & 31) - li;
  // N and kBlock are multiples of A: whole arenas drop out together; the mask is per arena (first agent's entry)
  const bool go = (i < N) && !(mask && !mask[i - li]);
  const unsigned lanes = __ballot_sync(0xffffffffu, go);
  if (!go) return;
  FixedwingRegs s;
  DfAgent ag;
  df_load_agent(st, ist, N, i, ag);
  float* row = smem + threadIdx.x * kDfObsStride;
  df_reset_agent<A, INJECT>(p, d, rng, start_pos, start_orn, noise, seq, random_spawn != 0, N, i, li, base, s, ag, row, lanes);
  fixedwing_store(st, ist, N, i, s);
  df_store_agent(st, ist, N, i, ag);
  ist[(int64_t)DI_STEP * N + i] = 0;
  if (obs)
    for (int k = 0; k < O; ++k) obs[i * O + k] = row[k];
}

// ---------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------
// k_df_step for tail_env_step / tail_env_reset
static auto df_step_launch(PfbContext* h, float* actions, const float* noise) {
  return [=](auto inject, auto randact, auto autoreset, int grid, cudaStream_t s, float* spare, const TailArgs& a) -> int {
    constexpr bool I = decltype(inject)::value, R = decltype(randact)::value, AR = decltype(autoreset)::value;
#define DF_ARGS h->fw, h->df, h->rng, h->buf.state, h->buf.istate, actions, noise, h->buf.obs, h->buf.reward, h->buf.term, h->buf.trunc, \
                h->buf.info, h->buf.start_pos, h->buf.start_orn, spare, a, h->n
    if (h->df.team_size == 1) k_df_step<2, I, R, AR><<<grid, kBlock, 0, s>>>(DF_ARGS);
    else k_df_step<4, I, R, AR><<<grid, kBlock, 0, s>>>(DF_ARGS);
#undef DF_ARGS
    return 0;
  };
}

int df_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s) {
  const int A = 2 * h->df.team_size;
  if (h->n % A) return fail("the number of envs (%lld) must be a multiple of the arena size %d", (long long)h->n, A);
  const int rnd = h->env.randomize_drop;  // reused as "draw the spawn on device" for the dogfight
  auto reset = [&](uint32_t seq, int g) -> int {
#define DR_ARGS h->fw, h->df, h->rng, h->buf.state, h->buf.istate, h->buf.start_pos, h->buf.start_orn, mask, noise, h->buf.obs, seq, rnd, h->n
    if (A == 2) { if (noise) k_df_reset<2, true><<<g, kBlock, 0, s>>>(DR_ARGS); else k_df_reset<2, false><<<g, kBlock, 0, s>>>(DR_ARGS); }
    else { if (noise) k_df_reset<4, true><<<g, kBlock, 0, s>>>(DR_ARGS); else k_df_reset<4, false><<<g, kBlock, 0, s>>>(DR_ARGS); }
#undef DR_ARGS
    return 0;
  };
  return tail_env_reset(h, mask, s, reset, df_step_launch(h, h->buf.setpoint, nullptr));
}

int df_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s) {
  const int A = 2 * h->df.team_size;
  if (h->n % A) return fail("the number of envs (%lld) must be a multiple of the arena size %d", (long long)h->n, A);
  return tail_env_step(h, noise, randact, s, df_step_launch(h, actions, noise));
}

// ===================================================================================================
// Split ("agent-major") variant — BASELINE.json configs[4] as written: the agents of one arena live on
// DIFFERENT ranks, so the combat state needs one exchange per Aviary step.  Per Aviary step:
//     k_df_split_physics  (integrate my aircraft, publish a 20-float payload per agent)
//     exchange            either ncclAllGather of the payload table (host side), or NONE: the physics kernel stores every
//                         payload directly into all ranks' tables over NVLink peer memory, followed by a cross-rank barrier
//     k_df_split_combat   (pairwise combat state, health, rewards, terminations from the gathered table)
// Global agent id gid = k * num_arenas + g (member k of arena g); rank r owns gids [r*n_local, (r+1)*n_local).
// 1-vs-1 arenas (team_size 1).  No in-kernel autoreset: reset() is a collective call.
// ===================================================================================================
constexpr int kPayload = 20;  // pos'(3) fwd(3) gv(3) w(3) euler(3) health(1) contact(1) + pad to 5 float4
enum { PL_POS = 0, PL_FWD = 3, PL_GV = 6, PL_W = 9, PL_EUL = 12, PL_HEALTH = 15, PL_CONTACT = 16 };

__device__ __forceinline__ void df_publish(const FixedwingRegs& s, const DfAgent& ag, float* __restrict__ out) {
  const Rot<rreal>& R = s.R;
  const float fx = (float)R.m00, fy = (float)R.m10, fz = (float)R.m20;
  float roll, pitch, yaw;
  euler_from_quat((float)s.qx, (float)s.qy, (float)s.qz, (float)s.qw, roll, pitch, yaw);
  float4* o = reinterpret_cast<float4*>(out);
  o[0] = make_float4((float)s.px - 0.35f * fx, (float)s.py - 0.35f * fy, (float)s.pz - 0.35f * fz, fx);
  o[1] = make_float4(fy, fz, (float)s.vx, (float)s.vy);
  o[2] = make_float4((float)s.vz, s.wx, s.wy, s.wz);
  o[3] = make_float4(roll, pitch, yaw, ag.health);
  o[4] = make_float4((s.flags & FLAG_CONTACT_ARRAY) ? 1.0f : 0.0f, 0.f, 0.f, 0.f);
}

// first = 1: take the action, roll past/current actions (start of env.step); warm = 1: reset + warm-up
template <bool INJECT>
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_df_split_physics(const __grid_constant__ FixedwingParams p, const __grid_constant__ DogfightParams d, const __grid_constant__ RngParams rng,
                       float* __restrict__ st, int32_t* __restrict__ ist, const float* __restrict__ actions, const float* __restrict__ noise,
                       const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ payload,
                       const uint64_t* __restrict__ peers, int world, int64_t slot0, const uint64_t* __restrict__ peer_flags, int rank,
                       int epoch, unsigned* __restrict__ ticket, int first, int do_reset, uint32_t seq, uint32_t sub, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i < N) {
  FixedwingRegs s;
  DfAgent ag;
  df_load_agent(st, ist, N, i, ag);
  if (do_reset) {
    fixedwing_reset(p, s, start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i], start_orn[3 * i + 1], start_orn[3 * i + 2]);
    s.vx = (vreal)(20.0f * (float)s.R.m00); s.vy = (vreal)(20.0f * (float)s.R.m10); s.vz = (vreal)(20.0f * (float)s.R.m20);
    body_update_state(s);
    ag.health = 1.0f; ag.acc_reward = 0.0f; ag.hits = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) { ag.dist[k] = 0.0f; ag.ang[k] = 0.0f; }
    auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
    for (int k = 0; k < d.warmup_steps; ++k) fixedwing_aviary_step<0>(p, s, nz);
    ist[(int64_t)DI_STEP * N + i] = 0;
  } else {
    fixedwing_load(st, ist, N, i, s);
    if (first) {
      const bool i_done = (s.flags & FLAG_AGENT_DONE) != 0;
      float4 a4 = __ldg(reinterpret_cast<const float4*>(actions) + i);
      const float act[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) { ag.past[k] = ag.cur[k]; ag.cur[k] = i_done ? 0.0f : act[k]; }
    }
    s.sp[0] = ag.cur[0]; s.sp[1] = ag.cur[1]; s.sp[2] = ag.cur[2]; s.sp[3] = ag.cur[3] * 0.5f + 0.5f;
    // one Aviary step; the noise stream position is (env-step sequence, Aviary step index)
    auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_ENV_STEP, p.noise_loc, 4);  // ratio > 2 path: one call per step
    nz.seek(sub);
    if (fixedwing_full_model(p)) fixedwing_aviary_step<0, true>(p, s, nz);
    else fixedwing_aviary_step<0>(p, s, nz);
  }
  fixedwing_store(st, ist, N, i, s);
  df_store_agent(st, ist, N, i, ag);
  if (peers) {
    // fused exchange: the payload goes straight into the table of EVERY rank (peer stores over NVLink, 80 bytes = 5 float4
    // per agent per peer) instead of into a local buffer that a separate all-gather would then move; slot0 = float offset
    // of this rank's first agent inside the (double-buffered) table.  The stores are visible to the peers once this
    // kernel has completed; the cross-rank barrier that follows on the stream orders the readers behind it.
    for (int r = 0; r < world; ++r) df_publish(s, ag, reinterpret_cast<float*>(peers[r]) + slot0 + (int64_t)kPayload * i);
  } else {
    df_publish(s, ag, payload + (int64_t)kPayload * i);
  }
  }  // i < N
  if (peer_flags) {
    // in-kernel signalling: once EVERY CTA's peer stores are fenced, the last CTA to finish raises this rank's flag in all
    // ranks' flag arrays (release, system scope); the combat kernels wait on those flags instead of on a barrier launch
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned t = atomicAdd(ticket, 1u);
      if (t == gridDim.x - 1) {
        *ticket = 0u;
        __threadfence_system();
        for (int r = 0; r < world; ++r) {
          int* flag = reinterpret_cast<int*>(peer_flags[r]) + rank;
          asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
        }
      }
    }
  }
}

// combat state for 1-vs-1 arenas from the gathered payload table [num_agents][kPayload]
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_df_split_combat(const __grid_constant__ DogfightParams d, float* __restrict__ st, int32_t* __restrict__ ist,
                      const float* table /* NOT __restrict__: other GPUs store into it while this kernel waits (peer-signal) */,
                      float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ term,
                      uint8_t* __restrict__ trunc, uint8_t* __restrict__ info, int64_t first_gid, int64_t num_arenas, int last,
                      const int* __restrict__ wait_flags, int world, int epoch, int64_t N) {
  if (wait_flags) {  // every rank's physics kernel has raised its flag for this exchange (acquire, system scope)
    if ((int)threadIdx.x < world) {
      // bounded: a peer that never launches (crashed rank) must not hang this GPU.  After 2 s the wait gives up; the combat
      // then reads a stale table, which the caller sees as a parity failure, not as a dead box
      unsigned long long t0, t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      int v;
      do {
        asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(wait_flags + threadIdx.x) : "memory");
        if (v >= epoch) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      } while (t1 - t0 < 2000000000ull);
    }
    __syncthreads();
  }
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  const int64_t gid = first_gid + i;
  const int li = (int)(gid / num_arenas);
  const int64_t g = gid - (int64_t)li * num_arenas;
  const int64_t pid = (int64_t)(1 - li) * num_arenas + g;  // my opponent
  // the payload rows are copied into registers with ld.global.cg (L2, never the read-only / L1 path): with in-kernel
  // signalling the table was written by other GPUs during this kernel's lifetime, after the acquire above
  float me[kPayload], ot[kPayload];
#pragma unroll
  for (int k = 0; k < kPayload; ++k) {
    me[k] = __ldcg(table + kPayload * gid + k);
    ot[k] = __ldcg(table + kPayload * pid + k);
  }
  FixedwingRegs s;
  DfAgent ag;
  fixedwing_load(st, ist, N, i, s);
  df_load_agent(st, ist, N, i, ag);
  const int step_count = ist[(int64_t)DI_STEP * N + i];
  const float px = me[PL_POS], py = me[PL_POS + 1], pz = me[PL_POS + 2];
  const float fx = me[PL_FWD], fy = me[PL_FWD + 1], fz = me[PL_FWD + 2];
  const float jx = ot[PL_POS], jy = ot[PL_POS + 1], jz = ot[PL_POS + 2];
  const float jfx = ot[PL_FWD], jfy = ot[PL_FWD + 1], jfz = ot[PL_FWD + 2];
  const float sx = jx - px, sy = jy - py, sz = jz - pz;
  const float dist = sqrtf(sx * sx + sy * sy + sz * sz);
  const float cx = sy * fz - sz * fy, cy = sz * fx - sx * fz, cz = sx * fy - sy * fx;
  const float ang = atan2_f(sqrtf(cx * cx + cy * cy + cz * cz), sx * fx + sy * fy + sz * fz);
  const float dx = sy * jfz - sz * jfy, dy = sz * jfx - sx * jfz, dz = sx * jfy - sy * jfx;
  const float ang_ji = atan2_f(sqrtf(dx * dx + dy * dy + dz * dz), -(sx * jfx + sy * jfy + sz * jfz));
  const bool rng = dist < d.lethal_distance;
  const bool ch_ij = fabsf(ang) < 1.57079632679f, ch_ji = fabsf(ang_ji) < 1.57079632679f;
  const bool h_ij = (ang < d.lethal_angle) && rng && ch_ij;
  const bool h_ji = (ang_ji < d.lethal_angle) && rng && ch_ji;
  float er = 0.0f, close_pen = 0.0f;
  if (!d.sparse_reward) {
    er += (!rng && ch_ij) ? 4.0f * fmaxf(ag.dist[0] - dist, 0.0f) : 0.0f;
    float da = rng ? (ag.ang[0] - ang) : 0.0f;
    if (da < 0.0f) da *= d.aggressiveness;
    er += 30.0f * da;
    const float inv_ij = (rng && ch_ij) ? fast_rcp(ang + 0.1f) : 0.0f;
    const float inv_ji = (rng && ch_ji) ? fast_rcp(ang_ji + 0.1f) : 0.0f;
    er += 3.0f * (inv_ij - (1.0f - d.aggressiveness) * inv_ji);
    close_pen = dist < 5.0f ? 10.0f * (5.0f - dist) : 0.0f;
  }
  er += 20.0f * ((h_ij ? 1.0f : 0.0f) - (1.0f - d.aggressiveness) * (h_ji ? 1.0f : 0.0f));
  ag.dist[0] = dist; ag.ang[0] = ang;
  // healths: mine from the hit I received; the opponent's is recomputed from the hit I made
  ag.hits += h_ji ? 1 : 0;
  ag.health = fmaxf(ag.health - d.damage_per_hit * (h_ji ? 1.0f : 0.0f), 0.0f);
  const float n_h = fmaxf(ot[PL_HEALTH] - d.damage_per_hit * (h_ij ? 1.0f : 0.0f), 0.0f);
  const float dorigin = sqrtf(px * px + py * py + pz * pz), j_dorigin = sqrtf(jx * jx + jy * jy + jz * jz);
  const bool collided = me[PL_CONTACT] != 0.0f, oob = dorigin > d.dome;
  const float h_final = (collided || oob) ? 0.0f : ag.health;
  const float opp_h = (ot[PL_CONTACT] != 0.0f || j_dorigin > d.dome) ? 0.0f : n_h;
  if (last) {
    const Rot<rreal>& R = s.R;
    float* o = obs + 37 * i;
    int n = 0;
    o[n++] = s.wx; o[n++] = s.wy; o[n++] = s.wz;
    o[n++] = me[PL_EUL]; o[n++] = me[PL_EUL + 1]; o[n++] = me[PL_EUL + 2];
    o[n++] = s.vb.x; o[n++] = s.vb.y; o[n++] = s.vb.z;
    o[n++] = px; o[n++] = py; o[n++] = pz;
    for (int k = 0; k < kMaxSurfaces; ++k) o[n++] = s.act[k];
    o[n++] = s.thr;
    o[n++] = ag.health;
    for (int k = 0; k < 4; ++k) o[n++] = ag.past[k];
    const float vx = ot[PL_GV], vy = ot[PL_GV + 1], vz = ot[PL_GV + 2];
    const bool inactive = (n_h <= 0.0f) && (jz < 2.0f) && (vx * vx + vy * vy + vz * vz < 0.01f);
    if (!inactive) {
      o[n++] = ot[PL_W]; o[n++] = ot[PL_W + 1]; o[n++] = ot[PL_W + 2];
      o[n++] = ot[PL_EUL] - me[PL_EUL]; o[n++] = ot[PL_EUL + 1] - me[PL_EUL + 1]; o[n++] = ot[PL_EUL + 2] - me[PL_EUL + 2];
      o[n++] = ((float)R.m00 * vx + (float)R.m10 * vy + (float)R.m20 * vz) - s.vb.x;
      o[n++] = ((float)R.m01 * vx + (float)R.m11 * vy + (float)R.m21 * vz) - s.vb.y;
      o[n++] = ((float)R.m02 * vx + (float)R.m12 * vy + (float)R.m22 * vz) - s.vb.z;
      o[n++] = (float)R.m00 * sx + (float)R.m10 * sy + (float)R.m20 * sz;
      o[n++] = (float)R.m01 * sx + (float)R.m11 * sy + (float)R.m21 * sz;
      o[n++] = (float)R.m02 * sx + (float)R.m12 * sy + (float)R.m22 * sz;
      o[n++] = n_h;
      o[n++] = 0.0f;
    }
    while (n < 37) o[n++] = 0.0f;
  }
  er += d.cooperativeness * (h_ij ? 1.0f : 0.0f);
  float br = 0.0f;
  if (!d.sparse_reward) br = tanhf(0.1f * pz - 1.0f) - tanhf(0.0025f * dorigin - 1.0f) - close_pen;
  ag.acc_reward += er + br;
  if (step_count > d.max_steps) s.flags |= FLAG_TRUNC;
  if (ag.health <= 1e-3f) s.flags |= FLAG_TERM | FLAG_DF_DEAD;
  if (collided) { s.flags |= FLAG_TERM | FLAG_COLLISION; ag.acc_reward = -1000.0f; }
  if (oob) { s.flags |= FLAG_TERM | FLAG_OOB; ag.acc_reward = -1000.0f; }
  ag.health = h_final;
  if (opp_h <= 0.0f && h_final > 0.0f) { s.flags |= FLAG_TERM | FLAG_DF_WIN; ag.acc_reward = 300.0f; }
  uint32_t flags = s.flags;
  if (last == 1) {
    const bool was_done = (flags & FLAG_AGENT_DONE) != 0;
    reward[i] = ag.acc_reward;
    if (!was_done) ag.acc_reward = 0.0f;
    ist[(int64_t)DI_STEP * N + i] = step_count + 1;
    if (flags & (FLAG_TERM | FLAG_TRUNC)) flags |= FLAG_AGENT_DONE;
    term[i] = (flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (flags & FLAG_TRUNC) ? 1 : 0;
    if (info)
      info[i] = (uint8_t)(((flags & FLAG_OOB) ? 1 : 0) | ((flags & FLAG_COLLISION) ? 2 : 0) | ((flags & FLAG_DF_DEAD) ? 4 : 0) | ((flags & FLAG_DF_WIN) ? 8 : 0));
  }
  ist[(int64_t)DI_FLAGS * N + i] = (int32_t)flags;
  df_store_agent(st, ist, N, i, ag);
}

int df_split_physics(PfbContext* h, const float* actions, const float* noise, float* payload, const uint64_t* peers, int world,
                     int64_t slot0, const uint64_t* peer_flags, int rank, int epoch, int first, int do_reset, int sub, cudaStream_t s) {
  if (h->df.team_size != 1) return fail("the split (all-gather) dogfight path is built for team_size 1");
  const uint32_t seq = do_reset ? (0x80000000u | (uint32_t)h->reset_seq) : (uint32_t)h->step_seq;
  if (do_reset) h->reset_seq += 1;
  const int g = grid_for(h->n);
  unsigned* ticket = reinterpret_cast<unsigned*>(h->d_counters) + 4;  // word 4 of the counter block: not part of the rotating queues
  if (noise)
    k_df_split_physics<true><<<g, kBlock, 0, s>>>(h->fw, h->df, h->rng, h->buf.state, h->buf.istate, actions, noise, h->buf.start_pos,
                                                  h->buf.start_orn, payload, peers, world, slot0, peer_flags, rank, epoch, ticket, first, do_reset,
                                                  seq, (uint32_t)sub, h->n);
  else
    k_df_split_physics<false><<<g, kBlock, 0, s>>>(h->fw, h->df, h->rng, h->buf.state, h->buf.istate, actions, nullptr, h->buf.start_pos,
                                                   h->buf.start_orn, payload, peers, world, slot0, peer_flags, rank, epoch, ticket, first, do_reset,
                                                   seq, (uint32_t)sub, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

int df_split_combat(PfbContext* h, const float* table, int64_t first_gid, int64_t num_arenas, int last, const int* wait_flags, int world,
                    int epoch, cudaStream_t s) {
  if (h->df.team_size != 1) return fail("the split (all-gather) dogfight path is built for team_size 1");
  if (wait_flags && (world < 1 || world > kBlock)) return fail("the in-kernel wait supports 1..%d ranks, got %d", kBlock, world);
  k_df_split_combat<<<grid_for(h->n), kBlock, 0, s>>>(h->df, h->buf.state, h->buf.istate, table, h->buf.obs, h->buf.reward, h->buf.term,
                                                      h->buf.trunc, h->buf.info, first_gid, num_arenas, last, wait_flags, world, epoch, h->n);
  LAUNCH_CHECK(h);
  if (last) h->step_seq += 1;
  return 0;
}
