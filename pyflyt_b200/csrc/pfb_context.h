// pfb_context.h — private to libpyflyt_b200: the handle, error plumbing and launch helpers shared by
// the per-vehicle translation units (pfb_lib.cu, pfb_fixedwing.cu, ...).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <type_traits>

#include "../../include/pyflyt_b200.h"
#include "pfb_fixedwing.cuh"
#include "pfb_quadx.cuh"
#include "pfb_rocket.cuh"

// thread-local error string (pfb_last_error); returns -1
int pfb_fail(const char* fmt, ...);
#define fail pfb_fail

#define CUDA_OK(expr)                                                                    \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) return fail("%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

struct RngParams {
  uint32_t k0, k1;        // Philox key (seed)
  uint32_t env_offset_lo; // global id of local env 0 (multi-GPU sharding keeps streams rank-independent)
  uint32_t env_offset_hi;
};

struct PfbContext {
  PfbModel model;
  PfbEnvConfig env;
  int64_t n;
  int device;
  pfb::QuadXParams qx;
  pfb::HoverParams hover;
  pfb::FixedwingParams fw;
  pfb::WaypointParams wp;
  pfb::DogfightParams df;
  pfb::RocketParams rk;
  pfb::LandingParams land;
  RngParams rng;
  PfbBuffers buf;
  bool bound;
  int mode;               // Aviary-level flight mode
  int32_t* d_counters;    // [4] rotating done-list counters: step k appends to [k%4], reads [(k-1)%4], zeroes [(k+1)%4]
  int32_t* d_done_list;   // [4][N] rotating lists of envs (arenas) that finished on a step; list (k-1)%4 is also read by the
                          // side-stream spare rebuild of step k, which step k+2 waits for before list (k+3)%4 is reused
  uint64_t step_seq;      // env.step() calls so far (selects counters/lists, keys the Philox streams)
  uint64_t aviary_seq;    // pfb_aviary_step calls so far
  uint64_t reset_seq;     // pfb_env_reset calls so far
  int64_t launches;
  pfb::QxWaypointParams qwp;
  int sm_count;
  // QuadX-Hover reset pipeline (pfb_lib.cu, "spare post-reset states"): library-owned spares + the side stream that rebuilds them
  float* d_spare;          // spare post-reset states (env-major records), zero-initialised; nullptr = warm-ups run inline
  int2* d_consumed;        // QuadX-Hover fused rollout: (env, episode to rebuild) for every spare a launch consumed
  int fused_ready;         // every env has its spares kRolloutAhead ahead and the step pipeline is drained (cleared by single steps / resets)
  uint32_t* d_elist;       // QuadX-Hover: [4][N] episode number being built for each done-list entry (builder phase 0 -> phase 1)
  uint32_t* d_episode;     // QuadX-Hover: [N] episode number of each env's current valid spare (its buffer = episode & 1)
  cudaStream_t side;       // k_hover_spare runs here, concurrently with the following step launches
  cudaEvent_t ev_step;     // recorded on the caller's stream after a step launch; the side stream waits on it
  cudaEvent_t ev_spare[4]; // ev_spare[k % 4]: spares consumed by step k are rebuilt; step k + 2 waits on it
  int64_t side_launches;
  // optional per-step CUDA-event pairs around the dominant kernel (bench.py's roofline leg)
  int mapped_dyn_smem;    // dynamic shared memory requested by the step launch of pfb_env_step_mapped (bounds the CTAs resident per SM: several waves)
  int step_dyn_smem;      // what the next QuadX-Hover step launch requests (0 = everything resident in one wave)
  float* noise_dump;      // optional [substeps per env step][N] device buffer: the step kernel writes every noise draw it hands out (tests)
  cudaEvent_t* prof_ev;   // [2 * prof_cap]
  int prof_cap;
  int prof_n;
};

// One warp per CTA.  Measured on B200 (65 536-env Hover step, L2 flushed / warm): 32 threads 22.1 / 20.5 us, 64 threads
// 22.5 / 22.6 us, 128 threads 24.7 / 24.5 us: a CTA retires as soon as its own warp is done, so the SM back-fills sooner and
// the single wave has a shorter tail.  448 threads per SM resident (<= 146 regs/thread) for the generic kernels.
#ifndef PFB_BLOCK  // A/B knob (per translation unit): threads per CTA
#define PFB_BLOCK 32
#endif
constexpr int kBlock = PFB_BLOCK;
constexpr int kMinBlocks = 448 / kBlock > 0 ? 448 / kBlock : 1;
// the step kernels of the aerodynamic-surface vehicles (Fixedwing-Waypoints, Dogfight): the batch sizes they run at leave
// < 4 warps per SM, so registers are better spent on interleaving the surfaces than on residency.  Measured on B200 at 16 384
// aircraft (profiles/r02_aero_full_block.jsonl): 14 CTAs / SM (128 registers) 31.0 / 34.9 us per step, 8 CTAs / SM (145 / 176
// registers) 30.1 / 33.1 us.  PFB_AERO_MIN_BLOCKS: A/B knob
#ifndef PFB_AERO_MIN_BLOCKS
#define PFB_AERO_MIN_BLOCKS 8
#endif
constexpr int kAeroBlocks = PFB_AERO_MIN_BLOCKS;

static inline int grid_for(int64_t n) { return (int)((n + kBlock - 1) / kBlock); }

#define LAUNCH_CHECK(h)                                                     \
  do {                                                                      \
    cudaError_t _e = cudaGetLastError();                                    \
    if (_e != cudaSuccess) return fail("kernel launch failed: %s", cudaGetErrorString(_e)); \
    (h)->launches += 1;                                                     \
  } while (0)

// per-step bookkeeping shared by every env kind (rotating counters and lists, tail CTAs)
struct StepPlan {
  int32_t *cnt_cur, *cnt_prev, *cnt_next, *list_cur, *list_prev;
  uint32_t seq;
  int tail, grid;
  bool prof;
};
static inline StepPlan plan_step(PfbContext* h) {
  StepPlan p;
  const uint64_t k = h->step_seq;
  // four rotating done lists / counters: step k appends to [k % 4], its tail CTAs (and the side-stream spare rebuild, for the
  // envs that have one) read [(k - 1) % 4], and it zeroes counter [(k + 1) % 4]
  p.cnt_cur = h->d_counters + (k % 4);
  p.cnt_prev = h->d_counters + ((k + 3) % 4);
  p.cnt_next = h->d_counters + ((k + 1) % 4);
  p.list_cur = h->d_done_list + (k % 4) * h->n;
  p.list_prev = h->d_done_list + ((k + 3) % 4) * h->n;
  p.seq = (uint32_t)k;
  // tail CTAs (front of the grid) reset the envs that finished on the previous call; one per SM is
  // plenty for the ~1-3 % of envs that finish per step, and the loop is grid-strided anyway
  p.tail = 0;
  if (h->env.autoreset != 0) {
    p.tail = h->sm_count;
    int need = grid_for(h->n);
    if (p.tail > need) p.tail = need;
  }
  p.grid = grid_for(h->n) + p.tail;
  p.prof = h->prof_ev && h->prof_n < h->prof_cap;
  return p;
}

// template argument MODE (QuadX flight mode) from a run-time value
#define PFB_MODE_SWITCH(mode, BODY)                         \
  switch (mode) {                                           \
    case -1: { constexpr int MODE = -1; BODY; } break;      \
    case 0: { constexpr int MODE = 0; BODY; } break;        \
    case 1: { constexpr int MODE = 1; BODY; } break;        \
    case 2: { constexpr int MODE = 2; BODY; } break;        \
    case 3: { constexpr int MODE = 3; BODY; } break;        \
    case 4: { constexpr int MODE = 4; BODY; } break;        \
    case 5: { constexpr int MODE = 5; BODY; } break;        \
    case 6: { constexpr int MODE = 6; BODY; } break;        \
    case 7: { constexpr int MODE = 7; BODY; } break;        \
    default: return fail("`mode` must be between -1 and 7, got %d", mode); \
  }

// pfb_lib.cu: a masked user reset on an autoreset handle removes the masked envs / arenas from the pending done list
int pfb_drop_masked_done(PfbContext* h, const uint8_t* mask, cudaStream_t s);

// ---- NEXT_STEP autoreset by tail CTAs with spare post-reset states (DESIGN.md §4): QuadX-Waypoints, Fixedwing-Waypoints,
// Rocket-Landing and Dogfight.  The device half is pfb_tail_reset.cuh.
// The step kernels' bookkeeping arguments.  Normal launch: tail CTAs reset the entries of (prev_count, prev_list), finished
// envs are appended to (cur_count, cur_list), next_count is zeroed.  Build mode (build = 1, only tail CTAs): the spares of the
// entries of prev_list are rebuilt for the following episode, or of every env when prev_list is null.  The spare records
// themselves stay a separate __restrict__ kernel argument: the kernels read and write them next to the state tensor.
struct TailArgs {
  const int32_t* prev_count;
  const int32_t* prev_list;
  int32_t* cur_count;
  int32_t* cur_list;
  int32_t* next_count;
  int spare_copy;  // a tail CTA may copy a valid spare (0: inline_reset, every warm-up runs inline)
  int build;
  int tail_blocks;
  uint32_t step_seq;
};

// `launch(inject, randact, autoreset, grid, stream, spare, args)` launches the kind's step kernel with the spare records
// (nullptr: every reset runs its warm-up inline); the three flags are
// std::integral_constant<bool, ...> so that it can name the template instantiation.  Returns 0 or the result of fail().
using TailFalse = std::false_type;
using TailTrue = std::true_type;

template <typename Launch>
int tail_env_step(PfbContext* h, const float* noise, bool randact, cudaStream_t s, Launch&& launch) {
  if (h->env.autoreset && noise) return fail("injected noise (parity mode) is only supported with autoreset = 0");
  const StepPlan pl = plan_step(h);
  float* spare = h->env.autoreset ? h->d_spare : nullptr;
  // the rebuild of the spares consumed by step k - 2 must be complete before step k (an env cannot finish again sooner)
  if (spare && h->step_seq >= 2) CUDA_OK(cudaStreamWaitEvent(s, h->ev_spare[(h->step_seq - 2) % 4], 0));
  if (pl.prof) CUDA_OK(cudaEventRecord(h->prof_ev[2 * h->prof_n], s));
  TailArgs a{pl.cnt_prev, pl.list_prev, pl.cnt_cur, pl.list_cur, pl.cnt_next, (spare && !h->env.inline_reset) ? 1 : 0, 0, pl.tail, pl.seq};
  int e;
  if (h->env.autoreset) e = randact ? launch(TailFalse{}, TailTrue{}, TailTrue{}, pl.grid, s, spare, a) : launch(TailFalse{}, TailFalse{}, TailTrue{}, pl.grid, s, spare, a);
  else if (noise) e = launch(TailTrue{}, TailFalse{}, TailFalse{}, pl.grid, s, spare, a);
  else e = randact ? launch(TailFalse{}, TailTrue{}, TailFalse{}, pl.grid, s, spare, a) : launch(TailFalse{}, TailFalse{}, TailFalse{}, pl.grid, s, spare, a);
  if (e) return e;
  LAUNCH_CHECK(h);
  if (pl.prof) {
    CUDA_OK(cudaEventRecord(h->prof_ev[2 * h->prof_n + 1], s));
    h->prof_n += 1;
  }
  if (spare) {  // rebuild the spares this launch consumed, on the side stream, ordered behind it, while the next launches run
    CUDA_OK(cudaEventRecord(h->ev_step, s));
    CUDA_OK(cudaStreamWaitEvent(h->side, h->ev_step, 0));
    a.spare_copy = 0;
    a.build = 1;
    a.tail_blocks = h->sm_count;
    if (int e2 = launch(TailFalse{}, TailFalse{}, TailTrue{}, h->sm_count, h->side, spare, a)) return e2;
    LAUNCH_CHECK(h);
    CUDA_OK(cudaEventRecord(h->ev_spare[h->step_seq % 4], h->side));
  }
  h->step_seq += 1;
  return 0;
}

// `reset(seq, grid)` launches the kind's reset kernel with its episode number; `launch` is the kind's step launch as above
template <typename Reset, typename Launch>
int tail_env_reset(PfbContext* h, const uint8_t* mask, cudaStream_t s, Reset&& reset, Launch&& launch) {
  const uint32_t seq = 0x80000000u | (uint32_t)h->reset_seq++;
  const int g = grid_for(h->n);
  float* spare = h->env.autoreset ? h->d_spare : nullptr;
  if (spare) {
    // the spares are rewritten below: the last rebuild must have finished
    if (h->step_seq > 0) CUDA_OK(cudaStreamWaitEvent(s, h->ev_spare[(h->step_seq - 1) % 4], 0));
    if (!mask) CUDA_OK(cudaMemsetAsync(h->d_counters, 0, 4 * sizeof(int32_t), s));  // a full reset empties the autoreset queues
    else if (pfb_drop_masked_done(h, mask, s)) return -1;  // a masked one takes its envs out of the pending done list
  }
  if (int e = reset(seq, g)) return e;
  LAUNCH_CHECK(h);
  if (spare) {  // every env gets a fresh spare: the step kernel in build mode over all envs, same stream
    const TailArgs a{nullptr, nullptr, nullptr, nullptr, nullptr, 0, 1, g, 0u};
    if (int e = launch(TailFalse{}, TailFalse{}, TailTrue{}, g, s, spare, a)) return e;
    LAUNCH_CHECK(h);
  }
  h->mode = 0;
  return 0;
}

// fixedwing translation unit (pfb_fixedwing.cu)
int fw_build_params(const PfbModel& m, const PfbEnvConfig* env, pfb::FixedwingParams& p, pfb::WaypointParams& w);
int fw_state_rows();
int fw_istate_rows();
int fw_obs_dim(const PfbContext* h);
int fw_reset(PfbContext* h, const uint8_t* mask, cudaStream_t s);
int fw_set_mode(PfbContext* h, int mode, cudaStream_t s);
int fw_aviary_step(PfbContext* h, int n_steps, const float* noise, cudaStream_t s);
int fw_observe(PfbContext* h, cudaStream_t s);
int fw_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s);
int fw_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s);

// rocket translation unit (pfb_rocket.cu)
int rk_build_params(const PfbModel& m, const PfbEnvConfig* env, pfb::RocketParams& p, pfb::LandingParams& l);
int rk_state_rows();
int rk_istate_rows();
int rk_obs_dim(const PfbContext* h);
int rk_reset(PfbContext* h, const uint8_t* mask, cudaStream_t s);
int rk_set_mode(PfbContext* h, int mode, cudaStream_t s);
int rk_set_velocity(PfbContext* h, const float* lin, const float* ang, cudaStream_t s);
int rk_aviary_step(PfbContext* h, int n_steps, const float* noise, cudaStream_t s);
int rk_observe(PfbContext* h, cudaStream_t s);
int rk_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s);
int rk_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s);

// dogfight translation unit (pfb_dogfight.cu): fixedwing vehicles, arenas of 2*team_size adjacent envs
int df_build_params(const PfbEnvConfig* env, pfb::DogfightParams& d);
int df_obs_dim(const PfbContext* h);
int df_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s);
int df_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s);
int df_spare_rows();
int df_split_physics(PfbContext* h, const float* actions, const float* noise, float* payload, const uint64_t* peers, int world, int64_t slot0,
                     const uint64_t* peer_flags, int rank, int epoch, int first, int do_reset, int sub, cudaStream_t s);
int df_split_combat(PfbContext* h, const float* table, int64_t first_gid, int64_t num_arenas, int last, const int* wait_flags, int world, int epoch,
                    cudaStream_t s);

// QuadX-Waypoints translation unit (pfb_quadx_wp.cu)
int qwp_state_rows();
int qwp_istate_rows();
int qwp_obs_dim(const PfbContext* h);
int qwp_spare_rows();
int qwp_env_reset(PfbContext* h, const uint8_t* mask, const float* noise, cudaStream_t s);
int qwp_env_step(PfbContext* h, float* actions, const float* noise, bool randact, cudaStream_t s);
