// pfb_tail_reset.cuh — device half of the NEXT_STEP autoreset shared by the QuadX-Waypoints, Fixedwing-Waypoints,
// Rocket-Landing and Dogfight step kernels (DESIGN.md §4); the host half is tail_env_step / tail_env_reset in pfb_context.h.
//
// A step launch is `tail_blocks` tail CTAs followed by the regular CTAs.  A regular thread steps its own env (an env a tail CTA
// owns on this launch is skipped) and appends the envs that finish to this launch's done list.  Tail CTAs stride over the
// previous launch's done list and reset those envs, normally by copying the env's spare post-reset state; in build mode they
// compute those spares instead.  A work item is one env, or one arena of E adjacent envs (the dogfight).
#pragma once

#include "pfb_context.h"
#include "pfb_quadx.cuh"

namespace pfb {

// The helpers take threadIdx.x from the kernel (TailWork::tid): read there, its launch bounds tell the compiler it is below
// kBlock; a read inside a helper would not know that and, merged with the kernel's own reads, would lose it for them too.
struct TailWork {
  unsigned tid;         // threadIdx.x
  bool tail;            // this CTA is a tail CTA
  int64_t block_first;  // first env of a regular CTA
  int t, t_end, t_stride;
};

// E = envs per work item.  The previous launch's done list is read-only for this launch (__ldg).
template <int E, bool AUTORESET>
__device__ __forceinline__ TailWork tail_schedule(const TailArgs& a, int64_t N, unsigned tid) {
  TailWork w;
  w.tid = tid;
  w.tail = AUTORESET && (int)blockIdx.x < a.tail_blocks;
  w.block_first = w.tail ? 0 : (int64_t)((int)blockIdx.x - (AUTORESET ? a.tail_blocks : 0)) * kBlock;
  if (w.tail) {
    if (blockIdx.x == 0 && w.tid == 0 && !a.build) *a.next_count = 0;
    w.t = (blockIdx.x * kBlock + w.tid) / E;
    w.t_end = a.prev_list ? __ldg(a.prev_count) : (int)(N / E);  // build mode after a user reset: every item
    w.t_stride = a.tail_blocks * kBlock / E;
  } else {
    w.t = 0;
    w.t_end = (w.block_first + w.tid < N) ? 1 : 0;
    w.t_stride = 1;
  }
  return w;
}

// the env of work item w.t that the calling thread handles; `li` = its index inside the item
template <int E>
__device__ __forceinline__ int64_t tail_env(const TailArgs& a, const TailWork& w, int li) {
  return w.tail ? (a.prev_list ? (int64_t)__ldg(a.prev_list + w.t) : (int64_t)w.t * E) + li : w.block_first + w.tid;
}

// a regular thread leaves an env to the tail CTAs: it finished on the previous launch (`done` flags) or a tail CTA has already
// reset it on this one (this launch's fresh tag, pfb_quadx.cuh)
__device__ __forceinline__ bool tail_owns(uint32_t flags, uint32_t done, uint32_t step_seq) { return (flags & (done | fresh_tag(step_seq))) != 0; }

// ---- spare records: env-major, the kind's ROWS state words, then this header, then whatever the kind adds
template <int ROWS>
struct SpareHdr {
  static constexpr int VALID = ROWS, FLAGS = ROWS + 1, EPISODE = ROWS + 2, POSE = ROWS + 3 /* 6: start_pos, start_orn */, END = ROWS + 9;
};

struct SpareProbe {
  uint32_t episode;  // episode number of the reset (keys its Philox streams)
  bool hit;          // the record holds that episode, built from `pose`: copy it
};

// without a record the warm-up runs inline, keyed by the launch; build mode builds the episode after the stored one
template <int ROWS>
__device__ __forceinline__ SpareProbe spare_probe(const TailArgs& a, const float* rec, const float* pose, bool check_pose) {
  using H = SpareHdr<ROWS>;
  SpareProbe p{a.step_seq | 0x40000000u, false};
  if (rec) {
    p.episode = __float_as_uint(rec[H::EPISODE]) + (a.build ? 1u : 0u);
    p.hit = !a.build && a.spare_copy && rec[H::VALID] != 0.0f;
    if (check_pose) {
#pragma unroll
      for (int k = 0; k < 6; ++k) p.hit = p.hit && (rec[H::POSE + k] == pose[k]);
    }
  }
  return p;
}

// a record being built is invalid until spare_seal; `pose` (nullptr: not recorded) is the start pose it is built from
template <int ROWS>
__device__ __forceinline__ void spare_open(float* rec, const float* pose) {
  using H = SpareHdr<ROWS>;
  rec[H::VALID] = 0.0f;
  if (pose) {
#pragma unroll
    for (int k = 0; k < 6; ++k) rec[H::POSE + k] = pose[k];
  }
}

template <int ROWS>
__device__ __forceinline__ void spare_seal(float* rec, uint32_t flags, uint32_t episode) {
  using H = SpareHdr<ROWS>;
  rec[H::FLAGS] = __uint_as_float(flags);
  rec[H::EPISODE] = __uint_as_float(episode);
  rec[H::VALID] = 1.0f;
}

// warp-aggregated append of `i` to this launch's done list by the lanes of `active` whose `done` is set
__device__ __forceinline__ void append_done(const TailArgs& a, const TailWork& w, unsigned active, bool done, int64_t i) {
  const unsigned m = __ballot_sync(active, done);
  if (done) {
    const int lane = w.tid & 31;
    const int leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(a.cur_count, __popc(m));
    base = __shfl_sync(m, base, leader);
    a.cur_list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
  }
}

// a regular CTA's observation rows (O floats each, STRIDE apart in shared memory) to obs, coalesced; the rows of envs a tail
// CTA owns (`skip`) are left to it
template <int STRIDE>
__device__ __forceinline__ void flush_obs_tile(const float* smem, uint8_t* row_skip, bool skip, float* __restrict__ obs, const TailWork& w,
                                               int O, int64_t N) {
  const int64_t block_first = w.block_first;
  row_skip[w.tid] = skip ? 1 : 0;
  __syncthreads();
  int64_t rows = N - block_first;
  if (rows > kBlock) rows = kBlock;
  const int total = (int)rows * O;
  float* dst = obs + block_first * O;
  const int dr = kBlock / O, dc = kBlock - dr * O;
  int r = w.tid / O, c = w.tid - r * O;
  for (int j = w.tid; j < total; j += kBlock) {
    if (!row_skip[r]) dst[j] = smem[r * STRIDE + c];
    r += dr; c += dc;
    if (c >= O) { c -= O; ++r; }
  }
}

}  // namespace pfb
