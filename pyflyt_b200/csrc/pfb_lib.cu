// pfb_lib.cu — CUDA kernels (sm_100a) and the C-ABI of libpyflyt_b200.so (include/pyflyt_b200.h).
//
// One thread integrates one env; the whole env step (control ticks, physics substeps, reward,
// termination, observation) happens in registers between one coalesced SoA load and one store.
// Row-major API buffers (actions [N][4], observations [N][O]) are moved with 16-byte vector loads
// and a shared-memory transpose so that global traffic stays fully coalesced.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "../../include/pyflyt_b200.h"
#include "pfb_context.h"
#include "pfb_noise.cuh"

using namespace pfb;

// ---------------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
int pfb_fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return -1;
}
#include "pfb_quadx_host.h"

// ---------------------------------------------------------------------------------------------------
// kernels — Aviary surface
// ---------------------------------------------------------------------------------------------------
// QuadX handles keep their state WARP-TILED (pfb_quadx.cuh) except QuadX-Waypoints, whose kernels (pfb_quadx_wp.cu) still use
// the field-major [F][N] rows + istate; TILED selects the addressing of the kernels both layouts share.
template <int MODE, bool TILED>
__device__ __forceinline__ void qx_load_any(const float* __restrict__ st, const int32_t* __restrict__ ist, int rows, int64_t N, int64_t i,
                                            QuadXRegs& s, int& step_count) {
  if (TILED) {
    quadx_load_tile<MODE, kTileGroupStride>(st + qx_tile_base(i, rows), s, step_count);
  } else {
    quadx_load<MODE>(st, ist, N, i, s);
    step_count = ist[(int64_t)QI_STEP * N + i];
  }
}
template <int MODE, bool TILED>
__device__ __forceinline__ void qx_store_any(float* __restrict__ st, int32_t* __restrict__ ist, int rows, int64_t N, int64_t i,
                                             const QuadXRegs& s, int step_count) {
  if (TILED) {
    quadx_store_tile<MODE, kTileGroupStride>(st + qx_tile_base(i, rows), s, step_count);
  } else {
    quadx_store<MODE>(st, ist, N, i, s);
    ist[(int64_t)QI_STEP * N + i] = step_count;
  }
}

// Aviary.reset + QuadX.reset + update_state (aviary.py:218-312, quadx.py:222-231)
template <bool TILED>
__global__ void __launch_bounds__(kBlock) k_quadx_reset(float* __restrict__ st, int32_t* __restrict__ ist, int rows,
                                                        float* __restrict__ setpoint, const float* __restrict__ start_pos,
                                                        const float* __restrict__ start_orn,
                                                        const uint8_t* __restrict__ mask, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  QuadXRegs s;
  quadx_reset(s, start_pos[3 * i + 0], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i + 0],
              start_orn[3 * i + 1], start_orn[3 * i + 2]);
  qx_store_any<7, TILED>(st, ist, rows, N, i, s, 0);  // mode 7 touches every PID row
  if (setpoint) reinterpret_cast<float4*>(setpoint)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// Aviary.set_mode -> QuadX.set_mode (quadx.py:233-373): preset the setpoint, fresh attitude/position PIDs
template <int MODE, bool TILED>
__global__ void __launch_bounds__(kBlock) k_quadx_set_mode(float* __restrict__ st, int32_t* __restrict__ ist, int rows,
                                                           float* __restrict__ setpoint, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  QuadXRegs s;
  int step_count;
  qx_load_any<7, TILED>(st, ist, rows, N, i, s, step_count);
  float4 sp = reinterpret_cast<const float4*>(setpoint)[i];
  s.sp[0] = sp.x; s.sp[1] = sp.y; s.sp[2] = sp.z; s.sp[3] = sp.w;
  quadx_set_mode<MODE>(s);
  qx_store_any<7, TILED>(st, ist, rows, N, i, s, step_count);
  reinterpret_cast<float4*>(setpoint)[i] = make_float4(s.sp[0], s.sp[1], s.sp[2], s.sp[3]);
}

// n_steps x Aviary.step() (aviary.py:480-531)
template <int MODE, bool INJECT, bool TILED>
__global__ void __launch_bounds__(kBlock, kMinBlocks)
    k_quadx_aviary_step(const __grid_constant__ QuadXParams p, const __grid_constant__ RngParams rng,
                        float* __restrict__ st, int32_t* __restrict__ ist, int rows, const float* __restrict__ setpoint,
                        const float* __restrict__ noise, int n_steps, uint32_t seq, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  QuadXRegs s;
  int step_count;
  qx_load_any<MODE, TILED>(st, ist, rows, N, i, s, step_count);
  float4 sp = __ldg(reinterpret_cast<const float4*>(setpoint) + i);
  s.sp[0] = sp.x; s.sp[1] = sp.y; s.sp[2] = sp.z; s.sp[3] = sp.w;
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_AVIARY, p.noise_loc, p.ratio);
  for (int k = 0; k < n_steps; ++k) quadx_aviary_step<MODE>(p, s, nz);
  qx_store_any<MODE, TILED>(st, ist, rows, N, i, s, step_count);
}

// Aviary.state(i) / aux_state(i) / contact_array  -> row-major API buffers
template <bool TILED>
__global__ void __launch_bounds__(kBlock) k_quadx_observe(const float* __restrict__ st, const int32_t* __restrict__ ist, int rows,
                                                          float* __restrict__ drone_state, float* __restrict__ aux,
                                                          uint8_t* __restrict__ contact, int64_t N) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  QuadXRegs s;
  int step_count;
  qx_load_any<-1, TILED>(st, ist, rows, N, i, s, step_count);
  float o[12], a[4];
  quadx_drone_state(s, o, a);
  if (drone_state) {
    float4* d = reinterpret_cast<float4*>(drone_state + 12 * i);
    d[0] = make_float4(o[0], o[1], o[2], o[3]);
    d[1] = make_float4(o[4], o[5], o[6], o[7]);
    d[2] = make_float4(o[8], o[9], o[10], o[11]);
  }
  if (aux) reinterpret_cast<float4*>(aux)[i] = make_float4(a[0], a[1], a[2], a[3]);
  if (contact) contact[i] = (s.flags & FLAG_CONTACT_ARRAY) ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------------
// kernels — QuadX-Hover env (warp-tiled state)
// ---------------------------------------------------------------------------------------------------
// 512 threads per SM resident (<= 128 registers): the 2048 CTAs of a 65 536-env step and the 148 of the concurrent spare rebuild
// must all be resident at once, or the stragglers form a second wave
#ifndef PFB_HOVER_THREADS
#define PFB_HOVER_THREADS 512
#endif
constexpr int kHoverBlocks = PFB_HOVER_THREADS / kBlock;
constexpr int kObsMax = 24;  // floats per observation row (20 / 21, + 3 for MAQuadXHover)

// ---- spare post-reset states (DESIGN.md §4, "reset pipeline") ---------------------------------------
// env.reset() = start pose + `warmup_steps` Aviary steps (quadx_base_env.py:149-212): 3.3x the work of an env step and a
// strictly serial chain; run inline, even one finished env stretches the launch to the length of that chain.  So each env
// owns a SPARE, the post-warm-up state of its NEXT episode, with the warm-up noise keyed by (env id, episode number,
// Aviary step) so that it does not matter when it is computed.
//  * An env that finished on call k is reset on call k + 1 BY ITS OWN THREAD: the thread skips the physics loop and, at the
//    end of the launch, swaps the env's spare record in (staged into the warp's dead state-tile buffer by cp.async while the
//    other lanes integrate, kStageFloats below) — every observation row of a warp's tile is written by that warp.
//  * The spare it consumed is rebuilt INSIDE the following two step launches by a few BUILDER CTAs appended to the grid:
//    launch k + 1 (the one that consumes) integrates the first half of the next spare's warm-up, launch k + 2 the second
//    half — each half is shorter than an env step, so the builders never stretch a launch — and the spare is valid again
//    before launch k + 3, the earliest the env can be reset again.  A spare lives in buffer (episode & 3), so the builders
//    never write the record a resetting thread is reading.  One launch per env step: no side stream, no events.
//  * If the start pose was edited since a spare was built, or with inline_reset = 1, the spare is ignored and the warm-up
//    runs inline in the owning thread (same episode number, hence the same result).
// Library-owned: spare[kSpareBufs][N][SP_ROWS] ENV-MAJOR records (the QX_* state rows in record layout, group stride 4, then
// the words below) and episode[N], the episode number of each env's current valid spare (its buffer is episode & kSpareMask).
enum { SP_POSE = QX_ROWS, SP_VALID = QX_ROWS + 6, SP_FLAGS = QX_ROWS + 7, SP_EPISODE = QX_ROWS + 8,
       SP_SETPOINT = QX_ROWS + 12 /* 4: the flight mode's preset setpoint, carried between the two halves of a warm-up */, SP_ROWS = 80 };
static_assert(QX_ROWS % 4 == 0 && QX_ROWS + 16 <= SP_ROWS && SP_ROWS % 4 == 0, "spare record layout");
constexpr int kSpareBufs = 4;  // records per env, buffer = episode & 3: the step pipeline uses two neighbours (one being consumed, one being built);
constexpr uint32_t kSpareMask = kSpareBufs - 1;  // the fused rollout keeps three spares ahead (k_hover_rollout)
#ifndef PFB_WARM_SPLIT
#define PFB_WARM_SPLIT 5
#endif
constexpr int kWarmSplit = PFB_WARM_SPLIT;  // Aviary steps integrated by the first builder phase; every warm-up requantizes its state there

// cp.async.bulk (TMA, 1-D) shared -> global: one instruction moves a warp's whole observation tile
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
  const uint32_t sa = (uint32_t)__cvta_generic_to_shared(ssrc);
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(sa), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// cp.async.bulk (TMA, 1-D) global -> shared with mbarrier completion: the warp's state tile lands asynchronously while
// the warp runs its noise generator; try_wait is the point the loaded data is first needed
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_load_g2s(void* sdst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(sdst), b = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(gsrc), "r"(bytes), "r"(b)
               : "memory");
}
// `dep`: values that must have been COMPUTED before the wait starts (the asm consumes them, no instruction is emitted for
// them): keeps work that does not need the tile — the noise generator — in front of the wait instead of behind it
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, float d0 = 0.f, float d1 = 0.f, float d2 = 0.f, float d3 = 0.f,
                                          float d4 = 0.f, float d5 = 0.f, float d6 = 0.f, float d7 = 0.f) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(a),
      "r"(parity), "f"(d0), "f"(d1), "f"(d2), "f"(d3), "f"(d4), "f"(d5), "f"(d6), "f"(d7)
      : "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#ifdef PFB_TIMELINE
// experiment build (tools/exp_timeline.py): every warp of the step launch stamps %globaltimer at four points into the buffer
// that normally receives the noise dump: [warp][4] uint64 = entry, inputs landed, integration done, exit
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define PFB_TL(slot) do { if (noise_dump && threadIdx.x == 0) reinterpret_cast<unsigned long long*>(noise_dump)[(size_t)blockIdx.x * 4 + (slot)] = gtimer(); } while (0)
#else
#define PFB_TL(slot) do { } while (0)
#endif
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
// per-thread asynchronous copies global -> shared (LDGSTS): issued and forgotten, complete in the background, waited for with
// cp_async_wait_all() by the issuing thread, which may then read what it copied
__device__ __forceinline__ void cp_async16(float* sdst, const float* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(float* sdst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(sdst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// Staging of spare records (reset by the owning thread): a resetting lane copies its 320-byte record — in the step kernel also the
// start pose the record is checked against — into the warp's state-tile buffer, which is dead once the tile has been unpacked.
// The copies fly while the other lanes integrate; the swap at the end of the step then reads shared memory instead of making two
// or three DEPENDENT trips to L2 / DRAM (valid word -> pose -> state: ~600 cycles each in the ncu source view of round 2).
constexpr int kStageFloats = SP_ROWS + 8;

// env.reset() integrated inline (quadx_base_env.py:149-212): Aviary steps [from, to) of the warm-up that follows the start
// pose + set_mode.  The state is rounded to what a record holds (hi + lo words) before step kWarmSplit in EVERY path, so a
// warm-up integrated in two launches through a spare record equals one integrated in one go, bit for bit.
// The INLINE form is what the builder CTAs and the reset / build kernels run: `p` must be the kernel's __grid_constant__
// parameter so that the coefficients stay constant-bank operands.
template <int MODE, bool INJECT>
__device__ __forceinline__ void hover_warmup_inline(const QuadXParams& p, QuadXRegs& s, int from, int to, const RngParams& rng,
                                                    const float* __restrict__ noise, int64_t N, int64_t i, uint32_t seq) {
  auto nz = make_noise<INJECT>(noise, N, i, rng, seq, TAG_RESET, p.noise_loc, p.ratio);
  nz.seek((uint32_t)from);
#pragma unroll 1
  for (int k = from; k < to; ++k) {
    if (k == kWarmSplit) quadx_requantize(s);
    quadx_aviary_step<MODE>(p, s, nz);
  }
}
// Out-of-line form for the COLD fallback inside the step role (a spare that cannot be used): everything by value, so the
// caller's register-resident state never has its address taken.  Slow (the coefficient table is read from the stack copy),
// and rare.
template <int MODE>
__device__ __noinline__ QuadXRegs hover_warmup_cold(const QuadXParams p, QuadXRegs s, int to, const RngParams rng, int64_t N, int64_t i,
                                                    uint32_t seq) {
  hover_warmup_inline<MODE, false>(p, s, 0, to, rng, nullptr, N, i, seq);
  return s;
}
// a freshly constructed drone in flight mode MODE at its start pose (quadx.py:222-231, quadx_base_env.py:186-207)
template <int MODE>
__device__ __forceinline__ QuadXRegs hover_fresh(float px, float py, float pz, float ox, float oy, float oz) {
  QuadXRegs s;
  quadx_reset(s, px, py, pz, ox, oy, oz);
  quadx_set_mode<MODE>(s);
  return s;
}

// Builder CTAs of the step launch (the first 2 * builders CTAs of the grid): the first `builders` of them (phase 0) start the next
// spare of the envs that are being reset by this launch (done list of the previous launch), the others (phase 1) finish the
// spares started by the previous launch.  ONE copy of the warm-up loop serves both phases.
template <int MODE>
__device__ __forceinline__ void hover_build(const QuadXParams& p, const HoverParams& h, const RngParams& rng, int b, int builders,
                                            const int32_t* __restrict__ b0_count, const int32_t* __restrict__ b0_list,
                                            const int32_t* __restrict__ b1_count, const int32_t* __restrict__ b1_list,
                                            uint32_t* __restrict__ b0_elist, const uint32_t* __restrict__ b1_elist,
                                            const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                                            float* __restrict__ spare, uint32_t* __restrict__ episode, int64_t N, float* noise_dump = nullptr) {
  const int phase = b >= builders ? 1 : 0;
  const int slot = b - phase * builders;
  const int32_t* __restrict__ list = phase ? b1_list : b0_list;
  // The builders' chain of DEPENDENT cold loads (count -> list entry -> episode number -> record) is what they wait for while the
  // step CTAs' tile burst saturates DRAM: the first list entry (and, in phase 1, the episode number phase 0 left next to it) is
  // loaded speculatively together with the count — the lists are N entries long, so any index below N is readable
  int t = slot * kBlock + (int)threadIdx.x;
  const int64_t t_spec = t < N ? t : N - 1;
  int32_t i_spec = list[t_spec];
  uint32_t e_spec = phase ? b1_elist[t_spec] : 0u;
  const int t_end = phase ? *b1_count : *b0_count;
  const int split = h.warmup_steps < kWarmSplit ? h.warmup_steps : kWarmSplit;
#pragma unroll 1
  for (; t < t_end; t += builders * kBlock) {
    const int64_t i = i_spec;
    // the spare being built; the one being consumed (episode[i]) lives in the other buffer
    const uint32_t e = phase ? e_spec : episode[i] + 1u;
    float* rec = spare + ((int64_t)(e & kSpareMask) * N + i) * SP_ROWS;
    QuadXRegs s;
    float px = 0.f, py = 0.f, pz = 0.f, ox = 0.f, oy = 0.f, oz = 0.f;
    if (phase == 0) {
      px = start_pos[3 * i + 0]; py = start_pos[3 * i + 1]; pz = start_pos[3 * i + 2];
      ox = start_orn[3 * i + 0]; oy = start_orn[3 * i + 1]; oz = start_orn[3 * i + 2];
      s = hover_fresh<MODE>(px, py, pz, ox, oy, oz);
      b0_elist[t] = e;  // read by phase 1 of the next launch (same list, same position)
    } else {
      int dummy;
      quadx_load_tile<7, 4>(rec, s, dummy);
      const F4 sp = ld_f4(rec + SP_SETPOINT);
      s.sp[0] = sp.x; s.sp[1] = sp.y; s.sp[2] = sp.z; s.sp[3] = sp.w;
    }
#ifdef PFB_TIMELINE
    if (s.flags == 0xffffffffu) return;  // consume the loaded state before the stamp
#endif
    PFB_TL(1);
    hover_warmup_inline<MODE, false>(p, s, phase ? split : 0, phase ? h.warmup_steps : split, rng, nullptr, N, i, e);
    PFB_TL(2);
    quadx_store_tile<7, 4>(rec, s, 0);
    if (phase == 0) {
      st_f4(rec + SP_POSE, px, py, pz, ox);
      st_f4(rec + SP_POSE + 4, oy, oz, 0.0f, 0.0f);  // not valid yet
      st_f4(rec + SP_POSE + 8, f_from_bits(e), 0.0f, 0.0f, 0.0f);
      st_f4(rec + SP_SETPOINT, s.sp[0], s.sp[1], s.sp[2], s.sp[3]);
    } else {
      rec[SP_FLAGS] = f_from_bits(s.flags);
      rec[SP_VALID] = 1.0f;
      episode[i] = e;
    }
    const int tn = t + builders * kBlock;  // more finished envs than builder lanes (a synchronised truncation): next pass
    if (tn < t_end) {
      i_spec = list[tn];
      if (phase) e_spec = b1_elist[tn];
    }
  }
}

// env.step(action) for every env (quadx_base_env.py:269-301 + quadx_hover_env.py), ONE launch, one warp per CTA, one tile
// of 32 envs per warp.
//   RANDACT   actions are drawn on device, uniform in the env's action box (quadx_base_env.py:79-102)
//   AUTORESET gymnasium NEXT_STEP autoreset: an env that finished on the previous call is reset on this one (its action
//             is ignored; obs = first observation of the new episode, reward 0, flags cleared)
template <int MODE, bool INJECT, bool RANDACT, bool AUTORESET, bool MA>
__global__ void __launch_bounds__(kBlock, kHoverBlocks)
    k_hover_step(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h,
                 const __grid_constant__ RngParams rng, float* __restrict__ st, int rows, float* __restrict__ actions,
                 const float* __restrict__ noise, float* __restrict__ obs, float* __restrict__ reward, uint8_t* __restrict__ term,
                 uint8_t* __restrict__ trunc, uint8_t* __restrict__ info, const float* __restrict__ start_pos,
                 const float* __restrict__ start_orn, int32_t* __restrict__ cur_count, int32_t* __restrict__ cur_list,
                 int32_t* __restrict__ next_count, const int32_t* __restrict__ b0_count, const int32_t* __restrict__ b0_list,
                 const int32_t* __restrict__ b1_count, const int32_t* __restrict__ b1_list, uint32_t* __restrict__ b0_elist,
                 const uint32_t* __restrict__ b1_elist, float* __restrict__ spare, uint32_t* __restrict__ episode, int spare_copy, int builders,
                 float* __restrict__ noise_dump, uint32_t step_seq, int64_t N) {
  // builder CTAs come FIRST in the grid: their serial warm-up chain is the longest thing in the launch, so they must be
  // dispatched at t = 0, not behind the ~2000 step CTAs
  const int n_build = AUTORESET ? 2 * builders : 0;
  PFB_TL(0);
  if (AUTORESET && (int)blockIdx.x < n_build) {  // builder CTA (CTA-uniform role)
    hover_build<MODE>(p, h, rng, (int)blockIdx.x, builders, b0_count, b0_list, b1_count, b1_list, b0_elist, b1_elist, start_pos, start_orn, spare,
                      episode, N, noise_dump);
    PFB_TL(3);
    return;
  }
  const int tile = (int)blockIdx.x - n_build;
  if (h.stagger_ns > 0) {  // experiment: de-synchronise the memory phases of the single wave
    const int late = tile % h.stagger_mod;
    if (late) __nanosleep((unsigned)(late * h.stagger_ns));
  }
  __shared__ __align__(128) float smem[kBlock * kObsMax];
  const int O = (h.angle_representation == 0 ? 20 : 21) + (MA ? 3 : 0);
  const int lane = threadIdx.x;
  const int64_t tile_first = (int64_t)tile * kBlock;
  const int64_t i = tile_first + lane;
  const bool active = i < N;
  if (AUTORESET && tile == 0 && lane == 0) *next_count = 0;  // arm the counter the NEXT launch appends to
  float* rec = st + qx_tile_base(i, rows);  // the state tensor is padded to whole tiles: every lane may load

  // ---- the warp's state tile (groups 0 .. n-1: everything MODE reads) comes in with ONE cp.async.bulk (TMA) into shared
  //      memory; the noise generator and the action fetch run while it is in flight
  constexpr int kInGroups = qx_groups_moved<MODE>();
  __shared__ __align__(128) float stile[kInGroups * kTileGroupStride];
  __shared__ __align__(8) uint64_t mbar;
  if (lane == 0) {
    mbar_init(&mbar, 1);
    bulk_load_g2s(stile, st + qx_tile_base(tile_first, rows), (uint32_t)(kInGroups * kTileGroupStride * sizeof(float)), &mbar);
  }
  __syncwarp();
  float act[4] = {0.f, 0.f, 0.f, 0.f};
  float past[4] = {0.f, 0.f, 0.f, 0.f};
  auto nz = make_noise<INJECT>(noise, N, active ? i : 0, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
  nz.prefetch4();
#ifndef PFB_TIMELINE
  if (!INJECT && noise_dump && active) nz.set_dump(noise_dump + i, N);
#endif
  if (RANDACT) {
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
    if (active) reinterpret_cast<float4*>(actions)[i] = make_float4(act[0], act[1], act[2], act[3]);
  } else if (active) {
    float4 a4 = __ldg(reinterpret_cast<const float4*>(actions) + i);
    act[0] = a4.x; act[1] = a4.y; act[2] = a4.z; act[3] = a4.w;
  }
  // the episode number of this env's spare, for EVERY lane, in the shadow of the tile load: a lane that turns out to be
  // resetting can then pull its record towards L1 at once (nobody writes episode[i] of a resetting env during this launch)
  uint32_t e_next = (AUTORESET && spare && active) ? episode[i] : 0u;
  QuadXRegs s;
  int step_count;
  mbar_wait(&mbar, 0, nz.dep(0), nz.dep(1), nz.dep(2), nz.dep(3), nz.dep(4), nz.dep(5), nz.dep(6), nz.dep(7));  // the tile has landed
  quadx_load_tile<MODE, kTileGroupStride>(stile + lane * 4, s, step_count);  // LDS.128, conflict-free (lane-contiguous vectors)
  PFB_TL(1);
  // an env that finished on the previous call: this call is its reset (NEXT_STEP)
  const bool resetting = AUTORESET && active && (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0;
  const float* staged = nullptr;  // this lane's spare record + start pose in shared memory (see kStageFloats)
  if (AUTORESET && spare) {
    constexpr int kSlots = kInGroups * kTileGroupStride / kStageFloats;
    const unsigned reset_m = __ballot_sync(0xffffffffu, resetting);
    if (reset_m != 0u) {
      __syncwarp();  // every lane has unpacked its part of the tile: the buffer is free
      if (resetting) {
        const float* r = spare + ((int64_t)(e_next & kSpareMask) * N + i) * SP_ROWS;
        const int rank = __popc(reset_m & ((1u << lane) - 1u));
        if (rank < kSlots) {
          float* q = stile + rank * kStageFloats;
#pragma unroll
          for (int g = 0; g < SP_ROWS / 4; ++g) cp_async16(q + 4 * g, r + 4 * g);
#pragma unroll
          for (int k = 0; k < 3; ++k) { cp_async4(q + SP_ROWS + k, start_pos + 3 * i + k); cp_async4(q + SP_ROWS + 3 + k, start_orn + 3 * i + k); }
          staged = q;
        } else {  // more resetting lanes than slots (a synchronised truncation): towards L1 at least
          prefetch_l1(r); prefetch_l1(r + 32); prefetch_l1(r + 64); prefetch_l1(r + SP_ROWS - 1);
        }
      }
    }
  }
  int n_aviary = (active && !resetting) ? h.env_step_ratio : 0;
  float rew = -0.1f;
#pragma unroll
  for (int k = 0; k < 4; ++k) s.sp[k] = act[k];
  if (MA) {  // MAQuadXHover: flags are re-evaluated every step, rewards add up from 0, the obs shows the PREVIOUS action
    s.flags &= ~(uint32_t)(FLAG_TERM | FLAG_TRUNC | FLAG_OOB | FLAG_COLLISION);
    rew = 0.0f;
    const F4 cur = ld_f4(rec + (QM_CUR / 4) * kTileGroupStride);
    past[0] = cur.x; past[1] = cur.y; past[2] = cur.z; past[3] = cur.w;
    if (active) {
      st_f4(rec + (QM_PAST / 4) * kTileGroupStride, past[0], past[1], past[2], past[3]);
      st_f4(rec + (QM_CUR / 4) * kTileGroupStride, act[0], act[1], act[2], act[3]);
    }
  }
  float sx = 0.f, sy = 0.f, sz = 0.f;
  if (MA && active) { sx = start_pos[3 * i]; sy = start_pos[3 * i + 1]; sz = start_pos[3 * i + 2]; }
#pragma unroll 1
  for (int k = 0; k < n_aviary; ++k) {
    if (!MA && (s.flags & (FLAG_TERM | FLAG_TRUNC))) break;  // quadx_base_env.py:289-290
    quadx_aviary_step<MODE>(p, s, nz);
    if (MA) ma_hover_term_trunc_reward(h, s, step_count, sx, sy, sz, rew);
    else hover_term_trunc_reward(h, s, step_count, rew);
  }
  step_count += 1;
  PFB_TL(2);
  if (AUTORESET && __any_sync(0xffffffffu, resetting)) {
    if (resetting) {
      // env.reset(): begin_reset + end_reset (quadx_base_env.py:149-212) — normally a copy of the env's spare
      float px, py, pz, ox, oy, oz;
      if (staged) {
        cp_async_wait_all();
        px = staged[SP_ROWS + 0]; py = staged[SP_ROWS + 1]; pz = staged[SP_ROWS + 2];
        ox = staged[SP_ROWS + 3]; oy = staged[SP_ROWS + 4]; oz = staged[SP_ROWS + 5];
      } else {
        px = start_pos[3 * i + 0]; py = start_pos[3 * i + 1]; pz = start_pos[3 * i + 2];
        ox = start_orn[3 * i + 0]; oy = start_orn[3 * i + 1]; oz = start_orn[3 * i + 2];
      }
      bool hit = false;
      uint32_t nseq = step_seq | 0x40000000u;
      if (spare) {
        nseq = e_next;  // episode number: keys the warm-up noise
        const float* srec = staged ? staged : spare + ((int64_t)(e_next & kSpareMask) * N + i) * SP_ROWS;
        const F4 m0 = ld_f4(srec + SP_POSE), m1 = ld_f4(srec + SP_POSE + 4), m2 = ld_f4(srec + SP_POSE + 8);
        hit = spare_copy && m1.z != 0.0f && bits_from_f(m2.x) == e_next && m0.x == px && m0.y == py && m0.z == pz && m0.w == ox && m1.x == oy &&
              m1.y == oz;
        if (hit) {
          int dummy;
          quadx_load_tile<MODE, 4>(srec, s, dummy);
          const F4 pw = ld_f4(srec + QX_PWM);
          s.pwm[0] = pw.x; s.pwm[1] = pw.y; s.pwm[2] = pw.z; s.pwm[3] = pw.w;
          s.flags = bits_from_f(m1.w);
        }
      }
      if (!hit) {
        s = hover_warmup_cold<MODE>(p, hover_fresh<MODE>(px, py, pz, ox, oy, oz), h.warmup_steps, rng, N, i, nseq);
        quadx_requantize(s);  // an inline warm-up must leave exactly what a copied spare holds
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) { s.sp[k] = 0.0f; act[k] = 0.0f; }  // self.action = zeros (quadx_base_env.py:165)
      step_count = 0;
      rew = 0.0f;
    }
  }
  float* row = smem + lane * O;  // dense [32][O] tile, written out below by one bulk copy
  if (MA) ma_hover_observation(h, s, past, sx, sy, sz, row);
  else hover_observation(h, s, act, row);
  fence_async_smem();  // generic-proxy writes of this lane -> visible to the bulk-copy (async) proxy
  __syncwarp();
  // ---- this warp's observation tile obs[tile_first .. +rows][O] is contiguous in global memory and 16-byte aligned: ONE
  //      cp.async.bulk (TMA) moves it, issued before the state stores so that the engine's reads of shared memory overlap them
  int64_t nrows = N - tile_first;
  if (nrows > kBlock) nrows = kBlock;
  const uint32_t bytes = (uint32_t)nrows * (uint32_t)O * 4u;
  float* dst = obs + tile_first * O;
  const bool bulk = (bytes & 15u) == 0u;
  if (bulk) {
    if (lane == 0) bulk_store_s2g(dst, smem, bytes);
  } else {  // ragged last tile whose byte count is not a multiple of 16
    for (int j = lane; j < (int)nrows * O; j += kBlock) dst[j] = smem[j];
  }
  if (active) {
    quadx_store_tile<MODE, kTileGroupStride>(rec, s, step_count);
    reward[i] = rew;
    term[i] = (s.flags & FLAG_TERM) ? 1 : 0;
    trunc[i] = (s.flags & FLAG_TRUNC) ? 1 : 0;
    if (info) info[i] = (uint8_t)(((s.flags & FLAG_OOB) ? 1 : 0) | ((s.flags & FLAG_COLLISION) ? 2 : 0));
  }
  if (AUTORESET) {  // queue finished episodes: their spares are consumed by the next launch and rebuilt after it
    const bool done = active && (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0;
    const unsigned m = __ballot_sync(0xffffffffu, done);
    if (done) {
      const int leader = __ffs(m) - 1;
      int base = 0;
      if (lane == leader) base = atomicAdd(cur_count, __popc(m));
      base = __shfl_sync(m, base, leader);
      cur_list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
    }
  }
  if (bulk && lane == 0) bulk_store_wait_read();  // the CTA's shared memory must outlive the engine's reads
  PFB_TL(3);
}

// ---------------------------------------------------------------------------------------------------
// Fused rollout (SURVEY 8b: "n_env_steps > 1 = persistent rollout with on-device random actions"): T env steps of every env in
// ONE launch.  A warp loads its tile once, keeps the state in registers for the T steps and stores it once; each step still
// draws its action and noise from the same Philox counters as a single-step launch, integrates, and writes the step's
// observation tile (TMA), reward, flags and the action it drew, so after the launch every output buffer holds the results of
// the LAST of T env steps, like T calls of pfb_env_step.  The state is rounded to the record format at the end of every step —
// what the store / load of two launches does — so a fused launch performs the same arithmetic as T single-step launches; the
// results agree bit for bit except where two compiled copies of the same expression round differently (nvcc contracts
// multiply-adds per inlined copy: ~4e-5 of the env-steps see a one-ulp fp32 difference in a PID term; DESIGN.md 4,
// tests/test_gpu_parity.py::test_fused_rollout_equals_stepwise), and the fused path is pinned to the fp64 oracle on its own
// (tests/test_timed_path_parity.py::test_hover_fused_rollout_matches_oracle).
// Resets: an env that finished on step t takes, on step t + 1, the spare of its next episode out of kSpareBufs records kept
// kRolloutAhead ahead (k_hover_spare_ahead before the first fused launch, k_hover_spare_topup behind every one: all reset work
// stays inside the timed region); a missing spare (more than kRolloutAhead resets of one env inside a launch) is integrated
// inline by the cold path — the same episode number keys the same noise.
// ---------------------------------------------------------------------------------------------------
constexpr int kRolloutAhead = 3;
constexpr int kRolloutMaxSteps = 16;

// one env, one spare: episode `e` of env i, complete warm-up, into its buffer
template <int MODE>
__device__ __forceinline__ void hover_build_full(const QuadXParams& p, const HoverParams& h, const RngParams& rng, const float* __restrict__ start_pos,
                                                 const float* __restrict__ start_orn, float* __restrict__ spare, int64_t N, int64_t i, uint32_t e) {
  float* rec = spare + ((int64_t)(e & kSpareMask) * N + i) * SP_ROWS;
  const float px = start_pos[3 * i + 0], py = start_pos[3 * i + 1], pz = start_pos[3 * i + 2];
  const float ox = start_orn[3 * i + 0], oy = start_orn[3 * i + 1], oz = start_orn[3 * i + 2];
  QuadXRegs s = hover_fresh<MODE>(px, py, pz, ox, oy, oz);
  hover_warmup_inline<MODE, false>(p, s, 0, h.warmup_steps, rng, nullptr, N, i, e);
  quadx_store_tile<7, 4>(rec, s, 0);
  st_f4(rec + SP_POSE, px, py, pz, ox);
  st_f4(rec + SP_POSE + 4, oy, oz, 1.0f, f_from_bits(s.flags));
  st_f4(rec + SP_POSE + 8, f_from_bits(e), 0.0f, 0.0f, 0.0f);
}
// before the first fused launch (or after single-step launches): every env gets the spares episode[i] + 1 .. + kRolloutAhead - 1
// it does not have yet (episode[i] itself is valid by the step pipeline's invariant)
template <int MODE>
__global__ void __launch_bounds__(kBlock, kHoverBlocks)
    k_hover_spare_ahead(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ RngParams rng,
                        const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ spare,
                        const uint32_t* __restrict__ episode, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  const uint32_t e0 = episode[i];
#pragma unroll 1
  for (int a = 1; a < kRolloutAhead; ++a) {
    const uint32_t e = e0 + (uint32_t)a;
    const float* rec = spare + ((int64_t)(e & kSpareMask) * N + i) * SP_ROWS;
    const F4 m0 = ld_f4(rec + SP_POSE), m1 = ld_f4(rec + SP_POSE + 4), m2 = ld_f4(rec + SP_POSE + 8);
    const bool have = m1.z != 0.0f && bits_from_f(m2.x) == e && m0.x == start_pos[3 * i] && m0.y == start_pos[3 * i + 1] && m0.z == start_pos[3 * i + 2] &&
                      m0.w == start_orn[3 * i] && m1.x == start_orn[3 * i + 1] && m1.y == start_orn[3 * i + 2];
    if (!have) hover_build_full<MODE>(p, h, rng, start_pos, start_orn, spare, N, i, e);
  }
}
// behind a fused launch: the spares it consumed, listed as (env, episode to build)
template <int MODE>
__global__ void __launch_bounds__(kBlock, kHoverBlocks)
    k_hover_spare_topup(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ RngParams rng,
                        const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ spare,
                        const int32_t* __restrict__ count, const int2* __restrict__ list, int64_t N) {
  const int n = *count;
  for (int t = (int)(blockIdx.x * kBlock + threadIdx.x); t < n; t += (int)(gridDim.x * kBlock)) {
    const int2 en = list[t];
    hover_build_full<MODE>(p, h, rng, start_pos, start_orn, spare, N, (int64_t)en.x, (uint32_t)en.y);
  }
}
// switching from single-step launches to the fused rollout: the spares whose first half was integrated by the last step launch
// are finished here (phase 1 of hover_build on the list the next step launch would have used), so that episode[] is current
template <int MODE>
__global__ void __launch_bounds__(kBlock, kHoverBlocks)
    k_hover_drain(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ RngParams rng,
                  const int32_t* __restrict__ b1_count, const int32_t* __restrict__ b1_list, const uint32_t* __restrict__ b1_elist,
                  const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ spare, uint32_t* __restrict__ episode,
                  int builders, int64_t N) {
  hover_build<MODE>(p, h, rng, (int)blockIdx.x + builders, builders, b1_count, b1_list, b1_count, b1_list, nullptr, b1_elist, start_pos, start_orn, spare,
                    episode, N);
}

// 14 CTAs per SM: the 2048 tiles of a 65 536-env launch (no builder CTAs here) are still one wave, with 144 registers instead of 128
template <int MODE>
__global__ void __launch_bounds__(kBlock, 14)
    k_hover_rollout(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ RngParams rng,
                    float* __restrict__ st, int rows, float* __restrict__ actions, float* __restrict__ obs, float* __restrict__ reward,
                    uint8_t* __restrict__ term, uint8_t* __restrict__ trunc, uint8_t* __restrict__ info, const float* __restrict__ start_pos,
                    const float* __restrict__ start_orn, const float* __restrict__ spare, uint32_t* __restrict__ episode,
                    int32_t* __restrict__ consumed_count, int2* __restrict__ consumed_list, int32_t* __restrict__ last_count,
                    int32_t* __restrict__ last_list, uint32_t step_seq0, int T, int64_t N) {
  const int tile = (int)blockIdx.x;
  __shared__ __align__(128) float smem2[2][kBlock * kObsMax];  // the observation tile of step t leaves by TMA while step t + 1 fills the other one
  constexpr int kInGroups = qx_groups_moved<MODE>();
  __shared__ __align__(128) float stile[kInGroups * kTileGroupStride];
  __shared__ __align__(8) uint64_t mbar;
  const int O = h.angle_representation == 0 ? 20 : 21;
  const int lane = threadIdx.x;
  const int64_t tile_first = (int64_t)tile * kBlock;
  const int64_t i = tile_first + lane;
  const bool active = i < N;
  float* rec = st + qx_tile_base(i, rows);
  if (lane == 0) {
    mbar_init(&mbar, 1);
    bulk_load_g2s(stile, st + qx_tile_base(tile_first, rows), (uint32_t)(kInGroups * kTileGroupStride * sizeof(float)), &mbar);
  }
  __syncwarp();
  uint32_t e_local = active ? episode[i] : 0u;  // the next spare this env consumes
  float sx = 0.f, sy = 0.f, sz = 0.f, ox = 0.f, oy = 0.f, oz = 0.f;
  if (active) {
    sx = start_pos[3 * i + 0]; sy = start_pos[3 * i + 1]; sz = start_pos[3 * i + 2];
    ox = start_orn[3 * i + 0]; oy = start_orn[3 * i + 1]; oz = start_orn[3 * i + 2];
  }
  QuadXRegs s;
  int step_count;
  mbar_wait(&mbar, 0);
  quadx_load_tile<MODE, kTileGroupStride>(stile + lane * 4, s, step_count);
  __syncwarp();  // the tile buffer is dead from here on: it stages the spare records of resetting lanes (kStageFloats)
  int64_t nrows = N - tile_first;
  if (nrows > kBlock) nrows = kBlock;
  const uint32_t obs_bytes = (uint32_t)nrows * (uint32_t)O * 4u;
  const bool bulk = (obs_bytes & 15u) == 0u;
  float* obs_dst = obs + tile_first * O;
  const uint64_t g = ((uint64_t)rng.env_offset_hi << 32 | rng.env_offset_lo) + (uint64_t)i;
#pragma unroll 1
  for (int t = 0; t < T; ++t) {
    const uint32_t step_seq = step_seq0 + (uint32_t)t;
    // ---- the step's draws: motor noise and the action, same counters as a single-step launch
    auto nz = make_noise<false>(nullptr, N, active ? i : 0, rng, step_seq, TAG_ENV_STEP, p.noise_loc, p.ratio);
    nz.prefetch4();
    float act[4];
    {
      U4 r = philox4x32_10(U4{(uint32_t)g, (uint32_t)(g >> 32), step_seq, (uint32_t)TAG_ACTION << 24}, rng.k0, rng.k1);
      const float pi = 3.14159265358979323846f;
      if (MODE == -1) {
        act[0] = 0.8f * u32_to_unit_open(r.x); act[1] = 0.8f * u32_to_unit_open(r.y);
        act[2] = 0.8f * u32_to_unit_open(r.z); act[3] = 0.8f * u32_to_unit_open(r.w);
      } else {
        act[0] = pi * (2.0f * u32_to_unit_open(r.x) - 1.0f); act[1] = pi * (2.0f * u32_to_unit_open(r.y) - 1.0f);
        act[2] = pi * (2.0f * u32_to_unit_open(r.z) - 1.0f); act[3] = 0.8f * u32_to_unit_open(r.w);
      }
      if (active) reinterpret_cast<float4*>(actions)[i] = make_float4(act[0], act[1], act[2], act[3]);
    }
    const bool resetting = active && (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0;
    // the lanes that reset on this step are known now: their spare record starts its way to L1 and the slot on the top-up list
    // is taken (one atomic per warp) while the other lanes integrate
    const unsigned reset_m = __ballot_sync(0xffffffffu, resetting);
    int reset_base = 0;
    const float* staged = nullptr;  // this lane's spare record in shared memory (the dead state-tile buffer, see kStageFloats)
    if (reset_m != 0u) {
      constexpr int kSlots = kInGroups * kTileGroupStride / SP_ROWS;
      if (resetting) {
        const float* r = spare + ((int64_t)(e_local & kSpareMask) * N + i) * SP_ROWS;
        const int rank = __popc(reset_m & ((1u << lane) - 1u));
        if (rank < kSlots) {
          float* q = stile + rank * SP_ROWS;
#pragma unroll
          for (int g = 0; g < SP_ROWS / 4; ++g) cp_async16(q + 4 * g, r + 4 * g);
          staged = q;
        } else {
          prefetch_l1(r); prefetch_l1(r + 32); prefetch_l1(r + 64); prefetch_l1(r + SP_ROWS - 1);
        }
      }
      // one slot range on the top-up list per warp.  Inline PTX: a plain atomicAdd is rewritten by the compiler into its
      // warp-aggregated form, whose broadcast shuffle waits for the atomic's return HERE instead of after the integration
      if (lane == __ffs(reset_m) - 1)
        asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(reset_base) : "l"(consumed_count), "r"(__popc(reset_m)) : "memory");
    }
    const int n_aviary = (active && !resetting) ? h.env_step_ratio : 0;
    float rew = -0.1f;
#pragma unroll
    for (int k = 0; k < 4; ++k) s.sp[k] = act[k];
#pragma unroll 1
    for (int k = 0; k < n_aviary; ++k) {
      if (s.flags & (FLAG_TERM | FLAG_TRUNC)) break;  // quadx_base_env.py:289-290
      quadx_aviary_step<MODE>(p, s, nz);
      hover_term_trunc_reward(h, s, step_count, rew);
    }
    step_count += 1;
    if (reset_m != 0u) {
      if (resetting) {
        if (staged) cp_async_wait_all();
        const float* srec = staged ? staged : spare + ((int64_t)(e_local & kSpareMask) * N + i) * SP_ROWS;
        const F4 m0 = ld_f4(srec + SP_POSE), m1 = ld_f4(srec + SP_POSE + 4), m2 = ld_f4(srec + SP_POSE + 8);
        const bool hit = m1.z != 0.0f && bits_from_f(m2.x) == e_local && m0.x == sx && m0.y == sy && m0.z == sz && m0.w == ox && m1.x == oy && m1.y == oz;
        if (hit) {
          int dummy;
          quadx_load_tile<MODE, 4>(srec, s, dummy);
          const F4 pw = ld_f4(srec + QX_PWM);
          s.pwm[0] = pw.x; s.pwm[1] = pw.y; s.pwm[2] = pw.z; s.pwm[3] = pw.w;
          s.flags = bits_from_f(m1.w);
        } else {
          s = hover_warmup_cold<MODE>(p, hover_fresh<MODE>(sx, sy, sz, ox, oy, oz), h.warmup_steps, rng, N, i, e_local);
          quadx_requantize(s);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) { s.sp[k] = 0.0f; act[k] = 0.0f; }  // self.action = zeros (quadx_base_env.py:165)
        step_count = 0;
        rew = 0.0f;
      }
      // the consumed spares go on the top-up list: (env, episode that takes the freed place kRolloutAhead ahead)
      const int base = __shfl_sync(0xffffffffu, reset_base, __ffs(reset_m) - 1);
      if (resetting) {
        consumed_list[base + __popc(reset_m & ((1u << lane) - 1u))] = make_int2((int)i, (int)(e_local + (uint32_t)kRolloutAhead));
        e_local += 1u;
      }
    }
    // ---- outputs of the step
    float* smem = smem2[t & 1];
    if (bulk && lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");  // the copy that read THIS buffer two steps ago
    __syncwarp();
    hover_observation(h, s, act, smem + lane * O);
    fence_async_smem();
    __syncwarp();
    if (bulk) {
      if (lane == 0) bulk_store_s2g(obs_dst, smem, obs_bytes);
    } else {
      for (int j = lane; j < (int)nrows * O; j += kBlock) obs_dst[j] = smem[j];
    }
    if (active) {
      reward[i] = rew;
      term[i] = (s.flags & FLAG_TERM) ? 1 : 0;
      trunc[i] = (s.flags & FLAG_TRUNC) ? 1 : 0;
      if (info) info[i] = (uint8_t)(((s.flags & FLAG_OOB) ? 1 : 0) | ((s.flags & FLAG_COLLISION) ? 2 : 0));
    }
    quadx_requantize(s);  // what storing the state and loading it again in the next launch does to the fp64-carried fields
  }
  if (active) {
    quadx_store_tile<MODE, kTileGroupStride>(rec, s, step_count);
    episode[i] = e_local;
  }
  // hand-over to the single-step pipeline: the envs that finished on the LAST step are the done list its next launch expects
  const bool done = active && (s.flags & (FLAG_TERM | FLAG_TRUNC)) != 0;
  const unsigned m = __ballot_sync(0xffffffffu, done);
  if (m != 0u) {
    int base = 0;
    if (lane == __ffs(m) - 1) base = atomicAdd(last_count, __popc(m));
    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
    if (done) last_list[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
  }
  if (bulk && lane == 0) bulk_store_wait_read();  // the CTA's shared memory must outlive the engine's reads
}

// After a user reset of every env: each env gets a complete fresh spare (dense warps, all envs).
template <int MODE>
__global__ void __launch_bounds__(kBlock, kHoverBlocks)
    k_hover_spare_build(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h, const __grid_constant__ RngParams rng,
                        const float* __restrict__ start_pos, const float* __restrict__ start_orn, float* __restrict__ spare,
                        uint32_t* __restrict__ episode, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  const uint32_t e = episode[i] + 1u;
  float* rec = spare + ((int64_t)(e & kSpareMask) * N + i) * SP_ROWS;
  const float px = start_pos[3 * i + 0], py = start_pos[3 * i + 1], pz = start_pos[3 * i + 2];
  const float ox = start_orn[3 * i + 0], oy = start_orn[3 * i + 1], oz = start_orn[3 * i + 2];
  QuadXRegs s = hover_fresh<MODE>(px, py, pz, ox, oy, oz);
  hover_warmup_inline<MODE, false>(p, s, 0, h.warmup_steps, rng, nullptr, N, i, e);
  quadx_store_tile<7, 4>(rec, s, 0);
  st_f4(rec + SP_POSE, px, py, pz, ox);
  st_f4(rec + SP_POSE + 4, oy, oz, 1.0f, f_from_bits(s.flags));
  st_f4(rec + SP_POSE + 8, f_from_bits(e), 0.0f, 0.0f, 0.0f);
  episode[i] = e;
}

// env.reset() for all / masked envs
template <int MODE, bool INJECT>
__global__ void __launch_bounds__(kBlock)
    k_hover_reset(const __grid_constant__ QuadXParams p, const __grid_constant__ HoverParams h,
                  const __grid_constant__ RngParams rng, float* __restrict__ st, int rows,
                  const float* __restrict__ start_pos, const float* __restrict__ start_orn,
                  const uint8_t* __restrict__ mask, const float* __restrict__ noise, float* __restrict__ obs,
                  uint32_t seq, int64_t N) {
  const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  if (i >= N) return;
  if (mask && !mask[i]) return;
  const int O = (h.angle_representation == 0 ? 20 : 21) + (h.ma ? 3 : 0);
  float row[kObsMax];
  QuadXRegs s = hover_fresh<MODE>(start_pos[3 * i + 0], start_pos[3 * i + 1], start_pos[3 * i + 2], start_orn[3 * i + 0], start_orn[3 * i + 1],
                                  start_orn[3 * i + 2]);
  hover_warmup_inline<MODE, INJECT>(p, s, 0, h.warmup_steps, rng, noise, N, i, seq);
  float* rec = st + qx_tile_base(i, rows);
  const float zero[4] = {0.f, 0.f, 0.f, 0.f};  // self.action = zeros (quadx_base_env.py:165)
  if (h.ma) {  // past_actions is NOT cleared by a reset in the reference: it still holds the previous episode's value
    const F4 pa = ld_f4(rec + (QM_PAST / 4) * kTileGroupStride);
    const float past[4] = {pa.x, pa.y, pa.z, pa.w};
    ma_hover_observation(h, s, past, start_pos[3 * i], start_pos[3 * i + 1], start_pos[3 * i + 2], row);
  } else {
    hover_observation(h, s, zero, row);
  }
  quadx_store_tile<7, kTileGroupStride>(rec, s, 0);
  if (obs) {
#pragma unroll
    for (int k = 0; k < kObsMax; ++k)
      if (k < O) obs[i * O + k] = row[k];
  }
}

// A masked pfb_env_reset on an autoreset handle of the tail-CTA env kinds: an env that finished on the previous step sits in
// the done list the NEXT step's tail CTAs consume; reset by hand, it must not be reset again by them while its regular thread
// steps it (two writers for one env).  Drop the masked entries from that list: in-place compaction by ONE CTA, chunk by chunk
// (a chunk is read completely before anything is written, and the write cursor never passes the read cursor).
__global__ void __launch_bounds__(1024) k_drop_masked_done(int32_t* __restrict__ list, int32_t* __restrict__ count, const uint8_t* __restrict__ mask) {
  __shared__ int kept;
  const int n = *count;
  if (threadIdx.x == 0) kept = 0;
  __syncthreads();
  for (int first = 0; first < n; first += blockDim.x) {
    const int t = first + (int)threadIdx.x;
    const int32_t e = t < n ? list[t] : -1;
    const bool keep = t < n && !mask[e];
    __syncthreads();  // the whole chunk is in registers
    if (keep) list[atomicAdd(&kept, 1)] = e;  // order inside the list does not matter: every entry is an independent env / arena
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = kept;
}
int pfb_drop_masked_done(PfbContext* h, const uint8_t* mask, cudaStream_t s) {
  if (!mask || !h->env.autoreset || !h->d_done_list) return 0;
  const uint64_t k = h->step_seq;  // the next step: its tail CTAs read list [(k - 1) % 4]
  k_drop_masked_done<<<1, 1024, 0, s>>>(h->d_done_list + ((k + 3) % 4) * h->n, h->d_counters + ((k + 3) % 4), mask);
  LAUNCH_CHECK(h);
  return 0;
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
extern "C" {

const char* pfb_last_error(void) { return g_err; }
int pfb_abi_version(void) { return PFB_ABI_VERSION; }
int pfb_sizeof_model(void) { return (int)sizeof(PfbModel); }
int pfb_sizeof_env_config(void) { return (int)sizeof(PfbEnvConfig); }
int pfb_sizeof_buffers(void) { return (int)sizeof(PfbBuffers); }

int pfb_create(const PfbModel* model, const PfbEnvConfig* env, int64_t n_envs, int device, uint64_t seed, PfbHandle* out) {
  if (!model || !out) return fail("pfb_create: null argument");
  if (model->abi_version != PFB_ABI_VERSION) return fail("PfbModel ABI %d != library ABI %d", model->abi_version, PFB_ABI_VERSION);
  if (n_envs <= 0) return fail("n_envs must be positive");
  if (model->kind != PFB_KIND_QUADX && model->kind != PFB_KIND_FIXEDWING && model->kind != PFB_KIND_ROCKET)
    return fail("unknown vehicle kind %d", model->kind);
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail("no CUDA device: libpyflyt_b200 has no CPU fallback (%s)", e != cudaSuccess ? cudaGetErrorString(e) : "0 devices");
  if (device < 0 || device >= count) return fail("device %d out of range (have %d)", device, count);
  CUDA_OK(cudaSetDevice(device));
  PfbContext* c = new (std::nothrow) PfbContext();
  if (!c) return fail("out of host memory");
  memset(c, 0, sizeof(*c));
  c->model = *model;
  if (env) c->env = *env;
  c->n = n_envs;
  c->device = device;
  if (model->kind == PFB_KIND_QUADX) {
    if (build_quadx_params(*model, c->qx) != 0) { delete c; return -1; }
  } else if (model->kind == PFB_KIND_FIXEDWING) {
    if (fw_build_params(*model, env, c->fw, c->wp) != 0) { delete c; return -1; }
    if (df_build_params(env, c->df) != 0) { delete c; return -1; }
    if (env && env->env_kind == PFB_ENV_DOGFIGHT && (n_envs % (2 * env->team_size)) != 0) {
      delete c;
      return fail("n_envs (%lld) must be a multiple of the arena size 2*team_size = %d", (long long)n_envs, 2 * env->team_size);
    }
  } else {
    if (rk_build_params(*model, env, c->rk, c->land) != 0) { delete c; return -1; }
  }
  c->hover.env_step_ratio = env ? env->env_step_ratio : 1;
  c->hover.max_steps = env ? env->max_steps : 0;
  c->hover.angle_representation = env ? env->angle_representation : 1;
  c->hover.sparse_reward = env ? env->sparse_reward : 0;
  c->hover.warmup_steps = env ? env->warmup_steps : 0;
  c->hover.flight_mode = env ? env->flight_mode : 0;
  {
    double dome = env ? env->flight_dome_size : INFINITY;
    c->hover.dome2 = (float)(dome * dome);
  }
  c->hover.ma = (env && env->env_kind == PFB_ENV_MA_QUADX_HOVER) ? 1 : 0;
  c->hover.stagger_ns = 0;
  c->hover.stagger_mod = 1;
  if (const char* e = getenv("PFB_HOVER_STAGGER")) {
    int ns = 0, mod = 2;
    if (sscanf(e, "%d,%d", &ns, &mod) >= 1 && ns >= 0 && ns <= 20000 && mod >= 1 && mod <= 8) { c->hover.stagger_ns = ns; c->hover.stagger_mod = mod; }
  }
  if (c->hover.ma && env->autoreset) {
    delete c;
    return fail("MAQuadXHover is a per-agent epilogue: arenas are reset by the caller (pfb_env_reset with a mask), autoreset must be 0");
  }
  if (env && env->env_kind != PFB_ENV_NONE) {
    const bool ok = (model->kind == PFB_KIND_QUADX && env->env_kind == PFB_ENV_QUADX_HOVER) ||
                    (model->kind == PFB_KIND_QUADX && env->env_kind == PFB_ENV_QUADX_WAYPOINTS) ||
                    (model->kind == PFB_KIND_QUADX && env->env_kind == PFB_ENV_MA_QUADX_HOVER) ||
                    (model->kind == PFB_KIND_FIXEDWING && env->env_kind == PFB_ENV_FIXEDWING_WAYPOINTS) ||
                    (model->kind == PFB_KIND_FIXEDWING && env->env_kind == PFB_ENV_DOGFIGHT) ||
                    (model->kind == PFB_KIND_ROCKET && env->env_kind == PFB_ENV_ROCKET_LANDING);
    if (!ok) {
      delete c;
      return fail("env kind %d is not available for vehicle kind %d in this library", env->env_kind, model->kind);
    }
  }
  if (env && env->env_kind == PFB_ENV_QUADX_WAYPOINTS) {
    if (env->num_targets < 1 || env->num_targets > kMaxTargets) {
      delete c;
      return fail("num_targets must be in 1..%d, got %d", kMaxTargets, env->num_targets);
    }
    c->qwp.env_step_ratio = env->env_step_ratio;
    c->qwp.max_steps = env->max_steps;
    c->qwp.sparse_reward = env->sparse_reward;
    c->qwp.warmup_steps = env->warmup_steps;
    c->qwp.num_targets = env->num_targets;
    c->qwp.use_yaw_targets = env->use_yaw_targets ? 1 : 0;
    c->qwp.dome = (float)env->flight_dome_size;
    c->qwp.dome2 = (float)(env->flight_dome_size * env->flight_dome_size);
    c->qwp.goal_reach_distance = (float)env->goal_reach_distance;
    c->qwp.goal_reach_angle = (float)env->goal_reach_angle;
    c->qwp.min_height = 0.1f;  // quadx_waypoints_env.py:88
  }
  c->rng.k0 = (uint32_t)seed;
  c->rng.k1 = (uint32_t)(seed >> 32);
  c->mode = 0;
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  c->sm_count = prop.multiProcessorCount;
  // pfb_env_step_mapped: the kernel reads / writes host memory over PCIe, which is the bottleneck by 10x; with every CTA resident
  // in one wave the bus idles while all warps compute and then takes the whole output at once.  Requesting dynamic shared
  // memory the kernel never touches caps the CTAs resident per SM, so the step runs as several waves and the output of a wave
  // crosses the bus while the next one computes.  PFB_MAPPED_DYN_SMEM overrides (bytes, <= 48 KB; 0 = one wave).
  c->mapped_dyn_smem = 12 * 1024;  // measured on B200 (tools/exp_mapped_waves.py): 149.5 us / step in one wave, 144.8 us with 12-28 KB
  if (const char* e = getenv("PFB_MAPPED_DYN_SMEM")) {
    const int v = atoi(e);
    if (v >= 0 && v <= 40 * 1024) c->mapped_dyn_smem = v;
  }
  CUDA_OK(cudaMalloc(&c->d_counters, 8 * sizeof(int32_t)));  // [0..3] rotating autoreset counters, [4] ticket of the split dogfight
  CUDA_OK(cudaMemset(c->d_counters, 0, 8 * sizeof(int32_t)));
  CUDA_OK(cudaMalloc(&c->d_done_list, 4 * (size_t)n_envs * sizeof(int32_t)));
  if (env && env->autoreset && (env->env_kind == PFB_ENV_QUADX_HOVER || env->env_kind == PFB_ENV_FIXEDWING_WAYPOINTS ||
                                 env->env_kind == PFB_ENV_QUADX_WAYPOINTS || env->env_kind == PFB_ENV_ROCKET_LANDING ||
                                 env->env_kind == PFB_ENV_DOGFIGHT)) {
    // spare post-reset states: env-major records (QuadX-Hover: two per env, double-buffered by episode parity, rebuilt by
    // builder CTAs inside the step launches; the other env kinds: one per env, rebuilt on a library-owned side stream)
    const bool hover = env->env_kind == PFB_ENV_QUADX_HOVER;
    const size_t rec = env->env_kind == PFB_ENV_QUADX_WAYPOINTS ? (size_t)qwp_spare_rows()
                       : (env->env_kind == PFB_ENV_DOGFIGHT ? (size_t)df_spare_rows() : (size_t)SP_ROWS * (hover ? kSpareBufs : 1));
    CUDA_OK(cudaMalloc(&c->d_spare, rec * (size_t)n_envs * sizeof(float)));
    CUDA_OK(cudaMemset(c->d_spare, 0, rec * (size_t)n_envs * sizeof(float)));
    if (hover) {
      CUDA_OK(cudaMalloc(&c->d_consumed, (size_t)(kRolloutMaxSteps / 2 + 1) * (size_t)n_envs * sizeof(int2)));  // (env, episode) per reset of a fused launch
      CUDA_OK(cudaMalloc(&c->d_elist, 4 * (size_t)n_envs * sizeof(uint32_t)));
      CUDA_OK(cudaMemset(c->d_elist, 0, 4 * (size_t)n_envs * sizeof(uint32_t)));
      CUDA_OK(cudaMalloc(&c->d_episode, (size_t)n_envs * sizeof(uint32_t)));
      CUDA_OK(cudaMemset(c->d_episode, 0, (size_t)n_envs * sizeof(uint32_t)));
    } else {
      int prio_lo = 0, prio_hi = 0;  // the rebuild is small and latency-critical: let its CTAs go first when slots free up
      CUDA_OK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
      CUDA_OK(cudaStreamCreateWithPriority(&c->side, cudaStreamNonBlocking, prio_hi));
      CUDA_OK(cudaEventCreateWithFlags(&c->ev_step, cudaEventDisableTiming));
      for (int k = 0; k < 4; ++k) CUDA_OK(cudaEventCreateWithFlags(&c->ev_spare[k], cudaEventDisableTiming));
    }
  }
  *out = c;
  return 0;
}

int pfb_destroy(PfbHandle h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  if (h->d_spare) {
    if (h->side) {
      cudaStreamSynchronize(h->side);
      cudaStreamDestroy(h->side);
      cudaEventDestroy(h->ev_step);
      for (int k = 0; k < 4; ++k) cudaEventDestroy(h->ev_spare[k]);
    }
    cudaFree(h->d_spare);
    if (h->d_episode) cudaFree(h->d_episode);
    if (h->d_elist) cudaFree(h->d_elist);
    if (h->d_consumed) cudaFree(h->d_consumed);
  }
  cudaFree(h->d_counters);
  cudaFree(h->d_done_list);
  if (h->prof_ev) {
    for (int i = 0; i < 2 * h->prof_cap; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev;
  }
  delete h;
  return 0;
}

int pfb_set_env_offset(PfbHandle h, uint64_t first_global_env) {
  if (!h) return fail("null handle");
  h->rng.env_offset_lo = (uint32_t)first_global_env;
  h->rng.env_offset_hi = (uint32_t)(first_global_env >> 32);
  return 0;
}

static inline bool is_fw(PfbHandle h) { return h->model.kind == PFB_KIND_FIXEDWING; }
static inline bool is_rk(PfbHandle h) { return h->model.kind == PFB_KIND_ROCKET; }
static inline bool is_qwp(PfbHandle h) { return h->model.kind == PFB_KIND_QUADX && h->env.env_kind == PFB_ENV_QUADX_WAYPOINTS; }
static inline bool is_ma(PfbHandle h) { return h->model.kind == PFB_KIND_QUADX && h->env.env_kind == PFB_ENV_MA_QUADX_HOVER; }
static inline bool is_df(PfbHandle h) { return h->model.kind == PFB_KIND_FIXEDWING && h->env.env_kind == PFB_ENV_DOGFIGHT; }
static inline bool is_tiled(PfbHandle h) { return h->model.kind == PFB_KIND_QUADX && h->env.env_kind != PFB_ENV_QUADX_WAYPOINTS; }
static inline int qx_rows(PfbHandle h) { return h->env.env_kind == PFB_ENV_MA_QUADX_HOVER ? QM_ROWS : QX_ROWS; }
int pfb_state_rows(PfbHandle h) { return is_rk(h) ? rk_state_rows() : (is_fw(h) ? fw_state_rows() : (is_qwp(h) ? qwp_state_rows() : qx_rows(h))); }
int pfb_state_layout(PfbHandle h) { return h && is_tiled(h) ? PFB_LAYOUT_WARP_TILED : PFB_LAYOUT_FIELD_MAJOR; }
int64_t pfb_state_floats(PfbHandle h) {
  if (!h) return 0;
  if (is_tiled(h)) return ((h->n + kTileLanes - 1) / kTileLanes) * qx_tile_floats(qx_rows(h));  // padded to whole tiles
  return (int64_t)pfb_state_rows(h) * h->n;
}
int pfb_istate_rows(PfbHandle h) { return is_rk(h) ? rk_istate_rows() : (is_fw(h) ? fw_istate_rows() : (is_qwp(h) ? qwp_istate_rows() : QI_ROWS)); }
int pfb_setpoint_dim(PfbHandle h) { return is_rk(h) ? 7 : ((is_fw(h) && h->env.env_kind == PFB_ENV_NONE) ? 6 : 4); }
int pfb_obs_dim(PfbHandle h) { return is_df(h) ? df_obs_dim(h) : is_rk(h) ? rk_obs_dim(h) : (is_fw(h) ? fw_obs_dim(h) : (is_qwp(h) ? qwp_obs_dim(h) : (h->hover.angle_representation == 0 ? 20 : 21) + (is_ma(h) ? 3 : 0))); }
int pfb_aux_dim(PfbHandle h) { return is_rk(h) ? 9 : (is_fw(h) ? 6 : 4); }

int pfb_bind(PfbHandle h, const PfbBuffers* b) {
  if (!h || !b) return fail("pfb_bind: null argument");
  if (!b->state || !b->istate || !b->setpoint || !b->start_pos || !b->start_orn)
    return fail("pfb_bind: state, istate, setpoint, start_pos and start_orn are mandatory");
  if (((uintptr_t)b->setpoint & 15) || ((uintptr_t)b->state & 15)) return fail("pfb_bind: buffers must be 16-byte aligned");
  h->buf = *b;
  h->bound = true;
  return 0;
}

#define REQUIRE_BOUND(h)                                   \
  if (!(h)) return fail("null handle");                    \
  if (!(h)->bound) return fail("buffers not bound: call pfb_bind first"); \
  CUDA_OK(cudaSetDevice((h)->device));


int pfb_reset(PfbHandle h, const uint8_t* mask, void* stream) {
  if (h) h->fused_ready = 0;
  REQUIRE_BOUND(h);
  cudaStream_t s = (cudaStream_t)stream;
  if (is_fw(h)) return fw_reset(h, mask, s);
  if (is_rk(h)) return rk_reset(h, mask, s);
  if (is_tiled(h)) k_quadx_reset<true><<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.setpoint, h->buf.start_pos, h->buf.start_orn, mask, h->n);
  else k_quadx_reset<false><<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.setpoint, h->buf.start_pos, h->buf.start_orn, mask, h->n);
  LAUNCH_CHECK(h);
  if (!mask) h->mode = 0;  // QuadX.reset() calls set_mode(0) (quadx.py:224)
  return 0;
}

int pfb_set_mode(PfbHandle h, int mode, void* stream) {
  REQUIRE_BOUND(h);
  cudaStream_t s = (cudaStream_t)stream;
  if (is_fw(h)) return fw_set_mode(h, mode, s);
  if (is_rk(h)) return rk_set_mode(h, mode, s);
  if (is_tiled(h)) { PFB_MODE_SWITCH(mode, (k_quadx_set_mode<MODE, true><<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.setpoint, h->n))); }
  else { PFB_MODE_SWITCH(mode, (k_quadx_set_mode<MODE, false><<<grid_for(h->n), kBlock, 0, s>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.setpoint, h->n))); }
  LAUNCH_CHECK(h);
  h->mode = mode;
  return 0;
}

int pfb_aviary_step(PfbHandle h, int n_steps, const float* noise, void* stream) {
  REQUIRE_BOUND(h);
  if (n_steps <= 0) return fail("n_steps must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  if (is_fw(h)) return fw_aviary_step(h, n_steps, noise, s);
  if (is_rk(h)) return rk_aviary_step(h, n_steps, noise, s);
  const int mode = h->mode;
  const uint32_t seq = (uint32_t)h->aviary_seq++;
#define AV_ARGS h->qx, h->rng, h->buf.state, h->buf.istate, qx_rows(h), h->buf.setpoint, noise, n_steps, seq, h->n
  const int g = grid_for(h->n);
  if (is_tiled(h)) {
    if (noise) { PFB_MODE_SWITCH(mode, (k_quadx_aviary_step<MODE, true, true><<<g, kBlock, 0, s>>>(AV_ARGS))); }
    else { PFB_MODE_SWITCH(mode, (k_quadx_aviary_step<MODE, false, true><<<g, kBlock, 0, s>>>(AV_ARGS))); }
  } else {
    if (noise) { PFB_MODE_SWITCH(mode, (k_quadx_aviary_step<MODE, true, false><<<g, kBlock, 0, s>>>(AV_ARGS))); }
    else { PFB_MODE_SWITCH(mode, (k_quadx_aviary_step<MODE, false, false><<<g, kBlock, 0, s>>>(AV_ARGS))); }
  }
#undef AV_ARGS
  LAUNCH_CHECK(h);
  return 0;
}

int pfb_set_base_velocity(PfbHandle h, const float* lin_vel, const float* ang_vel, void* stream) {
  REQUIRE_BOUND(h);
  if (!lin_vel || !ang_vel) return fail("pfb_set_base_velocity: null argument");
  if (is_rk(h)) return rk_set_velocity(h, lin_vel, ang_vel, (cudaStream_t)stream);
  return fail("pfb_set_base_velocity is only built for the rocket (the one vehicle whose env calls resetBaseVelocity)");
}

int pfb_observe_state(PfbHandle h, void* stream) {
  REQUIRE_BOUND(h);
  if (is_fw(h)) return fw_observe(h, (cudaStream_t)stream);
  if (is_rk(h)) return rk_observe(h, (cudaStream_t)stream);
  if (is_tiled(h)) k_quadx_observe<true><<<grid_for(h->n), kBlock, 0, (cudaStream_t)stream>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.drone_state, h->buf.aux_state, h->buf.contact, h->n);
  else k_quadx_observe<false><<<grid_for(h->n), kBlock, 0, (cudaStream_t)stream>>>(h->buf.state, h->buf.istate, qx_rows(h), h->buf.drone_state, h->buf.aux_state, h->buf.contact, h->n);
  LAUNCH_CHECK(h);
  return 0;
}

static int require_env(PfbHandle h) {
  if (h->env.env_kind == PFB_ENV_NONE) return fail("handle was created without an env epilogue");
  if (!h->buf.obs || !h->buf.reward || !h->buf.term || !h->buf.trunc) return fail("obs/reward/term/trunc buffers are not bound");
  return 0;
}

int pfb_env_reset(PfbHandle h, const uint8_t* mask, const float* noise, void* stream) {
  REQUIRE_BOUND(h);
  if (require_env(h)) return -1;
  h->fused_ready = 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (is_df(h)) return df_env_reset(h, mask, noise, s);
  if (is_fw(h)) return fw_env_reset(h, mask, noise, s);
  if (is_rk(h)) return rk_env_reset(h, mask, noise, s);
  if (is_qwp(h)) return qwp_env_reset(h, mask, noise, s);
  const int mode = h->hover.flight_mode;
  // resets draw from their own Philox stream; the high bit keeps them apart from in-step autoresets
  const uint32_t seq = 0x80000000u | (uint32_t)h->reset_seq++;
  if (h->d_spare && !mask) CUDA_OK(cudaMemsetAsync(h->d_counters, 0, 4 * sizeof(int32_t), s));  // a full reset empties the rebuild queues
#define HR_ARGS h->qx, h->hover, h->rng, h->buf.state, qx_rows(h), h->buf.start_pos, h->buf.start_orn, mask, noise, h->buf.obs, seq, h->n
  if (noise) { PFB_MODE_SWITCH(mode, (k_hover_reset<MODE, true><<<grid_for(h->n), kBlock, 0, s>>>(HR_ARGS))); }
  else { PFB_MODE_SWITCH(mode, (k_hover_reset<MODE, false><<<grid_for(h->n), kBlock, 0, s>>>(HR_ARGS))); }
#undef HR_ARGS
  LAUNCH_CHECK(h);
  if (h->d_spare && !mask) {  // every env gets a fresh spare.  A masked reset keeps the spares: they are keyed by (env, episode
                              // number) and stay valid; a masked env simply is not `done` on the next step
    PFB_MODE_SWITCH(mode, (k_hover_spare_build<MODE><<<grid_for(h->n), kBlock, 0, s>>>(h->qx, h->hover, h->rng, h->buf.start_pos, h->buf.start_orn,
                                                                                      h->d_spare, h->d_episode, h->n)));
    LAUNCH_CHECK(h);
  }
  h->mode = mode;
  return 0;
}

static int env_step_impl(PfbHandle h, float* actions, const float* noise, bool randact, cudaStream_t s) {
  if (is_df(h)) return df_env_step(h, actions, noise, randact, s);
  if (is_fw(h)) return fw_env_step(h, actions, noise, randact, s);
  if (is_rk(h)) return rk_env_step(h, actions, noise, randact, s);
  if (is_qwp(h)) return qwp_env_step(h, actions, noise, randact, s);
  const int mode = h->hover.flight_mode;
  const bool autoreset = h->env.autoreset != 0;
  const uint64_t k = h->step_seq;
  // four rotating done lists / counters: step k appends the envs that finish to [k % 4]; its builder CTAs start the next
  // spares of [(k - 1) % 4] (the envs this launch resets) and finish those of [(k - 2) % 4]; it zeroes counter [(k + 1) % 4]
  int32_t* cnt_cur = h->d_counters + (k % 4);
  int32_t* cnt_b0 = h->d_counters + ((k + 3) % 4);
  int32_t* cnt_b1 = h->d_counters + ((k + 2) % 4);
  int32_t* cnt_next = h->d_counters + ((k + 1) % 4);
  int32_t* list_cur = h->d_done_list + (k % 4) * h->n;
  int32_t* list_b0 = h->d_done_list + ((k + 3) % 4) * h->n;
  int32_t* list_b1 = h->d_done_list + ((k + 2) % 4) * h->n;
  uint32_t* elist_b0 = h->d_elist ? h->d_elist + ((k + 3) % 4) * h->n : nullptr;  // episode numbers next to the list entries: written by
  uint32_t* elist_b1 = h->d_elist ? h->d_elist + ((k + 2) % 4) * h->n : nullptr;  // builder phase 0, read by phase 1 of the next launch
  const uint32_t seq = (uint32_t)k;
  const bool spares = autoreset && h->d_spare != nullptr;
  const int spare_copy = (spares && h->env.inline_reset != 1) ? 1 : 0;
  const int tiles = grid_for(h->n);
  const int builders = spares ? (h->sm_count < tiles ? h->sm_count : tiles) : 0;
  const int grid = tiles + 2 * builders;
  const bool prof = h->prof_ev && h->prof_n < h->prof_cap;
  const size_t dyn_smem = (size_t)h->step_dyn_smem;
  if (prof) CUDA_OK(cudaEventRecord(h->prof_ev[2 * h->prof_n], s));
#define STEP_ARGS h->qx, h->hover, h->rng, h->buf.state, qx_rows(h), actions, noise, h->buf.obs, h->buf.reward, h->buf.term, h->buf.trunc,    \
                  h->buf.info, h->buf.start_pos, h->buf.start_orn, cnt_cur, list_cur, cnt_next, cnt_b0, list_b0, cnt_b1, list_b1, elist_b0,   \
                  elist_b1, h->d_spare, h->d_episode, spare_copy, builders, h->noise_dump, seq, h->n
  if (autoreset) {
    if (noise) return fail("injected noise (parity mode) is only supported with autoreset = 0");
    if (randact) {
      PFB_MODE_SWITCH(mode, (k_hover_step<MODE, false, true, true, false><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS)));
    } else {
      PFB_MODE_SWITCH(mode, (k_hover_step<MODE, false, false, true, false><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS)));
    }
  } else if (h->hover.ma) {
    if (randact) return fail("MAQuadXHover has no on-device action generator");
    if (noise) { PFB_MODE_SWITCH(mode, (k_hover_step<MODE, true, false, false, true><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS))); }
    else { PFB_MODE_SWITCH(mode, (k_hover_step<MODE, false, false, false, true><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS))); }
  } else {
    if (noise) {
      PFB_MODE_SWITCH(mode, (k_hover_step<MODE, true, false, false, false><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS)));
    } else if (randact) {
      PFB_MODE_SWITCH(mode, (k_hover_step<MODE, false, true, false, false><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS)));
    } else {
      PFB_MODE_SWITCH(mode, (k_hover_step<MODE, false, false, false, false><<<grid, kBlock, dyn_smem, s>>>(STEP_ARGS)));
    }
  }
#undef STEP_ARGS
  LAUNCH_CHECK(h);
  if (prof) {
    CUDA_OK(cudaEventRecord(h->prof_ev[2 * h->prof_n + 1], s));
    h->prof_n += 1;
  }
  h->step_seq += 1;
  h->fused_ready = 0;  // the step pipeline owns the spares again
  return 0;
}

int pfb_sizeof_wind(void) { return (int)sizeof(PfbWind); }

int pfb_set_wind(PfbHandle h, const PfbWind* wind) {
  if (!h) return fail("null handle");
  WindParams w;
  memset(&w, 0, sizeof(w));
  if (wind && wind->kind != PFB_WIND_NONE) {
    if (wind->kind < PFB_WIND_CONSTANT || wind->kind > PFB_WIND_EXP) return fail("unknown wind kind %d", wind->kind);
    if (!(wind->z_ref > 0.0)) return fail("wind z_ref must be positive");
    if (wind->kind == PFB_WIND_LOG && !(wind->z0 > 0.0 && wind->z0 < wind->z_ref)) return fail("log wind profile needs 0 < z0 < z_ref");
    w.kind = wind->kind;
    w.bx = (float)wind->base[0]; w.by = (float)wind->base[1]; w.bz = (float)wind->base[2];
    w.inv_zref = (float)(1.0 / wind->z_ref);
    w.alpha = (float)wind->alpha;
    if (wind->kind == PFB_WIND_LOG) {
      w.z0 = (float)wind->z0;
      w.inv_z0 = (float)(1.0 / wind->z0);
      w.inv_log = (float)(1.0 / log(wind->z_ref / wind->z0));
    }
  }
  h->qx.wind = w;
  h->fw.wind = w;
  h->rk.wind = w;
  return 0;
}

int pfb_reseed(PfbHandle h, uint64_t seed, void* stream) {
  if (!h) return fail("null handle");
  CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)stream;
  if (h->side) CUDA_OK(cudaStreamSynchronize(h->side));  // no spare rebuild of the old streams may still be in flight
  h->rng.k0 = (uint32_t)seed;
  h->rng.k1 = (uint32_t)(seed >> 32);
  h->fused_ready = 0;
  h->step_seq = 0;
  h->aviary_seq = 0;
  h->reset_seq = 0;
  CUDA_OK(cudaMemsetAsync(h->d_counters, 0, 8 * sizeof(int32_t), s));
  if (h->d_episode) CUDA_OK(cudaMemsetAsync(h->d_episode, 0, (size_t)h->n * sizeof(uint32_t), s));
  return 0;
}

int pfb_set_noise_dump(PfbHandle h, float* dump) {
  if (!h) return fail("null handle");
  h->noise_dump = dump;
  return 0;
}

int pfb_env_step(PfbHandle h, const float* actions, const float* noise, void* stream) {
  REQUIRE_BOUND(h);
  if (require_env(h)) return -1;
  if (actions && ((uintptr_t)actions & 15)) return fail("pfb_env_step: actions must be 16-byte aligned");
  return env_step_impl(h, actions ? const_cast<float*>(actions) : h->buf.setpoint, noise, false, (cudaStream_t)stream);
}

// QuadX-Hover with autoreset: n_steps >= kFusedMinSteps run as fused launches of up to kRolloutMaxSteps env steps (k_hover_rollout)
static bool hover_fused_ok(PfbHandle h) {
  return h->model.kind == PFB_KIND_QUADX && h->env.env_kind == PFB_ENV_QUADX_HOVER && h->env.autoreset != 0 && h->env.inline_reset == 0 &&
         h->d_spare != nullptr && h->d_consumed != nullptr && h->noise_dump == nullptr && !(h->prof_ev && h->prof_n < h->prof_cap);
}
constexpr int kFusedMinSteps = 4;
static int hover_rollout_fused(PfbHandle h, int n_steps, cudaStream_t s) {
  const int mode = h->hover.flight_mode;
  const int tiles = grid_for(h->n);
  if (!h->fused_ready) {
    // finish what the single-step pipeline left half done, then bring every env's spares kRolloutAhead ahead
    const uint64_t k = h->step_seq;
    const int builders = h->sm_count < tiles ? h->sm_count : tiles;
    if (k >= 2) {
      PFB_MODE_SWITCH(mode, (k_hover_drain<MODE><<<builders, kBlock, 0, s>>>(h->qx, h->hover, h->rng, h->d_counters + ((k + 2) % 4),
                                                                            h->d_done_list + ((k + 2) % 4) * h->n, h->d_elist + ((k + 2) % 4) * h->n,
                                                                            h->buf.start_pos, h->buf.start_orn, h->d_spare, h->d_episode, builders, h->n)));
      LAUNCH_CHECK(h);
    }
    PFB_MODE_SWITCH(mode, (k_hover_spare_ahead<MODE><<<tiles, kBlock, 0, s>>>(h->qx, h->hover, h->rng, h->buf.start_pos, h->buf.start_orn, h->d_spare,
                                                                              h->d_episode, h->n)));
    LAUNCH_CHECK(h);
    h->fused_ready = 1;
  }
  int topup_grid = 8 * h->sm_count;
  if (topup_grid > tiles) topup_grid = tiles;
  while (n_steps > 0) {
    const int T = n_steps < kRolloutMaxSteps ? n_steps : kRolloutMaxSteps;
    const uint64_t k0 = h->step_seq, k_last = k0 + (uint64_t)T - 1;
    CUDA_OK(cudaMemsetAsync(h->d_counters, 0, 8 * sizeof(int32_t), s));  // [0..3] step pipeline lists, [5] spares consumed by this launch
    PFB_MODE_SWITCH(mode, (k_hover_rollout<MODE><<<tiles, kBlock, 0, s>>>(
                              h->qx, h->hover, h->rng, h->buf.state, qx_rows(h), h->buf.setpoint, h->buf.obs, h->buf.reward, h->buf.term, h->buf.trunc,
                              h->buf.info, h->buf.start_pos, h->buf.start_orn, h->d_spare, h->d_episode, h->d_counters + 5, h->d_consumed,
                              h->d_counters + (k_last % 4), h->d_done_list + (k_last % 4) * h->n, (uint32_t)k0, T, h->n)));
    LAUNCH_CHECK(h);
    PFB_MODE_SWITCH(mode, (k_hover_spare_topup<MODE><<<topup_grid, kBlock, 0, s>>>(h->qx, h->hover, h->rng, h->buf.start_pos, h->buf.start_orn, h->d_spare,
                                                                                   h->d_counters + 5, h->d_consumed, h->n)));
    LAUNCH_CHECK(h);
    h->step_seq += (uint64_t)T;
    n_steps -= T;
  }
  return 0;
}

int pfb_env_rollout(PfbHandle h, int n_steps, void* stream) {
  REQUIRE_BOUND(h);
  if (require_env(h)) return -1;
  static const int fused_min = getenv("PFB_FUSED_MIN") ? atoi(getenv("PFB_FUSED_MIN")) : kFusedMinSteps;  // tests / experiments
  if (n_steps >= fused_min && hover_fused_ok(h)) return hover_rollout_fused(h, n_steps, (cudaStream_t)stream);
  for (int k = 0; k < n_steps; ++k)
    if (env_step_impl(h, h->buf.setpoint, nullptr, true, (cudaStream_t)stream)) return -1;
  return 0;
}

int pfb_env_step_host(PfbHandle h, const float* host_actions, float* host_obs, float* host_reward, uint8_t* host_term,
                      uint8_t* host_trunc, void* stream) {
  REQUIRE_BOUND(h);
  if (require_env(h)) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int O = pfb_obs_dim(h);
  CUDA_OK(cudaMemcpyAsync(h->buf.setpoint, host_actions, (size_t)h->n * pfb_setpoint_dim(h) * sizeof(float), cudaMemcpyHostToDevice, s));
  if (env_step_impl(h, h->buf.setpoint, nullptr, false, s)) return -1;
  // obs | reward | term | trunc laid out back to back on both sides (what the Python mirror allocates): one copy, one
  // PCIe transaction stream instead of four latency-bound ones
  const size_t ob = (size_t)h->n * O * sizeof(float), rb = (size_t)h->n * sizeof(float), fb = (size_t)h->n;
  const char* d0 = (const char*)h->buf.obs;
  char* h0 = (char*)host_obs;
  const bool packed = (const char*)h->buf.reward == d0 + ob && (const char*)h->buf.term == d0 + ob + rb && (const char*)h->buf.trunc == d0 + ob + rb + fb &&
                      (char*)host_reward == h0 + ob && (char*)host_term == h0 + ob + rb && (char*)host_trunc == h0 + ob + rb + fb;
  if (packed) {
    CUDA_OK(cudaMemcpyAsync(host_obs, h->buf.obs, ob + rb + 2 * fb, cudaMemcpyDeviceToHost, s));
    return 0;
  }
  CUDA_OK(cudaMemcpyAsync(host_obs, h->buf.obs, ob, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaMemcpyAsync(host_reward, h->buf.reward, rb, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaMemcpyAsync(host_term, h->buf.term, fb, cudaMemcpyDeviceToHost, s));
  CUDA_OK(cudaMemcpyAsync(host_trunc, h->buf.trunc, fb, cudaMemcpyDeviceToHost, s));
  return 0;
}

// Zero-copy variant of pfb_env_step_host: the step kernel reads the actions from, and writes obs / reward / term / trunc
// straight into, PINNED (device-mapped) host memory.  The PCIe transfers then overlap the launch tile by tile instead of
// bracketing it as two copies; no staging through the bound device buffers.
int pfb_env_step_mapped(PfbHandle h, const float* host_actions, float* host_obs, float* host_reward, uint8_t* host_term,
                        uint8_t* host_trunc, void* stream) {
  REQUIRE_BOUND(h);
  if (require_env(h)) return -1;
  if (!host_actions || !host_obs || !host_reward || !host_term || !host_trunc) return fail("pfb_env_step_mapped: null argument");
  void *da = nullptr, *dob = nullptr, *dr = nullptr, *dte = nullptr, *dtr = nullptr;
  if (cudaHostGetDevicePointer(&da, (void*)host_actions, 0) != cudaSuccess || cudaHostGetDevicePointer(&dob, host_obs, 0) != cudaSuccess ||
      cudaHostGetDevicePointer(&dr, host_reward, 0) != cudaSuccess || cudaHostGetDevicePointer(&dte, host_term, 0) != cudaSuccess ||
      cudaHostGetDevicePointer(&dtr, host_trunc, 0) != cudaSuccess) {
    cudaGetLastError();
    return fail("pfb_env_step_mapped: the host buffers must be pinned (cudaHostAlloc / cudaHostRegister) memory");
  }
  if (((uintptr_t)da & 15) || ((uintptr_t)dob & 15)) return fail("pfb_env_step_mapped: actions and obs must be 16-byte aligned");
  const PfbBuffers saved = h->buf;
  h->buf.obs = (float*)dob; h->buf.reward = (float*)dr; h->buf.term = (uint8_t*)dte; h->buf.trunc = (uint8_t*)dtr;
  h->step_dyn_smem = h->mapped_dyn_smem;
  const int rc = env_step_impl(h, (float*)da, nullptr, false, (cudaStream_t)stream);
  h->step_dyn_smem = 0;
  h->buf = saved;
  return rc;
}

// ---- MAFixedwingDogfight, split variant: an arena's agents on different ranks (DESIGN.md §7)
int pfb_dogfight_payload_dim(void) { return 20; }

int pfb_dogfight_physics(PfbHandle h, const float* actions, const float* noise, float* payload_out, int first, int do_reset, int aviary_index,
                         void* stream) {
  REQUIRE_BOUND(h);
  if (!is_df(h)) return fail("handle is not a dogfight env");
  if (!payload_out) return fail("pfb_dogfight_physics: null payload buffer");
  return df_split_physics(h, actions ? actions : h->buf.setpoint, noise, payload_out, nullptr, 0, 0, nullptr, 0, 0, first, do_reset, aviary_index,
                          (cudaStream_t)stream);
}

int pfb_dogfight_physics_peer(PfbHandle h, const float* actions, const float* noise, const uint64_t* peer_tables_dev, int world,
                             int64_t slot_offset_floats, const uint64_t* peer_flags_dev, int rank, int epoch, int first, int do_reset,
                             int aviary_index, void* stream) {
  REQUIRE_BOUND(h);
  if (!is_df(h)) return fail("handle is not a dogfight env");
  if (!peer_tables_dev || world < 1) return fail("pfb_dogfight_physics_peer: need the device array of peer table pointers");
  return df_split_physics(h, actions ? actions : h->buf.setpoint, noise, nullptr, peer_tables_dev, world, slot_offset_floats, peer_flags_dev, rank,
                          epoch, first, do_reset, aviary_index, (cudaStream_t)stream);
}

int pfb_dogfight_combat(PfbHandle h, const float* payload_table, int64_t first_global_agent, int64_t num_arenas, int last, void* stream) {
  REQUIRE_BOUND(h);
  if (!is_df(h)) return fail("handle is not a dogfight env");
  if (require_env(h)) return -1;
  return df_split_combat(h, payload_table, first_global_agent, num_arenas, last, nullptr, 0, 0, (cudaStream_t)stream);
}

int pfb_dogfight_combat_wait(PfbHandle h, const float* payload_table, int64_t first_global_agent, int64_t num_arenas, int last,
                             const int32_t* flags, int world, int epoch, void* stream) {
  REQUIRE_BOUND(h);
  if (!is_df(h)) return fail("handle is not a dogfight env");
  if (require_env(h)) return -1;
  if (!flags) return fail("pfb_dogfight_combat_wait: null flag array");
  return df_split_combat(h, payload_table, first_global_agent, num_arenas, last, flags, world, epoch, (cudaStream_t)stream);
}

// One whole env step of the split dogfight with the fused exchange: env_step_ratio x (physics with peer stores + in-kernel
// signal, combat with in-kernel wait).  Nothing between the kernels needs the host, so the step is ONE call.
int pfb_dogfight_split_step(PfbHandle h, const float* actions, const uint64_t* peer_tables_dev, const uint64_t* peer_flags_dev,
                            const float* local_tables, const int32_t* local_flags, int world, int rank, int epoch0,
                            int64_t first_global_agent, int64_t num_arenas, void* stream) {
  REQUIRE_BOUND(h);
  if (!is_df(h)) return fail("handle is not a dogfight env");
  if (require_env(h)) return -1;
  if (!peer_tables_dev || !peer_flags_dev || !local_tables || !local_flags) return fail("pfb_dogfight_split_step: null argument");
  const int64_t na = 2 * num_arenas;
  const int ratio = h->env.env_step_ratio;
  for (int k = 0; k < ratio; ++k) {
    const int epoch = epoch0 + k;          // exchange number, 1-based; its parity selects the half of the double-buffered table
    const int phase = (epoch - 1) & 1;
    if (df_split_physics(h, actions ? actions : h->buf.setpoint, nullptr, nullptr, peer_tables_dev, world, (phase * na + first_global_agent) * 20,
                         peer_flags_dev, rank, epoch, k == 0, 0, k, (cudaStream_t)stream))
      return -1;
    if (df_split_combat(h, local_tables + phase * na * 20, first_global_agent, num_arenas, k == ratio - 1, local_flags, world, epoch,
                        (cudaStream_t)stream))
      return -1;
  }
  return 0;
}

int64_t pfb_launch_count(PfbHandle h) { return h ? h->launches : 0; }

int pfb_profile_begin(PfbHandle h, int capacity) {
  if (!h) return fail("null handle");
  CUDA_OK(cudaSetDevice(h->device));
  if (h->prof_ev) {
    for (int i = 0; i < 2 * h->prof_cap; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev;
    h->prof_ev = nullptr;
  }
  h->prof_cap = 0;
  h->prof_n = 0;
  if (capacity <= 0) return 0;
  h->prof_ev = new (std::nothrow) cudaEvent_t[2 * (size_t)capacity];
  if (!h->prof_ev) return fail("out of host memory");
  for (int i = 0; i < 2 * capacity; ++i) CUDA_OK(cudaEventCreate(&h->prof_ev[i]));
  h->prof_cap = capacity;
  return 0;
}

int pfb_profile_read(PfbHandle h, float* ms_out, int capacity) {
  if (!h) return fail("null handle");
  CUDA_OK(cudaSetDevice(h->device));
  int n = h->prof_n < capacity ? h->prof_n : capacity;
  for (int i = 0; i < n; ++i) CUDA_OK(cudaEventElapsedTime(&ms_out[i], h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
  return n;
}

}  // extern "C"
