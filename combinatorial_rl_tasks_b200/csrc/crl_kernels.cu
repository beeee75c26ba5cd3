// crl_kernels.cu -- sm_100a kernels and the C ABI (include/crl_b200.h) of the
// batched Point-robot zone-task simulator.
//
// One thread per env.  Per env-step a thread (order as executed, see step_kernel)
//   1. loads its state planes (two float4), its action (float2) and its N zone
//      centres (float2 each, plane-major so every load is a coalesced 256-B row),
//   2. tests the zone event on the PRE-physics position (TSP_env.py:54-69,
//      colour_match_env.py:106-120) -- fp32 screen, exact fp64 confirm,
//   3. applies reward / goal / timeout / done (TSP_env.py:37-42,71-72,
//      TTSP_env.py:62-71, colour_match_env.py:86-93,122-123, Engine.step) -- none of it
//      depends on the post-physics state -- and writes the CrlResult record,
//   4. if the env finished and auto-reset is on, takes its next layout from the slot the
//      background sampler parked it in (prefetch_*_kernel); only if the slot is empty does
//      its warp build the layout cooperatively (32 rejection-sampling candidates per round),
//   5. stages its zone_obs row in shared memory, from where each warp's 32 rows (one
//      contiguous span of B x N x Z) leave with a single cp.async.bulk shared->global copy
//      (CRL_STEP_ZONE_OBS_DELTA: only the rows that change are built and written),
//   6. integrates all frameskip substeps in registers (crl_core.cuh) while that copy drains,
//   7. writes state and the 8-float obs row.
// Episode statistics go through warp ballots and one atomic per warp.  Also here: the
// goal-conditioned / WaitWrapper variant of the step (EXT), the host-facing steps
// (crl_step_host, crl_host_call_*), goal RPC kernels and crl_gae.
#include <cuda_runtime.h>

#include <atomic>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/crl_b200.h"
#include "crl_core.cuh"

namespace crl {

#ifndef CRL_THREADS
#define CRL_THREADS 64
#endif
constexpr int kThreads = CRL_THREADS;
constexpr unsigned kFull = 0xffffffffu;

struct KParams {
  // config
  int B, num_steps, frameskip, max_cd, seed_mode, env_offset;
  long long min_seed, max_seed;
  double thresh2;        // sqrt_threshold(zone_size)
  float r2_guard;        // fp32 screen radius^2
  double bonus_per_step; // time_saved_reward
  double beta_a, beta_b;
  float robot_keepout, zone_keepout, extent;
  unsigned flags;
  DivConst div_steps, div_cd;   // x / num_steps, x / max_cooldown (crl_core.cuh)
  unsigned long long action_seed, step_index;
  // state
  float4* pose;
  float4* aux;
  float2* zone_xy;
  uint32_t* zone_tmax;
  uint2* cooldown;
  long long* seed;
  uint32_t* episode;
  float4* origin;
  double* counters;
  float2* next_zone_xy;
  uint32_t* next_task;
  float4* next_origin;
  long long* next_seed;
  uint32_t* next_ready;
  uint32_t* stamp;
  uint32_t* act_count;          // stamp plane 2: NULL-action steps taken per 32 envs (CRL_STEP_ACTION_COUNTER)
  const uint32_t* epoch;        // CrlState.prefetch_epoch: last sampler round whose slots the step may trust
  uint32_t round;               // crl_prefetch_layouts: the round being run
  uint32_t* row_list;
  float* zone_obs_host;         // host-direct step: the caller's host zone_obs (device-mapped); changed rows go there
  unsigned long long* result_dev;   // host-direct step: the DEVICE copy of the result records (`result` is then the host's)
  int32_t* goal;
  const float2* bank_zone_xy;
  const float4* bank_origin;
  const uint32_t* bank_task;
  const float4* fixed;          // fixed placements (CrlState.fixed_layout), or nullptr
  uint32_t init_hi;             // visited mask an episode starts with (CrlConfig.initial_visited)
  uint32_t walled;              // CrlConfig.walled: the arena's wall boxes exist (EXT kernels only)
  // io
  const float2* actions;
  float4* obs;
  float* zone_obs;
  unsigned long long* result;  // CrlResult as one 8-byte word
  float* shaped;               // info['shaped_reward'] (goal-conditioned variants)
  const uint8_t* mask;
};

constexpr uint32_t kParBit = 0x8000u, kHiMask = 0x7fffu;

template <int TASK>
struct ZoneDim { static constexpr int Z = (TASK == CRL_TASK_TSP) ? 6 : 7; };

// Registers per thread the step kernel is compiled for.  Occupancy is set by the zone_obs stage (32 rows
// per warp in shared memory: 8 CTAs = 16 warps per SM at 15 zones, 12 CTAs = 24 warps at <= 8), and the
// register cap is chosen to LEAVE ROOM beside those CTAs: 8 x 64 x 112 = 57,344 (12 x 64 x 80 = 61,440) of
// the SM's 65,536 registers, so that four (two) 32-thread CTAs of the background layout sampler (64
// registers) fit without displacing a step CTA.  At 128 registers the step kernel fills the register file exactly, every
// sampler CTA costs the SM an eighth of its step warps for as long as it runs, and TimedTSP -- whose sampler
// runs all the time -- loses a fifth of its throughput (profiles/r02_notes.md).
#ifndef CRL_REGS_N15
#define CRL_REGS_N15 112
#endif
template <int N>
struct MaxRegs { static constexpr int v = N > 8 ? CRL_REGS_N15 : 80; };

// Registers describing one env between load and store.
template <int N>
struct Env {
  Body b;
  float ep_return;
  int steps;
  uint32_t hi;        // bits 0-14: visited mask or colour codes; bit 15: parity of the env's episode
                      // counter (= the next-layout slot its next reset takes, kParBit)
  float2 zone[N];
  uint32_t tmax[(N + 1) / 2];
  uint2 cd;
};

__device__ __forceinline__ uint32_t cd_get(const uint2& cd, int i) {
  const uint32_t w = i < 4 ? cd.x : cd.y;
  return (w >> (8 * (i & 3))) & 0xffu;
}
__device__ __forceinline__ void cd_set(uint2& cd, int i, uint32_t v) {
  uint32_t& w = i < 4 ? cd.x : cd.y;
  const int sh = 8 * (i & 3);
  w = (w & ~(0xffu << sh)) | (v << sh);
}
// every positive byte minus one (colour_match_env.py:98-100), SWAR on 4 bytes
__device__ __forceinline__ uint32_t cd_dec4(uint32_t w) {
  // nonzero-byte mask: 0x01 in each byte that is > 0
  const uint32_t nz = (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) >> 7 & 0x01010101u;
  return w - nz;
}

// ---- reset: draws for one env, made by a whole warp ---------------------------

// Philox key = the Engine seed in force for the draw (two 32-bit halves).
__device__ __forceinline__ U4 draw(long long seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t tag) {
  U4 ctr{c0, c1, c2, tag};
  return philox4x32(ctr, (uint32_t)(unsigned long long)seed, (uint32_t)((unsigned long long)seed >> 32));
}

// Marsaglia-Tsang gamma(a), a >= 1, from a counter stream (fp64: reset is off the hot path).
// General-shape fallback; the reference's shapes take gamma_half_integer below.
__device__ double gamma_mt(long long seed, double a, uint32_t zone, uint32_t which) {
  const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  for (uint32_t it = 0;; ++it) {
    const U4 r0 = draw(seed, it, zone, which, kTagTask);
    const U4 r1 = draw(seed, it, zone, which + 2u, kTagTask);
    const double u1 = u01d(r0.x, r0.y), u2 = u01d(r0.z, r0.w), u3 = u01d(r1.x, r1.y);
    const double x = sqrt(-2.0 * log(u1)) * cos(2.0 * kPi * u2);   // Box-Muller
    double v = 1.0 + c * x;
    if (v <= 0.0) continue;
    v = v * v * v;
    if (log(u3) < 0.5 * x * x + d - d * v + d * log(v) || it > 64u) return d * v;
  }
}

// gamma(k/2) for a small integer k, exactly and without rejection: the sum of floor(k/2)
// unit exponentials, -log(u_0 ... u_{m-1}), plus, for odd k, half the square of a standard
// normal, -log(U) cos^2(2 pi V) (Box-Muller squared).  TTSP_env.py:20 draws beta(3, 1.5):
// k = 6 and k = 3, i.e. three logs and one cosine per zone and no data-dependent loop.
// Uniform j of the stream is half j&1 of Philox block j>>1 (counter = (block, zone, which)).
__device__ double gamma_half_integer(long long seed, int k, uint32_t zone, uint32_t which) {
  const int m = k >> 1;
  double prod = 1.0, U = 1.0, V = 0.0;
  const int n_u = m + ((k & 1) ? 2 : 0);
  for (int j = 0; j < n_u; j += 2) {
    const U4 r = draw(seed, (uint32_t)(j >> 1), zone, which, kTagTask);
    const double ua = u01d(r.x, r.y), ub = u01d(r.z, r.w);
    if (j < m) prod *= ua; else if (j == m) U = ua; else V = ua;
    if (j + 1 < m) prod *= ub; else if (j + 1 == m) U = ub; else if (j + 1 < n_u) V = ub;
  }
  double g = -log(prod);
  if (k & 1) {
    const double c = cos(2.0 * kPi * V);
    g += -log(U) * (c * c);
  }
  return g;
}

// 2a if gamma_half_integer applies to shape a (2a a whole number in [1, 16]), else 0
CRL_HD int half_integer_shape(double a) {
  const double t = 2.0 * a;
  const int k = (int)t;
  return ((double)k == t && k >= 1 && k <= 16) ? k : 0;
}

__device__ double gamma_draw(long long seed, double a, uint32_t zone, uint32_t which) {
  const int k = half_integer_shape(a);
  return k ? gamma_half_integer(seed, k, zone, which) : gamma_mt(seed, a, zone, which);
}

// ColourMatch colour of one zone (colour_match_env.py:60-61, rs.choice of three): uniform
// over {0,1,2} by masked rejection on the 2-bit fields of a Philox word.
__device__ uint32_t colour_draw(long long seed, uint32_t zone) {
  uint32_t c = 3u;
  for (uint32_t it = 0; c == 3u && it < 64u; ++it) {
    const U4 r = draw(seed, it, zone, 0u, kTagTask);
    uint32_t bits = r.x;
    for (int q = 0; q < 16 && c == 3u; ++q, bits >>= 2) c = bits & 3u;
  }
  return c == 3u ? 0u : c;
}

// Rejection-sample robot + N zones exactly as Engine.sample_layout orders it (object by
// object, <= 100 tries each, first valid try wins, 100 misses abandon the layout), but
// 32 tries at a time across the warp.  Candidate j of object k in attempt L is a pure
// function of (seed, j, k, L) -- half (j & 1) of Philox block (j >> 1, k, L) -- so the
// outcome equals the sequential procedure's.
// `placed` is warp-private shared scratch of N+1 float2 (16-byte aligned).
// FIXED: honour CrlState.fixed_layout (hard instances).  A template parameter, not a run-time test,
// so that the step kernels of the registrations without fixed placements are compiled exactly as if
// the feature did not exist (ptxas' register allocation of the whole step kernel moved with it:
// TimedTSP 262,144 envs lost 9 % with the run-time test, profiles/r01_notes.md).
template <int N, bool FIXED>
__device__ void warp_layout(const KParams& p, long long seed, float2* placed, int lane) {
  const float ext = p.extent;
  constexpr int NP = (N + 2) / 2;                 // float4 pairs covering placed[0..N]
#pragma unroll 1
  for (uint32_t attempt = 0; attempt < 10000u; ++attempt) {
    bool ok_layout = true;
#pragma unroll 1
    for (int k = 0; k <= N && ok_layout; ++k) {
      const float keep = k == 0 ? p.robot_keepout : p.zone_keepout;
      float lo_x = -ext + keep, lo_y = lo_x, span = (ext - keep) - lo_x;
      // an object with a fixed location (CrlState.fixed_layout): a box of width 0 at that location,
      // so every try is the location itself (x = lo + 0 * u) and one miss means a hundred
      if (FIXED && p.fixed) {
        const float4 fx = p.fixed[k];
        if (fx.w == 1.f || fx.w == 3.f) { lo_x = fx.x; lo_y = fx.y; span = 0.f; }
      }
      // everything placed so far, read once per object with independent 16-byte loads
      float4 pl[NP];
#pragma unroll
      for (int q2 = 0; q2 < NP; ++q2) pl[q2] = reinterpret_cast<const float4*>(placed)[q2];
      bool found = false;
#pragma unroll 1
      for (int base = 0; base < 100 && !found; base += 32) {
        const int j = base + lane;
        // try j = half (j & 1) of Philox block (j >> 1): one block serves two tries
        const U4 r = draw(seed, (uint32_t)(j >> 1), (uint32_t)k, attempt, kTagLayout);
        const float x = __fadd_rn(lo_x, __fmul_rn(span, u01((j & 1) ? r.z : r.x)));
        const float y = __fadd_rn(lo_y, __fmul_rn(span, u01((j & 1) ? r.w : r.y)));
        bool valid = j < 100;
#pragma unroll
        for (int q = 0; q < N; ++q) {             // slots >= k hold stale values and are ignored
          const float ox = (q & 1) ? pl[q >> 1].z : pl[q >> 1].x;
          const float oy = (q & 1) ? pl[q >> 1].w : pl[q >> 1].y;
          const float need = __fadd_rn(q == 0 ? p.robot_keepout : p.zone_keepout, keep);
          const float dx = __fsub_rn(x, ox), dy = __fsub_rn(y, oy);
          const float d2 = __fmaf_rn(dy, dy, __fmul_rn(dx, dx));   // the form of the packed test in prefetch_layout_kernel
          valid = valid && (q >= k || d2 >= __fmul_rn(need, need));
        }
        const unsigned m = __ballot_sync(kFull, valid);
        if (m) {
          const int wlane = __ffs(m) - 1;
          const float wx = __shfl_sync(kFull, x, wlane), wy = __shfl_sync(kFull, y, wlane);
          if (lane == 0) placed[k] = make_float2(wx, wy);
          found = true;
        }
      }
      __syncwarp();
      ok_layout = found;
    }
    if (ok_layout) return;
  }
}

// The seed the reset number (episode + ahead) of env e will run with (lane-local), ahead = 0
// for the next reset.  CRL_SEED_INCREMENT: the env's current seed, +1 per further reset
// (Engine.reset: self._seed += 1).  CRL_SEED_FIXED_RANGE: FixedSeedsWrapper.reset, a uniform
// integer in [min_seed, max_seed] from the chooser's own stream (key = GLOBAL env index,
// counter = episode number).
__device__ __forceinline__ long long choose_seed(const KParams& p, int e, uint32_t episode, uint32_t ahead = 0u) {
  if (p.seed_mode != CRL_SEED_FIXED_RANGE) return p.seed[e] + (long long)ahead;
  const unsigned long long span = (unsigned long long)(p.max_seed - p.min_seed) + 1ull;
  const U4 r = draw((long long)(p.env_offset + e), episode + ahead, 0u, 0u, kTagSeed);
  const unsigned long long v = ((unsigned long long)r.x << 32) | r.y;
  return p.min_seed + (long long)(span ? (v % span) : v);
}

// All draws of one Engine.reset run with seed `chosen`, made by a whole warp: task draws
// with the seed BEFORE the increment (TTSP_env.py:20, colour_match_env.py:60), layout and
// heading with chosen + 1 (Engine.reset: self._seed += 1).  On return placed[0] = robot,
// placed[1..N] = zones (shared memory), lane i < N holds zone i's timeout / colour in
// `my_draw`, every lane holds rot0.
template <int TASK, int N, bool FIXED>
__device__ void warp_generate(const KParams& p, long long chosen, float2* placed, int lane,
                              uint32_t& my_draw, float& rot0) {
  my_draw = 0u;
  if (TASK == CRL_TASK_TTSP && lane < N) {
    const double ga = gamma_draw(chosen, p.beta_a, (uint32_t)lane, 0u);
    const double gb = gamma_draw(chosen, p.beta_b, (uint32_t)lane, 1u);
    const int t = (int)((ga / (ga + gb)) * (double)p.num_steps);
    my_draw = (uint32_t)min(max(t, 0), 65535);
  }
  if (TASK == CRL_TASK_CM && lane < N) my_draw = colour_draw(chosen, (uint32_t)lane);
  warp_layout<N, FIXED>(p, chosen + 1, placed, lane);
  const U4 rr = draw(chosen + 1, 0u, 0u, 0u, kTagRot);
  rot0 = __fmul_rn(6.2831855f, u01(rr.x));
  if (FIXED && p.fixed) { const float4 f0 = p.fixed[0]; if (f0.w >= 2.f) rot0 = f0.z; }   // Engine.robot_rot
  __syncwarp();
}

// next-layout slot states (CrlState.next_ready)
// kSlotReady + r: ready, filled by sampler round r.  A step trusts such a slot only if r <= *epoch, the
// last round the HOST has ordered before it (crl_prefetch_publish): everything that round wrote is then
// visible by stream order, so the step reads flag, seed and layout with plain independent loads -- one
// round trip, no acquire (each acquire used to invalidate the L1 under the warp's siblings) and no
// release when it hands the slot back (the next round's scan is ordered after the step by the host).
constexpr uint32_t kSlotEmpty = 0u, kSlotLayoutDone = 2u, kSlotClaimed = 3u, kSlotReady = 16u;

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}

// The hot way through an auto-reset, INLINE in the step kernel and lane-local: take the env's parked
// next layout if the slot (parity in the state word) holds a trusted one drawn for the seed this
// reset runs with.  Inline because a call would see the kernel parameters through a generic pointer
// (every `p.x` a memory load and a dependent round trip: ~10 us per resetting warp under load,
// profiles/r02_notes.md) where the kernel itself reads them from the constant bank; lean because it
// writes the new layout straight into the env's own registers, which are dead once the episode is
// over.  Returns false (env.zone / tmax clobbered, nothing stored) when the slot cannot be used: the
// out-of-line warp_reset then rebuilds the env.
template <int TASK, int N>
__device__ __forceinline__ bool reset_from_slot(const KParams& p, int e, Env<N>& env) {
  const int B = p.B;
  const uint32_t par = env.hi >> 15;
  uint32_t episode, col_word = 0u;
  long long chosen;
  float4 o;
  uint32_t* slot_flag = nullptr;
  if (p.bank_zone_xy) {
    // fixed task set (make_train_env's num_training_tasks maps): the map of seed `chosen` is entry
    // chosen - min_seed of the layout bank (a few KB, cache resident): copy it, nothing to sample
    episode = p.episode[e];
    chosen = choose_seed(p, e, episode);
    if (chosen < p.min_seed || chosen > p.max_seed) return false;
    const size_t k = (size_t)(chosen - p.min_seed);
    o = p.bank_origin[k];
#pragma unroll
    for (int i = 0; i < N; ++i) env.zone[i] = p.bank_zone_xy[k * N + i];
    if (TASK == CRL_TASK_TTSP) {
#pragma unroll
      for (int j = 0; j < (N + 1) / 2; ++j) env.tmax[j] = p.bank_task[k * ((N + 1) / 2) + j];
    }
    if (TASK == CRL_TASK_CM) col_word = p.bank_task[k];
  } else {
    if (!p.next_ready) return false;
    const size_t sb = (size_t)par * (size_t)B;
    slot_flag = p.next_ready + sb + e;
    const float2* nz = p.next_zone_xy + sb * N + e;
    const uint32_t flag = ld_relaxed_u32(slot_flag);
    const uint32_t trusted = ld_relaxed_u32(p.epoch);
    episode = p.episode[e];
    const long long parked_for = __ldcg(p.next_seed + sb + e);
    o = __ldcg(p.next_origin + sb + e);
#pragma unroll
    for (int i = 0; i < N; ++i) env.zone[i] = __ldcg(nz + (size_t)i * B);
    if (TASK == CRL_TASK_TTSP) {
      const uint32_t* nt = p.next_task + sb * ((N + 1) / 2) + e;
#pragma unroll
      for (int j = 0; j < (N + 1) / 2; ++j) env.tmax[j] = __ldcg(nt + (size_t)j * B);
    }
    if (TASK == CRL_TASK_CM) col_word = __ldcg(p.next_task + sb + e);
    chosen = choose_seed(p, e, episode);
    if (!(flag >= kSlotReady && flag - kSlotReady <= trusted && parked_for == chosen && (episode & 1u) == par)) return false;
  }
#pragma unroll
  for (int i = 0; i < N; ++i) p.zone_xy[(size_t)i * B + e] = env.zone[i];
  if (TASK == CRL_TASK_TTSP) {
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) p.zone_tmax[(size_t)j * B + e] = env.tmax[j];
  }
  env.b.X = o.x; env.b.Y = o.y; env.b.phi = wrap_pi(o.z);
  env.b.vx = env.b.vy = env.b.w = 0.f;
  env.ep_return = 0.f;
  env.steps = 0;
  env.hi = (TASK == CRL_TASK_CM ? col_word : p.init_hi) | (((episode + 1u) & 1u) ? kParBit : 0u);
  env.cd = make_uint2(0u, 0u);
  p.seed[e] = chosen + 1;                         // Engine.reset: self._seed += 1
  p.episode[e] = episode + 1u;
  p.origin[e] = make_float4(o.x, o.y, o.z, 0.f);
  if (p.goal) p.goal[e] = -1;                     // a new episode has no goal until set_goal
  if (slot_flag) *slot_flag = kSlotEmpty;         // plain store: the next sampler round is ordered after this kernel
  return true;
}

// Engine.reset for the lanes in `dm` (each lane = one env).  A lane whose next layout
// was prefetched (next_ready set for exactly the seed this reset runs with) only copies
// it: no sampling latency on the step's critical path.  The others are rebuilt one at a
// time by the whole warp.  Both ways produce the same layout: it is a pure function of
// the seed.
//
// The function is out of line (cold, register-hungry); `out` (the caller's Env copy) therefore
// lives in local memory.  It is WRITE-ONLY here: with the L1 thrashed by the step's streaming
// loads, a local load is an L2 round trip, and the 23
// plane stores used to read their values back from it one after the other (~14 us per resetting
// warp, profiles/r01_notes.md).  Now the new zone centres / timeouts go straight from registers
// to their planes, and the caller reads its copy back once, in one batch of independent loads.
template <int TASK, int N, bool FIXED, bool PAR_FROM_EPISODE = false>
__device__ __noinline__ void warp_reset(const KParams& p, unsigned dm, int lane, int e, float2* placed, uint32_t par_in,
                                        Env<N>& out) {
  const bool mine = (dm >> lane) & 1u;
  long long chosen = 0;
  uint32_t episode = 0;
  bool fast = false;
  float x0 = 0.f, y0 = 0.f, rot0 = 0.f;
  uint32_t col_word = 0u;
  const int B = p.B;
  uint32_t* slot_flag = nullptr;
  float2* zp = p.zone_xy + e;
  uint32_t* tp = p.zone_tmax + e;
  if (mine) {
    if (p.bank_zone_xy || !p.next_ready || PAR_FROM_EPISODE) episode = p.episode[e];
    if (p.bank_zone_xy && (chosen = choose_seed(p, e, episode)) >= p.min_seed && chosen <= p.max_seed) {
      // fixed task set: the map of seed `chosen` is entry chosen - min_seed of the layout bank
      // (a few KB, cache resident): copy it, nothing to sample
      const size_t k = (size_t)(chosen - p.min_seed);
      const float4 o = p.bank_origin[k];
      fast = true;
      x0 = o.x; y0 = o.y; rot0 = o.z;
#pragma unroll
      for (int i = 0; i < N; ++i) { const float2 z = p.bank_zone_xy[k * N + i]; zp[(size_t)i * B] = z; out.zone[i] = z; }
      if (TASK == CRL_TASK_TTSP) {
#pragma unroll
        for (int j = 0; j < (N + 1) / 2; ++j) {
          const uint32_t t = p.bank_task[k * ((N + 1) / 2) + j];
          tp[(size_t)j * B] = t; out.tmax[j] = t;
        }
      }
      if (TASK == CRL_TASK_CM) col_word = p.bank_task[k];
    } else if (p.next_ready) {
      // Reset number n takes slot n & 1, and that parity rides in the env's state word: the slot is
      // known without a load, so the episode counter, the env's seed, the slot's flag / seed / origin
      // / zone centres / task draws and the trusted epoch are ONE batch of independent loads.
      const uint32_t par = PAR_FROM_EPISODE ? (episode & 1u) : par_in;
      const size_t sb = (size_t)par * (size_t)B;
      slot_flag = p.next_ready + sb + e;
      const float2* nz = p.next_zone_xy + sb * N + e;
      const uint32_t* nt = p.next_task ? p.next_task + sb * (TASK == CRL_TASK_TTSP ? (N + 1) / 2 : 1) + e : nullptr;
      const uint32_t flag = ld_relaxed_u32(slot_flag);
      const uint32_t trusted = ld_relaxed_u32(p.epoch);
      if (!PAR_FROM_EPISODE) episode = p.episode[e];
      const long long parked_for = __ldcg(p.next_seed + sb + e);
      const float4 o = __ldcg(p.next_origin + sb + e);
      float2 z[N];
      uint32_t t[(N + 1) / 2];
#pragma unroll
      for (int i = 0; i < N; ++i) z[i] = __ldcg(nz + (size_t)i * B);
      if (TASK == CRL_TASK_TTSP) {
#pragma unroll
        for (int j = 0; j < (N + 1) / 2; ++j) t[j] = __ldcg(nt + (size_t)j * B);
      }
      if (TASK == CRL_TASK_CM) t[0] = __ldcg(nt);
      chosen = choose_seed(p, e, episode);
      const bool ready = flag >= kSlotReady && flag - kSlotReady <= trusted;
      if (ready && parked_for == chosen && (episode & 1u) == par) {
        fast = true;
        x0 = o.x; y0 = o.y; rot0 = o.z;
#pragma unroll
        for (int i = 0; i < N; ++i) { zp[(size_t)i * B] = z[i]; out.zone[i] = z[i]; }
        if (TASK == CRL_TASK_TTSP) {
#pragma unroll
          for (int j = 0; j < (N + 1) / 2; ++j) { tp[(size_t)j * B] = t[j]; out.tmax[j] = t[j]; }
        }
        if (TASK == CRL_TASK_CM) col_word = t[0];
      }
      // hand the slot back only if it held a finished layout (now consumed, or stale: drawn for a seed
      // this env has moved past); a slot the running sampler round owns is left alone.  The slot of
      // THIS reset is (episode & 1); a state word whose parity disagrees (seed() without a reset)
      // just samples inline and is corrected below.
      if (!ready || (episode & 1u) != par) slot_flag = nullptr;
    } else {
      chosen = choose_seed(p, e, episode);
    }
  }
  unsigned slow = __ballot_sync(kFull, mine && !fast);
  while (slow) {
    const int src = __ffs(slow) - 1;
    slow &= slow - 1;
    const long long ch = __shfl_sync(kFull, chosen, src);
    uint32_t my_draw;
    float r0;
    warp_generate<TASK, N, FIXED>(p, ch, placed, lane, my_draw, r0);
    uint32_t cw = 0u;
    uint32_t tm[(N + 1) / 2];
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) tm[j] = 0u;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const uint32_t d = __shfl_sync(kFull, my_draw, i);
      tm[i >> 1] |= d << (16 * (i & 1));
      cw |= d << (2 * i);
    }
    if (lane == src) {
      const float2 rb = placed[0];
      x0 = rb.x; y0 = rb.y; rot0 = r0; col_word = cw;
#pragma unroll
      for (int i = 0; i < N; ++i) { const float2 z = placed[1 + i]; zp[(size_t)i * B] = z; out.zone[i] = z; }
      if (TASK == CRL_TASK_TTSP) {
#pragma unroll
        for (int j = 0; j < (N + 1) / 2; ++j) { tp[(size_t)j * B] = tm[j]; out.tmax[j] = tm[j]; }
      }
    }
    __syncwarp();
  }
  if (mine) {
    out.b.X = x0; out.b.Y = y0; out.b.phi = wrap_pi(rot0);
    out.b.vx = out.b.vy = out.b.w = 0.f;
    out.ep_return = 0.f;
    out.steps = 0;
    out.hi = (TASK == CRL_TASK_CM ? col_word : p.init_hi) | (((episode + 1u) & 1u) ? kParBit : 0u);
    out.cd = make_uint2(0u, 0u);
    p.seed[e] = chosen + 1;                       // Engine.reset: self._seed += 1
    p.episode[e] = episode + 1u;
    p.origin[e] = make_float4(x0, y0, rot0, 0.f);
    if (p.goal) p.goal[e] = -1;                   // a new episode has no goal until set_goal
    // hand the slot back to the sampler: a plain store, the next round's scan is ordered after this
    // kernel by the host (crl_prefetch_layouts is enqueued behind the steps it follows)
    if (slot_flag) *slot_flag = kSlotEmpty;
  }
  const unsigned fm = __ballot_sync(kFull, mine && fast);
  if (lane == 0) {
    if (fm) atomicAdd(p.counters + 4, (double)__popc(fm));
    if (dm & ~fm) atomicAdd(p.counters + 5, (double)__popc(dm & ~fm));
  }
  __syncwarp();
}

// packed fp32 pairs (Blackwell: add / sub / mul / fma .f32x2), IEEE round-to-nearest per half
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long sub_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long mul_f32x2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ unsigned long long fma_f32x2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}

// ---- background prefetch of next layouts -------------------------------------------
// Every env has TWO next-layout slots: reset number n takes slot n & 1, so the layouts of
// its next two resets can be parked at once and an env that finishes again before the
// prefetcher has come round still finds its layout (with one slot, about one launch in two
// at 262,144 TimedTSP envs met an empty slot and stalled on the inline sampler).  The seeds
// of both resets are known in advance in both seed modes.  The prefetcher runs off the
// step's stream and the step never waits for it: slots change hands through acquire /
// release flags, and an env whose slot is empty samples inline with the identical result.
//
// Three kernels.  (0) prefetch_scan_kernel compacts the empty slots into a dense work list
// (env, slot, seed).  (A) prefetch_layout_kernel: the rejection sampler with ONE LANE PER
// LAYOUT.  The warp-cooperative sampler above spends a 32-candidate round on an object whose
// first candidate is usually valid (about 44 rounds of ~300 instructions per 15-zone layout);
// here each lane runs the sequential procedure itself, one candidate per iteration, so all
// 32 lanes do useful work (about 435 candidates per layout = 14 warp-rounds per layout).
// Lanes are persistent: a lane that finishes takes the next work item, so the long tail of
// the sampler (p99 is 4x the mean) does not idle a warp.  Candidate j of object k in attempt
// L is the same function of (seed, j, k, L) in both samplers: same layout bit for bit.
// (B) prefetch_task_kernel: TimedTSP timeouts / ColourMatch colours, one lane per (item,
// zone), two items per warp iteration.
// Slot states: empty -> claimed (in the work list) -> [layout parked, task draws pending] -> ready.
struct WorkItem { int e; uint32_t slot; long long seed; };   // 16 bytes; item 0 of the plane is the header
struct WorkHeader { uint32_t count, cursor, pad0, pad1; };

template <int N>
__global__ void __launch_bounds__(64) prefetch_scan_kernel(const __grid_constant__ KParams p, WorkItem* work) {
  WorkHeader* hdr = reinterpret_cast<WorkHeader*>(work);
  const int lane = threadIdx.x & 31;
  const int n_round = (p.B + 31) & ~31;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_round; e += gridDim.x * blockDim.x) {
    const bool in = e < p.B;
    const uint32_t episode = in ? p.episode[e] : 0u;
#pragma unroll
    for (uint32_t ahead = 0; ahead < 2u; ++ahead) {
      const uint32_t slot = (episode + ahead) & 1u;
      uint32_t* flag = p.next_ready + (size_t)slot * p.B + e;
      // claim with a compare-and-swap: two rounds that overlap (they should not: the host orders
      // them) can then never list the same slot twice
      const bool want = in && ld_relaxed_u32(flag) == kSlotEmpty && atomicCAS(flag, kSlotEmpty, kSlotClaimed) == kSlotEmpty;
      const unsigned m = __ballot_sync(kFull, want);
      if (m) {
        uint32_t base = 0u;
        if (lane == 0) base = atomicAdd(&hdr->count, (uint32_t)__popc(m));
        base = __shfl_sync(kFull, base, 0);
        if (want) {
          WorkItem it;
          it.e = e; it.slot = slot; it.seed = choose_seed(p, e, episode, ahead);
          work[1u + base + (uint32_t)__popc(m & ((1u << lane) - 1u))] = it;
        }
      }
    }
  }
}

// The objects placed so far live in REGISTERS (written through a predicated unrolled select, read
// with static indices): no shared memory, so that the sampler's resident CTAs never cost the
// step kernel a CTA slot (4 x 53.8 KB of TimedTSP staging leave 9 KB of an SM's 228 KB).
template <int N>
__global__ void __launch_bounds__(32) prefetch_layout_kernel(const __grid_constant__ KParams p, WorkItem* work,
                                                             uint32_t done_state) {
  float2 placed[N + 1];
#pragma unroll
  for (int q = 0; q <= N; ++q) placed[q] = make_float2(0.f, 0.f);
  WorkHeader* hdr = reinterpret_cast<WorkHeader*>(work);
  const int lane = threadIdx.x;
  const uint32_t count = hdr->count;              // final: the scan kernel precedes this one on the stream
  const float rk = p.robot_keepout, zk = p.zone_keepout, ext = p.extent;
  bool have = false, drained = false;
  int e = -1, k = 0, j = 0;
  uint32_t attempt = 0u, slot = 0u;
  long long layout_seed = 0;
  for (;;) {
    const unsigned idle = __ballot_sync(kFull, !have);
    if (idle && !drained) {                       // one atomic refills every idle lane of the warp
      uint32_t base = 0u;
      if (lane == 0) base = atomicAdd(&hdr->cursor, (uint32_t)__popc(idle));
      base = __shfl_sync(kFull, base, 0);
      drained = base + (uint32_t)__popc(idle) >= count;
      const uint32_t idx = base + (uint32_t)__popc(idle & ((1u << lane) - 1u));
      if (!have && idx < count) {
        const WorkItem it = work[1u + idx];
        e = it.e; slot = it.slot; layout_seed = it.seed + 1;   // Engine.reset: _seed += 1 before the layout
        have = true; k = 0; j = 0; attempt = 0u;
      }
    }
    if (__ballot_sync(kFull, have) == 0u) break;
    if (have) {
      // TWO tries of Engine.sample_layout's sequential procedure per iteration: tries j and j + 1 are
      // the two halves of one Philox block, so the block is computed once per iteration by every lane
      // (with one try per iteration the lanes' parities differ and the warp paid for the block every
      // time), and the two distance tests are independent chains.  The first valid try in index
      // order wins, exactly as before.
      const float keep = k == 0 ? rk : zk;
      float lo_x = -ext + keep, lo_y = lo_x, span = (ext - keep) - lo_x;
      bool pinned = false;                        // fixed location: a box of width 0, one try
      if (p.fixed) {
        const float4 fx = p.fixed[min(k, N)];
        if (fx.w == 1.f || fx.w == 3.f) { lo_x = fx.x; lo_y = fx.y; span = 0.f; pinned = true; }
      }
      const U4 r = draw(layout_seed, (uint32_t)(j >> 1), (uint32_t)k, attempt, kTagLayout);   // j is even
      const float x0 = __fadd_rn(lo_x, __fmul_rn(span, u01(r.x))), y0 = __fadd_rn(lo_y, __fmul_rn(span, u01(r.y)));
      const float x1 = __fadd_rn(lo_x, __fmul_rn(span, u01(r.z))), y1 = __fadd_rn(lo_y, __fmul_rn(span, u01(r.w)));
      const float need_r = __fadd_rn(rk, keep), need_z = __fadd_rn(zk, keep);
      const float need_r2 = __fmul_rn(need_r, need_r), need_z2 = __fmul_rn(need_z, need_z);
      // both tries against object q with PACKED fp32 arithmetic (sub / mul / fma .f32x2: FADD2, FMUL2, FFMA2 in SASS,
      // the object's coordinate broadcast): 4 floating-point instructions per object for the two tries instead of 10;
      // d2 = fma(dy, dy, fl(dx dx)) per try -- the design twin (oracle/crl_oracle.c) forms it the same way
      const unsigned long long X2 = pack_f32x2(x0, x1), Y2 = pack_f32x2(y0, y1);
      uint32_t bad0 = 0u, bad1 = 0u;              // bit q: too close to object q (no branches)
#pragma unroll
      for (int q = 0; q < N; ++q) {
        const float2 o = placed[q];
        const float lim = q == 0 ? need_r2 : need_z2;
        const unsigned long long dx = sub_f32x2(X2, pack_f32x2(o.x, o.x)), dy = sub_f32x2(Y2, pack_f32x2(o.y, o.y));
        float d20, d21;
        unpack_f32x2(fma_f32x2(dy, dy, mul_f32x2(dx, dx)), d20, d21);
        bad0 |= (d20 >= lim) ? 0u : (1u << q);
        bad1 |= (d21 >= lim) ? 0u : (1u << q);
      }
      const uint32_t live = (1u << k) - 1u;       // objects >= k hold stale values
      const bool ok0 = (bad0 & live) == 0u, ok1 = !pinned && (bad1 & live) == 0u;
      if (ok0 || ok1) {
        const float x = ok0 ? x0 : x1, y = ok0 ? y0 : y1;
#pragma unroll
        for (int q = 0; q <= N; ++q) if (q == k) placed[q] = make_float2(x, y);
        ++k; j = 0;
      } else if ((j += 2) >= (pinned ? 1 : 100)) {   // 100 misses abandon the layout
        j = 0; k = 0;
        if (++attempt >= 10000u) k = N + 1;       // as the twin: give up with what there is
      }
      if (k > N) {
        const U4 rr = draw(layout_seed, 0u, 0u, 0u, kTagRot);
        float rot0 = __fmul_rn(6.2831855f, u01(rr.x));
        if (p.fixed) { const float4 f0 = p.fixed[0]; if (f0.w >= 2.f) rot0 = f0.z; }
        const size_t sb = (size_t)slot * p.B;
        const float2 rb = placed[0];
        float2* nz = p.next_zone_xy + sb * N + e;
#pragma unroll
        for (int i = 0; i < N; ++i) nz[(size_t)i * p.B] = placed[1 + i];
        p.next_origin[sb + e] = make_float4(rb.x, rb.y, rot0, 0.f);
        p.next_seed[sb + e] = layout_seed - 1;
        st_release_u32(p.next_ready + sb + e, done_state);
        have = false;
      }
    }
  }
}

// crl_prefetch_publish: the trusted epoch only grows (a late publish of an older round is a no-op)
__global__ void publish_epoch_kernel(uint32_t* epoch, uint32_t round) {
  if (*epoch < round) *epoch = round;
}

template <int TASK, int N>
__global__ void __maxnreg__(64) prefetch_task_kernel(const __grid_constant__ KParams p, const WorkItem* work) {
  const WorkHeader* hdr = reinterpret_cast<const WorkHeader*>(work);
  const uint32_t count = hdr->count;
  const int lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  const uint32_t half = lane >> 4, zone = lane & 15;
  constexpr int T = TASK == CRL_TASK_TTSP ? (N + 1) / 2 : 1;
  for (uint32_t pair = warp; 2u * pair < count; pair += n_warps) {
    const uint32_t idx = 2u * pair + half;
    const bool live = idx < count;
    WorkItem it{-1, 0u, 0};
    if (live) it = work[1u + idx];
    const size_t sb = (size_t)it.slot * p.B;
    uint32_t my_draw = 0u;
    if (live && zone < N) {                       // task draws use the seed BEFORE the increment
      if (TASK == CRL_TASK_TTSP) {
        const double ga = gamma_draw(it.seed, p.beta_a, zone, 0u);
        const double gb = gamma_draw(it.seed, p.beta_b, zone, 1u);
        const int t = (int)((ga / (ga + gb)) * (double)p.num_steps);
        my_draw = (uint32_t)min(max(t, 0), 65535);
      } else {
        my_draw = colour_draw(it.seed, zone);
      }
    }
    if (TASK == CRL_TASK_TTSP) {
      const uint32_t hi = __shfl_down_sync(kFull, my_draw, 1);
      if (live && zone < N && !(zone & 1))
        p.next_task[(sb * T) + (size_t)(zone >> 1) * p.B + it.e] = my_draw | (zone + 1 < N ? hi << 16 : 0u);
    } else {
      uint32_t cw = zone < N ? my_draw << (2 * zone) : 0u;
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) cw |= __shfl_xor_sync(kFull, cw, o);   // within the half-warp
      if (live && zone == 0) p.next_task[sb + it.e] = cw;
    }
    __threadfence();
    __syncwarp();
    if (live && zone == 0) st_release_u32(p.next_ready + sb + it.e, kSlotReady + p.round);
  }
}

// ---- observation and store: shared by step, reset and reset_from_layout -------
template <int TASK, int N>
__device__ __forceinline__ void zone_row(const KParams& p, const Env<N>& env, float* row) {
  constexpr int Z = ZoneDim<TASK>::Z;
  const float third = 1.0f / 3.0f;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float r, g, b;
    if (TASK == CRL_TASK_CM) {
      const uint32_t c = (env.hi >> (2 * i)) & 3u;   // 0 B, 1 G, 2 R (ZoneEnvBase.py:68-77)
      r = c == 2u ? 1.f : 0.f; g = c == 1u ? 1.f : 0.f; b = c == 0u ? 1.f : 0.f;
    } else {
      const bool v = (env.hi >> i) & 1u;             // Yellow (1,1,0) / Cyan (0,1,1), TSP_env.py:9-10
      r = v ? 1.f : 0.f; g = 1.f; b = v ? 0.f : 1.f;
    }
    float* z = row + i * Z;
    if (Z == 6) {
      reinterpret_cast<float2*>(z)[0] = make_float2(env.zone[i].x * third, env.zone[i].y * third);
      reinterpret_cast<float2*>(z)[1] = make_float2(r, g);
      reinterpret_cast<float2*>(z)[2] = make_float2(b, 0.25f);
    } else {
      z[0] = env.zone[i].x * third; z[1] = env.zone[i].y * third;
      z[2] = r; z[3] = g; z[4] = b; z[5] = 0.25f;
      if (TASK == CRL_TASK_TTSP) {
        const bool v = (env.hi >> i) & 1u;
        const int tm = (int)((env.tmax[i >> 1] >> (16 * (i & 1))) & 0xffffu);
        // TTSP_env.py:23-27: (zone_max_steps - steps) / max_steps in fp64, visited -> 1; its
        // float32 cast equals the correctly rounded float32 quotient (double rounding of a
        // quotient of two small integers is innocuous: 53 >= 2*24 + 2)
        z[6] = v ? 1.0f : div_const((float)(tm - env.steps), p.div_steps);
      } else {
        // colour_match_env.py:79: np.float32(cooldown) / 150 is a float32 division
        z[6] = div_const((float)cd_get(env.cd, i), p.div_cd);
      }
    }
  }
}

// Stage this warp's 32 zone_obs rows in shared memory and send them: the rows are one
// contiguous span of zone_obs, so a single cp.async.bulk moves them.  Everything a row
// holds (zone centres, colours, time left, cooldowns) is known BEFORE the physics, so
// the copy is issued early and drains while the warp integrates; zone_obs_wait() must
// run before the CTA exits (the copy reads shared memory asynchronously).
template <int TASK, int N>
__device__ __forceinline__ void zone_obs_issue(const KParams& p, float* stage, int lane, int env0, int max_rows) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  const int n_valid = max(0, min(max_rows, p.B - env0));
  const uint32_t bytes = (uint32_t)n_valid * ROW * 4u;
  float* gdst = p.zone_obs + (size_t)env0 * ROW;
  if ((bytes & 15u) == 0u) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0 && n_valid > 0) {
      const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(stage);
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                   :: "l"(gdst), "r"(saddr), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  } else {   // ragged tail whose byte count is not a multiple of 16: plain coalesced stores
    __syncwarp();
    for (int i = lane; i < n_valid * ROW; i += 32) gdst[i] = stage[i];
  }
}

template <int TASK, int N>
__device__ __forceinline__ void zone_obs_send(const KParams& p, const Env<N>& env, bool valid,
                                              float* stage, int lane, int warp_env0, bool zero_row = false) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  if (valid) zone_row<TASK, N>(p, env, stage + lane * ROW);
  if (zero_row) {                                  // WaitWrapper.noop_obs (wrappers.py:46-50)
    for (int k = 0; k < ROW; ++k) stage[lane * ROW + k] = 0.f;
  }
  zone_obs_issue<TASK, N>(p, stage, lane, warp_env0, 32);
}

// The rows of `mask`'s lanes (the envs whose zone_obs row this step changed) from the warp's stage into `out`, each
// row by the whole warp with coalesced stores.  A handful of rows per launch.  Host-direct step (crl_host_call_step):
// `out` is the caller's host mirror of zone_obs (pinned, device-mapped), which so stays a byte-exact copy of the device
// one.  CRL_STEP_ZONE_OBS_DELTA: `out` is the device zone_obs itself.
// CRL_STEP_HOST_PLANES (TimedTSP, host mirror only): the host mirror is PLANE-major, float[Z][B][N] (the caller views
// it as (B, N, Z) through strides), so that the one column that moves every step -- time left, plane 6 -- is a
// contiguous [B][N] array: the warp writes its 32 x N values of it with fully coalesced stores, every step; a changed
// row (a visit, a reset) is N values in each of the other planes.
template <int TASK, int N>
__device__ __noinline__ void send_rows(const KParams& p, float* out, const float* stage, unsigned mask, int lane,
                                       int warp_env0) {
  constexpr int Z = ZoneDim<TASK>::Z, ROW = N * Z;
  if (TASK == CRL_TASK_TTSP && (p.flags & CRL_STEP_HOST_PLANES)) {
    const size_t plane = (size_t)p.B * N;
    const int n_valid = max(0, min(32, p.B - warp_env0));
    float* tl = out + 6 * plane + (size_t)warp_env0 * N;
    for (int i = lane; i < n_valid * N; i += 32) tl[i] = stage[(i / N) * ROW + (i % N) * Z + 6];
    while (mask) {
      const int src = __ffs(mask) - 1;
      mask &= mask - 1u;
      const float* row = stage + src * ROW;
      float* dst = out + (size_t)(warp_env0 + src) * N;
      for (int i = lane; i < 6 * N; i += 32) dst[(size_t)(i / N) * plane + (i % N)] = row[(i % N) * Z + (i / N)];
    }
    return;
  }
  while (mask) {
    const int src = __ffs(mask) - 1;
    mask &= mask - 1u;
    float* dst = out + (size_t)(warp_env0 + src) * ROW;
    const float* row = stage + src * ROW;
    for (int i = lane; i < ROW; i += 32) dst[i] = row[i];
  }
}

// zone_obs of the plain step: the warp's rows are staged and leave with one bulk copy.  CRL_STEP_ZONE_OBS_DELTA: only
// the lanes in `changed` (the warp's mask of rows this step changes) build their row; every other row of p.zone_obs
// already holds what this step would write, and a warp whose valid rows all change (every TimedTSP step) still sends
// its span with the one bulk copy.  Returns true when the bulk copy went out; otherwise the staged rows are left for
// send_rows.  One zone_row for both ways: a second inlined copy reloads the spilled parts of `env` a second time.
template <int TASK, int N>
__device__ __forceinline__ bool zone_obs_step(const KParams& p, const Env<N>& env, float* stage, int lane, int warp_env0,
                                              unsigned changed) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  const int n_valid = max(0, min(32, p.B - warp_env0));
  const unsigned all = n_valid >= 32 ? kFull : (1u << n_valid) - 1u;
  const unsigned m = (p.flags & CRL_STEP_ZONE_OBS_DELTA) ? changed : all;
  if ((m >> lane) & 1u) zone_row<TASK, N>(p, env, stage + lane * ROW);
  if (m != all) return false;
  zone_obs_issue<TASK, N>(p, stage, lane, warp_env0, 32);
  return true;
}

__device__ __forceinline__ void zone_obs_wait(int lane) {
  if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// State planes and the 8-float obs row (ZoneEnvBase.py:190-192, 220-224; order fixed by
// wrappers.py:136-142).  remaining = 1 - steps/num_steps: the reference's fp64 value cast
// to float32 equals the correctly rounded float32 quotient (num_steps - steps)/num_steps
// (the exact value is k/num_steps, never within 2^-53 of a float32 rounding boundary
// unless it is one), so one IEEE float division reproduces it bit for bit.
// `park`: the stored step count becomes the parked sentinel (CRL_STEP_WAIT); the observation
// still shows the real count.
constexpr int kParkedSteps = 0xffff;
__device__ void obs_rows_bulk(float4* obs, int B, float4 row0, float4 row1, bool valid, float* stage, int lane, int warp_env0);

template <int TASK, int N>
__device__ __forceinline__ void store_state_obs(const KParams& p, const Env<N>& env, int e, float c, float s,
                                                bool park = false) {
  p.pose[e] = make_float4(env.b.X, env.b.Y, env.b.phi, env.b.vx);
  p.aux[e] = make_float4(env.b.vy, env.b.w, env.ep_return,
                         __int_as_float((int)((uint32_t)(park ? kParkedSteps : env.steps) | (env.hi << 16))));
  if (TASK == CRL_TASK_CM) p.cooldown[e] = env.cd;
  const float remaining = div_const((float)(p.num_steps - env.steps), p.div_steps);
  p.obs[2 * (size_t)e] = make_float4(remaining, env.b.X * (1.0f / 3.0f), env.b.Y * (1.0f / 3.0f), c);
  p.obs[2 * (size_t)e + 1] = make_float4(s, env.b.vx * (1.0f / 1.5f), env.b.vy * (1.0f / 1.5f),
                                         env.b.w * (1.0f / 3.0f));
}

// the same with the obs rows leaving through obs_rows_bulk (host-direct steps); every lane of the warp calls it
template <int TASK, int N>
__device__ __forceinline__ void store_state_obs_host(const KParams& p, const Env<N>& env, bool valid, int e, float c, float s,
                                                     float* stage, int lane, int warp_env0) {
  if (valid) {
    p.pose[e] = make_float4(env.b.X, env.b.Y, env.b.phi, env.b.vx);
    p.aux[e] = make_float4(env.b.vy, env.b.w, env.ep_return, __int_as_float((int)((uint32_t)env.steps | (env.hi << 16))));
    if (TASK == CRL_TASK_CM) p.cooldown[e] = env.cd;
  }
  const float remaining = div_const((float)(p.num_steps - env.steps), p.div_steps);
  obs_rows_bulk(p.obs, p.B, make_float4(remaining, env.b.X * (1.0f / 3.0f), env.b.Y * (1.0f / 3.0f), c),
                make_float4(s, env.b.vx * (1.0f / 1.5f), env.b.vy * (1.0f / 1.5f), env.b.w * (1.0f / 3.0f)), valid, stage, lane,
                warp_env0);
}

// Host-direct step: p.obs is host memory.  The warp's 32 obs rows (1 KB, contiguous) leave as ONE bulk
// copy through the zone_obs stage (long drained by now) instead of 64 half-line stores: full-size PCIe writes.
// Takes the row by value: a reference to the caller's Env would put the whole Env into local memory.
__device__ __noinline__ void obs_rows_bulk(float4* obs, int B, float4 row0, float4 row1, bool valid, float* stage, int lane,
                                           int warp_env0) {
  if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the zone_obs copy has read the stage
  __syncwarp();
  if (valid) {
    float4* row = reinterpret_cast<float4*>(stage) + 2 * lane;
    row[0] = row0;
    row[1] = row1;
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  const int n_valid = max(0, min(32, B - warp_env0));
  if (lane == 0 && n_valid > 0) {
    const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(stage);
    float4* gdst = obs + 2 * (size_t)warp_env0;
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(saddr), "r"((uint32_t)n_valid * 32u) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  }
}

template <int TASK, int N>
__device__ __forceinline__ void load_env(const KParams& p, int e, Env<N>& env) {
  const float4 ps = p.pose[e];
  const float4 ax = p.aux[e];
#pragma unroll
  for (int i = 0; i < N; ++i) env.zone[i] = p.zone_xy[(size_t)i * p.B + e];
  if (TASK == CRL_TASK_TTSP) {
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) env.tmax[j] = p.zone_tmax[(size_t)j * p.B + e];
  }
  if (TASK == CRL_TASK_CM) env.cd = p.cooldown[e];
  env.b.X = ps.x; env.b.Y = ps.y; env.b.phi = ps.z; env.b.vx = ps.w;
  env.b.vy = ax.x; env.b.w = ax.y; env.ep_return = ax.z;
  const uint32_t bits = (uint32_t)__float_as_int(ax.w);
  env.steps = (int)(bits & 0xffffu);
  env.hi = bits >> 16;
}

// np.sqrt(np.sum(np.square(goal_pos - robot_pos))) in fp64, no fused multiply-add
// (TSP_next_city_env.py:38-42 dist_to_goal).
__device__ __forceinline__ double dist_np(float X, float Y, float zx, float zy) {
  const double dx = (double)zx - (double)X, dy = (double)zy - (double)Y;
  return __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

// ---- chained steps (CRL_STEP_CHAINED) ------------------------------------------------
// stamp[0][w] = steps started, stamp[1][w] = steps finished for envs [32 w, 32 w + 32).
// Every step takes a ticket t = started++ BEFORE it lets dependents launch, so tickets
// follow launch order; a chained step's warp then spins until finished == t, i.e. until
// its own previous step is done, instead of waiting for the whole preceding grid.  All
// CTAs of the preceding grid are resident before this grid may start (the trigger is
// their first instruction), so the wait cannot deadlock; the spin is bounded anyway.
__device__ __forceinline__ uint32_t chain_ticket(const KParams& p, int w, int lane) {
  uint32_t t = 0u;
  if (lane == 0 && w < (p.B + 31) / 32) t = atomicAdd(p.stamp + w, 1u);
  return t;
}

__device__ __forceinline__ void chain_wait(const KParams& p, int w, int lane, uint32_t ticket) {
  if (lane == 0 && w < (p.B + 31) / 32) {
    const uint32_t* fin = p.stamp + (p.B + 31) / 32 + w;
    uint32_t polls = 0;
    while (ld_acquire_u32(fin) != ticket) {
      __nanosleep(64);
      if (++polls > (1u << 22)) { atomicAdd(p.counters + 7, 1.0); break; }
    }
  }
  __syncwarp();
}

// Publish this warp's step: every lane's stores are ordered before lane 0 by the warp
// barrier, the bulk copy is waited for to completion, then one release store.
__device__ __forceinline__ void chain_release(const KParams& p, int w, int lane, uint32_t ticket) {
  __syncwarp();
  if (lane == 0) {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    // st.release is itself the fence (cumulative over the lanes' stores the warp barrier
    // ordered before it); a __threadfence() in front of it would make the warp sit through two
    if (w < (p.B + 31) / 32) st_release_u32(p.stamp + (p.B + 31) / 32 + w, ticket + 1u);
  }
}

// ---- the fused step ---------------------------------------------------------------
// Order inside the kernel.  Everything the reference decides in a step except the
// physics state itself depends only on the PRE-physics position and the counters
// (SURVEY.md Appendix B), so the task logic, the result word, the auto-reset and the
// whole zone_obs row come first and the bulk copy of zone_obs is in flight while the
// frameskip substeps run; state and the 8-float obs row are written last.
// EXT = true: the variant that also serves the goal-conditioned tasks (CRL_STEP_GOALS) and
// WaitWrapper semantics (CRL_STEP_WAIT); the plain rollout kernel carries none of it.
template <int TASK, int N, bool EXT, bool FIXED = false>
__global__ void __maxnreg__(MaxRegs<N>::v) step_kernel(const __grid_constant__ KParams p) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  extern __shared__ __align__(128) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * kThreads + threadIdx.x;
  const int warp_env0 = blockIdx.x * kThreads + warp * 32;
  const bool valid = e < p.B;
  float* stage = smem + warp * (32 * ROW);
  // Programmatic dependent launch: this grid may be scheduled while the previous kernel
  // of the stream is still draining; let the next one do the same, then wait here until
  // everything the previous kernel wrote (state, actions) is visible.
  uint32_t ticket = 0u;
  const bool ticketed = (p.flags & (CRL_STEP_CHAINED | CRL_STEP_CHAIN_START)) != 0u;
  if (ticketed) {
    // the ticket must be taken before dependents may launch: the operand makes the
    // trigger wait for the atomic's return
    ticket = chain_ticket(p, warp_env0 >> 5, lane);
    asm volatile("griddepcontrol.launch_dependents;" :: "r"(ticket) : "memory");
  } else {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  }
  if (p.flags & CRL_STEP_CHAINED) {
    // back-to-back steps: wait only for THIS warp's own previous step, not for the whole
    // preceding grid; the tail of one launch overlaps the head of the next
    chain_wait(p, warp_env0 >> 5, lane, ticket);
  } else {
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }

  // CRL_STEP_ACTION_COUNTER: the step index of the in-kernel action draw is step_index + the number of
  // such steps this group of 32 envs has taken (a device counter), so that a captured launch that
  // is REPLAYED still draws fresh iid actions at every replay.  Plain read-modify-write by lane 0:
  // steps of the same envs are ordered (whole-grid or chained wait above).  The load is ISSUED first
  // (the previous step wrote the word: an L2 hit) and CONSUMED behind the state loads: issued behind
  // them it returns behind them, and the shuffle then holds the warp until the last plane is in
  // (+19 % per launch at 65,536 PointTSP envs, profiles/r02_notes.md).
  uint32_t act_base = 0u;
  uint32_t* act_cnt = nullptr;
  if (!p.actions && (p.flags & CRL_STEP_ACTION_COUNTER) && lane == 0 && warp_env0 < p.B) {
    act_cnt = p.act_count + (warp_env0 >> 5);
    act_base = ld_relaxed_u32(act_cnt);
  }
  Env<N> env;
  float2 act = make_float2(0.f, 0.f);
  if (valid) load_env<TASK, N>(p, e, env);
  if (!p.actions && (p.flags & CRL_STEP_ACTION_COUNTER)) {
    if (act_cnt) *act_cnt = act_base + 1u;
    act_base = __shfl_sync(kFull, act_base, 0);
  }
  if (valid) {
    if (p.actions) {
      act = p.actions[e];
    } else {
      const unsigned ge = (unsigned)(p.env_offset + e);
      const unsigned long long si = p.step_index + act_base;
      U4 ctr{ge, (uint32_t)si, (uint32_t)(si >> 32), kTagAction};
      const U4 r = philox4x32(ctr, (uint32_t)p.action_seed, (uint32_t)(p.action_seed >> 32));
      act = make_float2(2.f * u01(r.x) - 1.f, 2.f * u01(r.y) - 1.f);
    }
  } else {
    env.b = Body{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    env.ep_return = 0.f; env.steps = 0; env.hi = 0u; env.cd = make_uint2(0u, 0u);
#pragma unroll
    for (int i = 0; i < N; ++i) env.zone[i] = make_float2(1e9f, 1e9f);
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) env.tmax[j] = 0xffffffffu;
  }

  // WaitWrapper (wrappers.py:29-54): an env whose episode ended under CRL_STEP_WAIT is parked
  // (stored step count = sentinel); stepping it is a no-op that reports zeros and done.
  const bool parked = EXT && (p.flags & CRL_STEP_WAIT) && valid && env.steps == kParkedSteps;
  const bool live = valid && !parked;
  // a parked env under an AUTO-RESET step (hier_base.py: step_no_reset for skill_len - 1 steps, then
  // step): the worker's env.step is WaitWrapper's no-op (reward 0, done, info {}), and `if done:
  // obs = env.reset()` (penv.py:7-10) then restarts it -- the call returns the new episode's first
  // observation and counts nothing
  const bool revive = EXT && parked && (p.flags & CRL_STEP_AUTO_RESET);
  // goal-conditioned variants: the goal zone and the distance to it BEFORE the physics, which
  // is the reference's last_dist_to_goal (set by set_goal or left by the previous step, both
  // at the position this step starts from)
  const bool goals = EXT && (p.flags & CRL_STEP_GOALS);
  int goal_zone = -1;
  float gzx = 0.f, gzy = 0.f;
  double dist_before = 0.0;
  Body old_b = env.b;
  bool reached = false, park_now = false;
  if (goals && live) {
    goal_zone = p.goal[e];
    if (goal_zone >= 0) {
#pragma unroll
      for (int j = 0; j < N; ++j) if (j == goal_zone) { gzx = env.zone[j].x; gzy = env.zone[j].y; }
      dist_before = dist_np(env.b.X, env.b.Y, gzx, gzy);
    }
  }
  int fired_out = -1;
  // lanes whose zone_obs row changed, when only those rows are written (zone_obs_host, CRL_STEP_ZONE_OBS_DELTA):
  // parked in shared memory, not in a register that would be live across the whole task logic of the ordinary step.
  // A physics-only step changes no row.
  __shared__ unsigned s_rows_mask[kThreads / 32];
  const bool some_rows = p.zone_obs_host || (p.flags & CRL_STEP_ZONE_OBS_DELTA);
  if (some_rows && lane == 0) s_rows_mask[warp] = 0u;
  bool fresh = false;   // true: this env was rebuilt by the auto-reset, no physics this call
  if (!(p.flags & CRL_STEP_PHYSICS_ONLY)) {
    // does this step rewrite the env's zone_obs row with different bytes? (CRL_STEP_TRACK_ROWS, CRL_STEP_ZONE_OBS_DELTA)
    // TimedTSP's time-left column moves every step: the whole row counts as changed -- unless the host mirror is
    // plane-major (CRL_STEP_HOST_PLANES), where that column is shipped as its own contiguous plane every step
    bool row_changed = TASK == CRL_TASK_TTSP && !(p.flags & CRL_STEP_HOST_PLANES);
    // (1) ColourMatch cooldowns tick before anything else (colour_match_env.py:98-100)
    if (TASK == CRL_TASK_CM) {
      row_changed = (env.cd.x | env.cd.y) != 0u;
      env.cd.x = cd_dec4(env.cd.x); env.cd.y = cd_dec4(env.cd.y);
    }
    // (2) zone event on the pre-physics position: first eligible zone in index order.
    // fp32 screen of all N zones without branches; the (rare) candidates are confirmed
    // with the exact fp64 predicate, lowest index first.
    uint32_t cand = 0u;
#pragma unroll
    for (int i = 0; i < N; ++i)
      if (near_zone(env.b.X, env.b.Y, env.zone[i].x, env.zone[i].y, p.r2_guard)) cand |= 1u << i;
    if (TASK == CRL_TASK_CM) {
      if (cand) {                                  // rare: keep only zones whose cooldown is 0
#pragma unroll
        for (int i = 0; i < N; ++i) if (cd_get(env.cd, i) != 0u) cand &= ~(1u << i);
      }
    } else {
      cand &= ~env.hi;                             // not yet visited (TSP_env.py:58)
    }
    int fired = -1;
    while (cand) {
      const int i = __ffs(cand) - 1;
      cand &= cand - 1u;
      float zx = 0.f, zy = 0.f;
#pragma unroll
      for (int j = 0; j < N; ++j) if (j == i) { zx = env.zone[j].x; zy = env.zone[j].y; }
      if (inside_zone(env.b.X, env.b.Y, zx, zy, p.thresh2)) { fired = i; break; }
    }
    // (3) reward, goal, timeout: none of it reads the post-physics state
    int event = 0;
    if (fired >= 0) {
      if (TASK == CRL_TASK_CM) {
        const int old_dist = hamming(env.hi, N);
        const uint32_t col = (env.hi >> (2 * fired)) & 3u;
        const uint32_t nxt = col == 2u ? 0u : col + 1u;         // Blue -> Green -> Red -> Blue
        env.hi = (env.hi & ~(3u << (2 * fired))) | (nxt << (2 * fired));
        cd_set(env.cd, fired, (uint32_t)p.max_cd);
        event = old_dist - hamming(env.hi, N);                  // colour_match_env.py:86-93
      } else {
        env.hi |= 1u << fired;
        event = 1;
      }
    }
    bool goal;
    if (TASK == CRL_TASK_CM) {
      // goal_dist == 0 (colour_match_env.py:122-123)  <=>  all N zones share one colour
      constexpr uint32_t kOnes = ((1u << (2 * N)) - 1u) & 0x55555555u;
      const uint32_t col = env.hi & kHiMask;
      goal = col == 0u || col == kOnes || col == 2u * kOnes;
    } else {
      goal = (env.hi & kHiMask) == ((1u << N) - 1u);
    }
    bool done = false;
    float reward = (float)event;
    if (goal) {                                    // reward_goal, fp64 as the reference (TSP_env.py:37-39)
      reward = (float)((double)event + (double)(p.num_steps - env.steps) * p.bonus_per_step);
      done = true;
    }
    // a finished env that is stepped on without a reset (the reference asserts instead) must not
    // run its 16-bit step count into the parked sentinel or the visited / colour bits
    env.steps = min(env.steps + 1, kParkedSteps - 1);
    if (env.steps >= p.num_steps) done = true;
    if (TASK == CRL_TASK_TTSP && !done) {
      // TTSP_env.py:67: any unvisited zone with (zone_max_steps - steps) / max_steps <= 0
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const int tm = (int)((env.tmax[i >> 1] >> (16 * (i & 1))) & 0xffffu);
        if (!((env.hi >> i) & 1u) && env.steps >= tm) done = true;
      }
    }
    env.ep_return += reward;
    done = done && live;
    goal = goal && live;
    if (EXT) {
      fired_out = fired;
      reached = goals && fired >= 0 && fired == goal_zone;
      park_now = (p.flags & CRL_STEP_WAIT) && done && !(p.flags & CRL_STEP_AUTO_RESET);
      if (parked) { reward = 0.f; event = 0; }
    }
    if (p.flags & (CRL_STEP_TRACK_ROWS | CRL_STEP_ZONE_OBS_DELTA)) {
      // a finished env's row changes too, if it is rebuilt below
      const bool ch = (live && (row_changed || fired >= 0 || (done && (p.flags & CRL_STEP_AUTO_RESET)))) || parked;
      const unsigned cm = __ballot_sync(kFull, ch);
      // the rows themselves are written below: to the host mirror, or only these rows of the device zone_obs
      if (some_rows && lane == 0) s_rows_mask[warp] = cm;
      if ((p.flags & CRL_STEP_TRACK_ROWS) && cm && lane == 0) atomicAdd(p.row_list, __popc(cm));
    }
    // (4) result word and episode statistics
    bool res_moved = false;
    if (valid) {
      // need_next_goal (TSP_next_city_env.py:69-75, TTSP_next_city_env.py:49-53): the goal zone
      // was reached, or the episode ended (timeouts included), or there is no goal to pursue
      const bool need_next = goals && live && (reached || done || goal_zone < 0);
      const unsigned long long word = (unsigned long long)__float_as_uint(reward) |
          ((unsigned long long)((done || parked) ? 1u : 0u) << 32) | ((unsigned long long)(goal ? 1u : 0u) << 40) |
          ((unsigned long long)(uint8_t)(int8_t)event << 48) | ((unsigned long long)(need_next ? 1u : 0u) << 56);
      if (p.result_dev) {
        // host-direct step: `result` is the caller's host array, which holds what the device copy holds.  A record is
        // all zeros except on an event, a done or a goal change, so it crosses the link only when it differs from the
        // one already there (0.5 of the 2.6 MB a 65,536-env call wrote; the link is what bounds that call)
        const unsigned long long prev = p.result_dev[e];
        p.result_dev[e] = word;
        if (prev != word) { p.result[e] = word; res_moved = true; }
      } else {
        p.result[e] = word;
      }
      if (EXT && goals && live && need_next && goal_zone >= 0) p.goal[e] = -1;
    }
    if (p.result_dev) {                            // records moved, cumulative: row_list[1]
      const unsigned mm = __ballot_sync(kFull, res_moved);
      if (mm && lane == 0) atomicAdd(p.row_list + 1, (uint32_t)__popc(mm));
    }
    const unsigned dm = __ballot_sync(kFull, done);
    const unsigned rm = EXT ? __ballot_sync(kFull, done || revive) : dm;   // envs to rebuild
    if (rm) {
      float ret = done ? env.ep_return : 0.f;
      float len = done ? (float)env.steps : 0.f;
      const unsigned gm = __ballot_sync(kFull, goal);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        ret += __shfl_xor_sync(kFull, ret, o);
        len += __shfl_xor_sync(kFull, len, o);
      }
      if (lane == 0 && dm) {
        atomicAdd(p.counters + 0, (double)ret);
        atomicAdd(p.counters + 1, (double)__popc(dm));
        atomicAdd(p.counters + 2, (double)__popc(gm));
        atomicAdd(p.counters + 3, (double)len);
      }
      // (5) auto-reset, penv.py:9-10: only the finished envs are rebuilt
      if (p.flags & CRL_STEP_AUTO_RESET) {
        fresh = done || revive;
        // hot way: the parked layout, lane-local and inline (reset_from_slot)
        const uint32_t par_in = env.hi >> 15;
        bool served = false;
        if (fresh) served = reset_from_slot<TASK, N>(p, e, env);
        const unsigned sm = __ballot_sync(kFull, served);
        if (lane == 0 && sm) atomicAdd(p.counters + 4, (double)__popc(sm));
        // cold way (layout bank, slot not usable: inline sampling by the whole warp), out of line.
        // A copy crosses the call so that `env` itself is dead across it and stays in registers
        // everywhere else (keeping it live costs spills in the hot path)
        const unsigned left = rm & ~sm;
        if (left) {
          Env<N> next = env;
          warp_reset<TASK, N, FIXED>(p, left, lane, e, reinterpret_cast<float2*>(stage), par_in, next);
          env = next;
        }
      }
    }
  }
  float c, s;
  if (!EXT) {
    // (6) zone_obs leaves now and drains under the physics
    // (CRL_STEP_NO_ZONE_OBS: a consumer that builds the zone rows from the state planes itself --
    // crl_zone_encode_state -- needs neither the rows nor their 360 / 420 / 168 bytes per env-step)
    // Staged rows that still go out one by one, through ONE call site of send_rows (each costs spill reloads): the
    // changed rows of a CRL_STEP_ZONE_OBS_DELTA step into zone_obs, or those of a host-direct step into the host
    // mirror (never both, see step_launch)
    unsigned rows = 0u;
    if (some_rows) {
      __syncwarp();
      rows = s_rows_mask[warp];
    }
    if (!(p.flags & CRL_STEP_NO_ZONE_OBS) && zone_obs_step<TASK, N>(p, env, stage, lane, warp_env0, rows) && !p.zone_obs_host)
      rows = 0u;
    if (rows || p.zone_obs_host) {
      __syncwarp();
      send_rows<TASK, N>(p, p.zone_obs_host ? p.zone_obs_host : p.zone_obs, stage, rows, lane, warp_env0);
    }
    // (7) physics: all frameskip substeps in registers
    if (fresh) {
      sincosf(env.b.phi, &s, &c);
    } else {
      substeps(env.b, act.x, act.y, p.frameskip, c, s);
      env.b.phi = wrap_pi(env.b.phi);
    }
    if (p.zone_obs_host) {
      // host-direct step: p.obs is host memory; the warp's 32 obs rows leave as one bulk copy
      store_state_obs_host<TASK, N>(p, env, valid, e, c, s, stage, lane, warp_env0);
    } else if (valid) {
      store_state_obs<TASK, N>(p, env, e, c, s);
    }
  } else {
    if (!(p.flags & CRL_STEP_NO_ZONE_OBS))
      zone_obs_send<TASK, N>(p, env, live || revive, stage, lane, warp_env0, parked && !revive);
    if (p.zone_obs_host) send_rows<TASK, N>(p, p.zone_obs_host, stage, s_rows_mask[warp], lane, warp_env0);
    // an env rebuilt by the auto-reset still integrates its OLD body: the shaped reward of the
    // episode's last step is measured at the post-physics position (TSP_next_city_env.py:57-67)
    Body pb = fresh ? old_b : env.b;
    if (p.walled) substeps<CRL_CONTACT_MODEL, true>(pb, act.x, act.y, p.frameskip, c, s, p.extent);   // ZoneEnvBase.py:55-62
    else substeps(pb, act.x, act.y, p.frameskip, c, s);
    if (fresh) {
      sincosf(env.b.phi, &s, &c);
    } else {
      env.b = pb;
      env.b.phi = wrap_pi(env.b.phi);
    }
    if (goals && live) {
      double shaped = 0.0;
      if (goal_zone >= 0 && !reached) {
        shaped = dist_before - dist_np(pb.X, pb.Y, gzx, gzy);
        // colour_match_next_city_env.py:125-127: a zone other than the goal changed colour
        if (TASK == CRL_TASK_CM && fired_out >= 0) shaped -= 1.0;
      }
      p.shaped[e] = (float)shaped;
    }
    if (parked && goals) p.shaped[e] = 0.f;
    if (parked && !revive) {
      p.obs[2 * (size_t)e] = make_float4(0.f, 0.f, 0.f, 0.f);
      p.obs[2 * (size_t)e + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else if (valid) {
      store_state_obs<TASK, N>(p, env, e, c, s, park_now);
    }
  }
  if (ticketed) {
    chain_release(p, warp_env0 >> 5, lane, ticket);
  } else {
    zone_obs_wait(lane);
  }
}

// Engine.reset on the device for masked envs.
template <int TASK, int N>
__global__ void __launch_bounds__(kThreads) reset_kernel(const __grid_constant__ KParams p) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  extern __shared__ __align__(128) float smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = blockIdx.x * kThreads + threadIdx.x;
  const int warp_env0 = blockIdx.x * kThreads + warp * 32;
  const bool valid = e < p.B;
  float* stage = smem + warp * (32 * ROW);
  Env<N> env;
  if (valid) load_env<TASK, N>(p, e, env);
  const bool want = valid && (p.mask == nullptr || p.mask[e] != 0);
  const unsigned m = __ballot_sync(kFull, want);
  if (m) warp_reset<TASK, N, true, true>(p, m, lane, e, reinterpret_cast<float2*>(stage), 0u, env);
  float c = 1.f, s = 0.f;
  if (valid) sincosf(env.b.phi, &s, &c);
  // the warp's 32 zone_obs rows leave as one bulk copy: rows of envs that were not reset are
  // rewritten from the state just loaded (a parked env's row of zeros becomes its real row)
  zone_obs_send<TASK, N>(p, env, valid, stage, lane, warp_env0);
  if (want) store_state_obs<TASK, N>(p, env, e, c, s);
  zone_obs_wait(lane);
}

// Host-supplied layouts: one thread per listed env.  Rows are written directly (this
// path serves equivalence tests, not throughput).
struct LayoutParams {
  const double* xy0; const double* rot0; const double* zone_xy;
  const int32_t* zone_max_steps; const int32_t* colours; const int32_t* env_ids; int n;
};

template <int TASK, int N>
__global__ void reset_from_layout_kernel(const KParams p, const LayoutParams L) {
  constexpr int ROW = N * ZoneDim<TASK>::Z;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.n) return;
  const int e = L.env_ids ? L.env_ids[i] : i;
  if (e < 0 || e >= p.B) return;
  Env<N> env;
  const float rot0 = (float)L.rot0[i];
  env.b = Body{(float)L.xy0[2 * i], (float)L.xy0[2 * i + 1], wrap_pi(rot0), 0.f, 0.f, 0.f};
  env.ep_return = 0.f; env.steps = 0; env.hi = TASK == CRL_TASK_CM ? 0u : p.init_hi; env.cd = make_uint2(0u, 0u);
#pragma unroll
  for (int j = 0; j < (N + 1) / 2; ++j) env.tmax[j] = 0u;
#pragma unroll
  for (int z = 0; z < N; ++z) {
    env.zone[z] = make_float2((float)L.zone_xy[((size_t)i * N + z) * 2], (float)L.zone_xy[((size_t)i * N + z) * 2 + 1]);
    p.zone_xy[(size_t)z * p.B + e] = env.zone[z];
    if (TASK == CRL_TASK_TTSP) {
      const uint32_t t = (uint32_t)min(max(L.zone_max_steps[(size_t)i * N + z], 0), 65535);
      env.tmax[z >> 1] |= t << (16 * (z & 1));
    }
    if (TASK == CRL_TASK_CM) env.hi |= ((uint32_t)L.colours[(size_t)i * N + z] & 3u) << (2 * z);
  }
  if (TASK == CRL_TASK_TTSP) {
#pragma unroll
    for (int j = 0; j < (N + 1) / 2; ++j) p.zone_tmax[(size_t)j * p.B + e] = env.tmax[j];
  }
  const uint32_t episode = p.episode[e] + 1u;
  p.episode[e] = episode;
  if (p.goal) p.goal[e] = -1;
  p.origin[e] = make_float4(env.b.X, env.b.Y, rot0, 0.f);
  p.pose[e] = make_float4(env.b.X, env.b.Y, env.b.phi, 0.f);
  p.aux[e] = make_float4(0.f, 0.f, 0.f, __int_as_float((int)((env.hi << 16) | ((episode & 1u) << 31))));
  if (TASK == CRL_TASK_CM) p.cooldown[e] = env.cd;
  float c, s;
  sincosf(env.b.phi, &s, &c);
  p.obs[2 * (size_t)e] = make_float4(1.0f, env.b.X * (1.0f / 3.0f), env.b.Y * (1.0f / 3.0f), c);
  p.obs[2 * (size_t)e + 1] = make_float4(s, 0.f, 0.f, 0.f);
  __align__(16) float row[ROW];
  zone_row<TASK, N>(p, env, row);
  float* g = p.zone_obs + (size_t)e * ROW;
#pragma unroll
  for (int k = 0; k < ROW; ++k) g[k] = row[k];
}

// qpos/qvel <-> world frame: world = xy0 + R(rot0) q_xy, heading = rot0 + q_theta.
__global__ void set_qpos_qvel_kernel(const KParams p, const double* qpos, const double* qvel,
                                     const int32_t* env_ids, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int e = env_ids ? env_ids[i] : i;
  if (e < 0 || e >= p.B) return;
  const float4 o = p.origin[e];
  const double c0 = cos((double)o.z), s0 = sin((double)o.z);
  const double x = qpos[3 * i], y = qpos[3 * i + 1], th = qpos[3 * i + 2];
  const double vx = qvel[3 * i], vy = qvel[3 * i + 1];
  double phi = fmod((double)o.z + th, 2.0 * kPi);
  if (phi > kPi) phi -= 2.0 * kPi;
  if (phi < -kPi) phi += 2.0 * kPi;
  float4 ps = p.pose[e], ax = p.aux[e];
  ps.x = (float)((double)o.x + c0 * x - s0 * y);
  ps.y = (float)((double)o.y + s0 * x + c0 * y);
  ps.z = (float)phi;
  ps.w = (float)(c0 * vx - s0 * vy);
  ax.x = (float)(s0 * vx + c0 * vy);
  ax.y = (float)qvel[3 * i + 2];
  p.pose[e] = ps;
  p.aux[e] = ax;
}

__global__ void get_qpos_qvel_kernel(const KParams p, double* qpos, double* qvel,
                                     const int32_t* env_ids, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int e = env_ids ? env_ids[i] : i;
  if (e < 0 || e >= p.B) return;
  const float4 o = p.origin[e];
  const float4 ps = p.pose[e], ax = p.aux[e];
  const double c0 = cos((double)o.z), s0 = sin((double)o.z);
  const double dx = (double)ps.x - (double)o.x, dy = (double)ps.y - (double)o.y;
  qpos[3 * i] = c0 * dx + s0 * dy;
  qpos[3 * i + 1] = -s0 * dx + c0 * dy;
  qpos[3 * i + 2] = (double)ps.z - (double)o.z;   // modulo 2 pi: the heading is kept wrapped
  qvel[3 * i] = c0 * (double)ps.w + s0 * (double)ax.x;
  qvel[3 * i + 1] = -s0 * (double)ps.w + c0 * (double)ax.x;
  qvel[3 * i + 2] = (double)ax.y;
}

// Goal RPCs of the goal-conditioned variants, batched (zone-goals penv.py:18-25, 75-99).
// set_goal (TSP_next_city_env.py:77-80, colour_match_next_city_env.py:135-138): goals[e] < 0
// leaves env e alone; an index out of range or (TSP/TimedTSP) an already visited zone is the
// reference's assertion failure: the goal stays unset and counters[6] counts it.
template <int TASK>
__global__ void set_goal_kernel(const KParams p, const int32_t* goals, int N) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  const int g = goals[e];
  if (g < 0) return;
  const uint32_t bits = (uint32_t)__float_as_int(p.aux[e].w);
  const bool ok = g < N && (TASK == CRL_TASK_CM || !((bits >> 16 >> g) & 1u));   // g < 15: never the parity bit
  if (ok) p.goal[e] = g; else atomicAdd(p.counters + 6, 1.0);
}

// needs_goal (goal_zone is None), get_goal (zone centre / 3; zeros when there is none) and
// get_available_goals (TSP: the unvisited zones; ColourMatch: all) for every env.
template <int TASK>
__global__ void goal_query_kernel(const KParams p, float2* goal_xy, uint8_t* needs, uint8_t* available, int N) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  const int g = p.goal[e];
  if (needs) needs[e] = g < 0 ? 1 : 0;
  if (goal_xy) {
    float2 z = make_float2(0.f, 0.f);
    if (g >= 0 && g < N) z = p.zone_xy[(size_t)g * p.B + e];
    goal_xy[e] = make_float2(z.x * (1.0f / 3.0f), z.y * (1.0f / 3.0f));
  }
  if (available) {
    const uint32_t bits = (uint32_t)__float_as_int(p.aux[e].w);
    for (int i = 0; i < N; ++i)
      available[(size_t)e * N + i] = (TASK == CRL_TASK_CM || !((bits >> 16 >> i) & 1u)) ? 1 : 0;
  }
}

// Generalised advantage estimation straight from the step's own result records
// (main/src/torch_ac/algos/base.py:195-205).  One thread per env walks its column of the
// [T+1][B] rollout backwards; every operation is a separate IEEE float32 operation in the order
// torch evaluates the reference's expressions, so the result is bit-identical to it.
__global__ void __launch_bounds__(128) gae_kernel(const unsigned long long* __restrict__ results,
                                                  const float* __restrict__ reward_override,
                                                  const float* __restrict__ values, const float* __restrict__ next_value,
                                                  float g, float gl, int T, int B, float* __restrict__ adv_out,
                                                  float* __restrict__ ret_out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  constexpr int U = 8;   // frames per batch of independent loads (the recurrence itself is serial)
  unsigned long long rec_next = results[(size_t)T * B + e];   // slot t+1 while frame t is processed
  float nm = ((rec_next >> 32) & 0xffu) ? 0.f : 1.f;          // the mask in force after the last step
  float nv = next_value[e], na = 0.f;
  for (int t0 = T - 1; t0 >= 0; t0 -= U) {
    unsigned long long rec[U];
    float val[U], ovr[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {                             // all loads of the batch in flight at once
      const int t = t0 - u;
      rec[u] = t >= 0 ? results[(size_t)t * B + e] : 0ull;    // slot t: outcome of step t-1, its done is masks[t]
      val[u] = t >= 0 ? values[(size_t)t * B + e] : 0.f;
      ovr[u] = (reward_override && t >= 0) ? reward_override[(size_t)(t + 1) * B + e] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int t = t0 - u;
      if (t < 0) break;
      const float reward = reward_override ? ovr[u] : __uint_as_float((uint32_t)rec_next);
      const float v = val[u];
      const float delta = __fsub_rn(__fadd_rn(reward, __fmul_rn(__fmul_rn(g, nv), nm)), v);
      const float a = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, na), nm));
      adv_out[(size_t)t * B + e] = a;
      if (ret_out) ret_out[(size_t)t * B + e] = __fadd_rn(v, a);
      rec_next = rec[u];
      nm = ((rec_next >> 32) & 0xffu) ? 0.f : 1.f;
      nv = v;
      na = a;
    }
  }
}

// Invariants of the state planes, counted per kind (crl_check_state): what a stray write or a
// broken reset would violate.  compute-sanitizer is not available on every pool; this is cheap
// enough to run after any rollout.
__global__ void check_state_kernel(const KParams p, int task, int N, unsigned long long* bad) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  const float4 ps = p.pose[e], ax = p.aux[e];
  const uint32_t bits = (uint32_t)__float_as_int(ax.w);
  const int steps = (int)(bits & 0xffffu);
  const uint32_t hi = (bits >> 16) & 0x7fffu;
  if ((bits >> 31) != (p.episode[e] & 1u)) atomicAdd(bad + 5, 1ull);   // slot parity out of step with the episode counter
  if (!(isfinite(ps.x) && isfinite(ps.y) && isfinite(ps.z) && isfinite(ps.w) && isfinite(ax.x) && isfinite(ax.y) &&
        isfinite(ax.z)))
    atomicAdd(bad + 0, 1ull);
  if (!(fabsf(ps.z) <= 3.1415935f)) atomicAdd(bad + 1, 1ull);                       // heading wrapped
  if (steps > p.num_steps && steps != kParkedSteps) atomicAdd(bad + 2, 1ull);
  const float lim = p.extent - p.zone_keepout + 1e-5f;
  bool zone_bad = false;
  for (int i = 0; i < N; ++i) {
    const float2 z = p.zone_xy[(size_t)i * p.B + e];
    const bool pinned = p.fixed && p.fixed[1 + i].w == 1.f;     // a fixed location may lie anywhere
    zone_bad |= !pinned && !(fabsf(z.x) <= lim && fabsf(z.y) <= lim);
  }
  if (zone_bad) atomicAdd(bad + 3, 1ull);
  bool hi_bad = false;
  if (task == CRL_TASK_CM) {
    for (int i = 0; i < 7; ++i) {
      const uint32_t c = (hi >> (2 * i)) & 3u;
      hi_bad |= i < N ? c == 3u : c != 0u;
    }
    const uint2 cd = p.cooldown[e];
    for (int i = 0; i < 8; ++i) hi_bad |= cd_get(cd, i) > (uint32_t)p.max_cd || (i >= N && cd_get(cd, i) != 0u);
  } else {
    hi_bad = (hi >> N) != 0u;
  }
  if (hi_bad) atomicAdd(bad + 4, 1ull);
  if (p.next_ready) {                             // 0 empty, 2 layout parked, 3 claimed, >= 16 ready (round r)
    const uint32_t f0 = p.next_ready[e], f1 = p.next_ready[(size_t)p.B + e];
    if (f0 == 1u || (f0 > 3u && f0 < kSlotReady) || f1 == 1u || (f1 > 3u && f1 < kSlotReady)) atomicAdd(bad + 5, 1ull);
  }
  if (p.goal && (p.goal[e] < -1 || p.goal[e] >= N)) atomicAdd(bad + 6, 1ull);
  if (task == CRL_TASK_TTSP) {
    bool t_bad = false;
    for (int i = 0; i < N; ++i) {
      const uint32_t tm = (p.zone_tmax[(size_t)(i >> 1) * p.B + e] >> (16 * (i & 1))) & 0xffffu;
      t_bad |= tm > (uint32_t)p.num_steps;
    }
    if (t_bad) atomicAdd(bad + 7, 1ull);
  }
}

// Rollout frames (crl_frame_capture): one thread per env writes the env's CrlFrame; the envs that start an episode (or
// all, `initial`) take a layout-table entry -- one atomic per warp -- and copy their zone centres (and timeouts) there.
struct CaptureParams {
  const float4* aux;
  const float2* zone_xy;
  const uint32_t* zone_tmax;
  const uint2* cooldown;
  const unsigned long long* result;   // CrlResult[B] of the step; NULL with `initial`
  uint4* frames;                      // CrlFrame[B] of this slot; frames - B: the previous slot
  float2* layout_xy;
  uint32_t* layout_tmax;
  uint32_t* fill;                     // entries handed out, entries requested
  uint32_t capacity;
  int B, N, initial;
};

__global__ void __launch_bounds__(256) frame_capture_kernel(const CaptureParams c) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  const bool live = e < c.B;
  const bool need = live && (c.initial || ((c.result[e] >> 32) & 0xffu) != 0ull);   // done
  const uint32_t ballot = __ballot_sync(kFull, need);
  uint32_t layout = CRL_FRAME_NO_LAYOUT;
  if (ballot) {
    const int leader = __ffs(ballot) - 1;
    uint32_t base = 0u;
    if (lane == leader) {
      base = atomicAdd(c.fill + 1, (uint32_t)__popc(ballot));
      const uint32_t end = base + (uint32_t)__popc(ballot);
      atomicMax(c.fill, end < c.capacity ? end : c.capacity);
    }
    base = __shfl_sync(kFull, base, leader);
    const uint32_t k = base + (uint32_t)__popc(ballot & ((1u << lane) - 1u));
    if (need && k < c.capacity) layout = k;
  }
  if (!live) return;
  if (!need) {
    layout = c.frames[e - (ptrdiff_t)c.B].y;                   // the episode goes on: the entry of the previous frame
  } else if (layout != CRL_FRAME_NO_LAYOUT) {
    for (int i = 0; i < c.N; ++i) c.layout_xy[(size_t)layout * c.N + i] = c.zone_xy[(size_t)i * c.B + e];
    if (c.layout_tmax) {
      const int nh = (c.N + 1) >> 1;
      for (int j = 0; j < nh; ++j) c.layout_tmax[(size_t)layout * nh + j] = c.zone_tmax[(size_t)j * c.B + e];
    }
  }
  const uint2 cd = c.cooldown ? c.cooldown[e] : make_uint2(0u, 0u);
  c.frames[e] = make_uint4((uint32_t)__float_as_int(c.aux[e].w), layout, cd.x, cd.y);
}

// Env copies (crl_copy_envs): pair i copies env src ids[i] onto env dst ids[i], plane by plane, bit for bit.  One side
// of the copy: its planes (NULL = not copied; the host made both sides agree) and its ids.
struct CopySide {
  float4* pose;
  float4* aux;
  float2* zone_xy;
  uint32_t* zone_tmax;
  uint2* cooldown;
  long long* seed;
  uint32_t* episode;
  float4* origin;
  int32_t* goal;
  float4* obs;
  float* zone_obs;
  unsigned long long* result;
  float* shaped;
  const int32_t* ids;   // NULL: pair i is env i
  int B;
};

struct CopyParams {
  CopySide dst, src;
  uint32_t* next_ready;   // dst's, or NULL
  uint32_t* rejected;     // pairs with an id out of range, or NULL
  int n;
};

// One thread per pair moves the 16-byte vectors, the scalars and the plane-major zone centres: a warp of consecutive
// dst ids writes whole 128-byte lines of every plane, and the gathered src reads of a branch (each src env read K times in
// a row) come from L2.  A warp's 32 zone_obs rows (N Z floats each, 4-byte aligned only) are one span of 32 N Z floats
// that lane j copies at j, j + 32, ...: consecutive dst rows are written at consecutive addresses.  Stores are streaming
// (st.global.cs): the dst is not read again here, the src may be.
template <int TASK, int N>
__global__ void __launch_bounds__(256) copy_envs_kernel(const __grid_constant__ CopyParams c) {
  constexpr int Z = ZoneDim<TASK>::Z, ROW = N * Z, NH = (N + 1) / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
  int s = -1, d = -1;
  bool bad = false;
  if (i < c.n) {
    s = c.src.ids ? c.src.ids[i] : i;
    d = c.dst.ids ? c.dst.ids[i] : i;
    if (s < 0 || s >= c.src.B || d < 0 || d >= c.dst.B) { bad = true; s = d = -1; }
  }
  if (c.rejected) {
    const uint32_t b = __ballot_sync(kFull, bad);
    if (b && lane == __ffs(b) - 1) atomicAdd(c.rejected, (uint32_t)__popc(b));
  }
  if (d >= 0) {
    const size_t Bs = c.src.B, Bd = c.dst.B;
    const float4 pose = c.src.pose[s], aux = c.src.aux[s], origin = c.src.origin[s];
    const long long seed = c.src.seed[s];
    const uint32_t episode = c.src.episode[s];
    float2 xy[N];
#pragma unroll
    for (int z = 0; z < N; ++z) xy[z] = c.src.zone_xy[z * Bs + s];
    uint32_t tmax[NH];
    if constexpr (TASK == CRL_TASK_TTSP) {
#pragma unroll
      for (int j = 0; j < NH; ++j) tmax[j] = c.src.zone_tmax[j * Bs + s];
    }
    uint2 cd;
    if constexpr (TASK == CRL_TASK_CM) cd = c.src.cooldown[s];
    const int32_t goal = c.src.goal ? c.src.goal[s] : 0;
    float4 o0, o1;
    if (c.src.obs) { o0 = c.src.obs[2 * (size_t)s]; o1 = c.src.obs[2 * (size_t)s + 1]; }
    const unsigned long long res = c.src.result ? c.src.result[s] : 0ull;
    const float shaped = c.src.shaped ? c.src.shaped[s] : 0.f;

    __stcs(c.dst.pose + d, pose);
    __stcs(c.dst.aux + d, aux);
    __stcs(c.dst.origin + d, origin);
    __stcs(c.dst.seed + d, seed);
    __stcs(c.dst.episode + d, episode);
#pragma unroll
    for (int z = 0; z < N; ++z) __stcs(c.dst.zone_xy + z * Bd + d, xy[z]);
    if constexpr (TASK == CRL_TASK_TTSP) {
#pragma unroll
      for (int j = 0; j < NH; ++j) __stcs(c.dst.zone_tmax + j * Bd + d, tmax[j]);
    }
    if constexpr (TASK == CRL_TASK_CM) __stcs(c.dst.cooldown + d, cd);
    if (c.dst.goal) __stcs(c.dst.goal + d, goal);
    if (c.dst.obs) { __stcs(c.dst.obs + 2 * (size_t)d, o0); __stcs(c.dst.obs + 2 * (size_t)d + 1, o1); }
    if (c.dst.result) __stcs(c.dst.result + d, res);
    if (c.dst.shaped) __stcs(c.dst.shaped + d, shaped);
    // the parked layouts were drawn for the old seed and episode: the next reset samples inline until a sampler round
    // refills the slots
    if (c.next_ready) { __stcs(c.next_ready + d, 0u); __stcs(c.next_ready + Bd + d, 0u); }
  }
  if (c.src.zone_obs) {
    // loads of U floats in flight per lane before their stores; the guard `f0 + 32 u < 32 ROW` is warp-uniform
    constexpr int U = 8;
    for (int f0 = 0; f0 < 32 * ROW; f0 += 32 * U) {
      float v[U];
      long long at[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        at[u] = -1;
        if (f0 + 32 * u < 32 * ROW) {
          const int f = f0 + 32 * u + lane, pr = f / ROW, k = f - pr * ROW;
          const int sp = __shfl_sync(kFull, s, pr), dp = __shfl_sync(kFull, d, pr);
          if (dp >= 0) {
            v[u] = c.src.zone_obs[(size_t)sp * ROW + k];
            at[u] = (long long)dp * ROW + k;
          }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (at[u] >= 0) __stcs(c.dst.zone_obs + at[u], v[u]);
    }
  }
}

// ---- host side ---------------------------------------------------------------------
static int zone_dim(int task) { return task == CRL_TASK_TSP ? 6 : 7; }

static int check_config(const CrlConfig* c) {
  if (!c) return CRL_ERR_NULL;
  if (c->task < 0 || c->task > 2) return CRL_ERR_CONFIG;
  if (c->num_envs <= 0 || c->num_zones <= 0 || c->num_zones > CRL_MAX_ZONES) return CRL_ERR_CONFIG;
  // bits 16-30 of the state word hold the visited mask / colour codes, bit 31 the episode parity
  if (c->task == CRL_TASK_CM ? c->num_zones > 7 : c->num_zones > 15) return CRL_ERR_CONFIG;
  if (c->num_steps <= 0 || c->num_steps > 65534) return CRL_ERR_CONFIG;   // 65535 = parked sentinel
  if (c->frameskip < 0 || c->max_cooldown < 0 || c->max_cooldown > 255) return CRL_ERR_CONFIG;
  if (c->seed_mode == CRL_SEED_FIXED_RANGE && c->max_seed < c->min_seed) return CRL_ERR_CONFIG;
  if (!(c->zone_size > 0.0)) return CRL_ERR_CONFIG;
  if (c->task != CRL_TASK_CM && (c->initial_visited >> c->num_zones) != 0u) return CRL_ERR_CONFIG;
  if (c->walled > 1u) return CRL_ERR_CONFIG;
  // walled: every placement stays keepout (>= 0.4) inside the extents, i.e. clear of the wall boxes of half-size 0.1
  if (c->walled && (c->robot_keepout < 0.2 || c->zone_keepout < 0.1)) return CRL_ERR_CONFIG;
  return CRL_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// DivConst for a divisor, proven once per distinct (divisor, numerator range) and cached.
static DivConst cached_div_const(int d, int n_lo, int n_hi) {
  struct Slot { int d, lo, hi; DivConst k; };
  static Slot slots[8];
  static int used = 0;
  for (int i = 0; i < used; ++i)
    if (slots[i].d == d && slots[i].lo == n_lo && slots[i].hi == n_hi) return slots[i].k;
  const DivConst k = make_div_const(d, n_lo, n_hi);
  if (used < 8) slots[used++] = Slot{d, n_lo, n_hi, k};
  return k;
}

static int fill_params(const CrlConfig* c, const CrlState* st, const CrlOut* out, KParams& p) {
  int rc = check_config(c);
  if (rc) return rc;
  if (!st || !st->pose || !st->aux || !st->zone_xy || !st->seed || !st->episode || !st->origin || !st->counters)
    return CRL_ERR_NULL;
  if (c->task == CRL_TASK_TTSP && !st->zone_tmax) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_CM && !st->cooldown) return CRL_ERR_NULL;
  if (!aligned16(st->pose) || !aligned16(st->aux) || !aligned16(st->zone_xy) || !aligned16(st->origin))
    return CRL_ERR_ALIGN;
  memset(&p, 0, sizeof(p));
  p.B = c->num_envs; p.num_steps = c->num_steps; p.frameskip = c->frameskip; p.max_cd = c->max_cooldown;
  p.seed_mode = c->seed_mode; p.env_offset = c->env_offset; p.min_seed = c->min_seed; p.max_seed = c->max_seed;
  p.thresh2 = sqrt_threshold(c->zone_size);
  p.r2_guard = (float)(c->zone_size * c->zone_size * 1.001 + 1e-5);
  p.bonus_per_step = c->time_saved_reward;
  p.beta_a = c->beta_a; p.beta_b = c->beta_b;
  // numerators: num_steps - steps and zone_max_steps - steps, both within +-65535
  p.div_steps = cached_div_const(c->num_steps, -65535, 65535);
  p.div_cd = cached_div_const(c->max_cooldown > 0 ? c->max_cooldown : 1, 0, 255);
  if (!p.div_steps.exact || !p.div_cd.exact) return CRL_ERR_CONFIG;   // never happens, see crl_core.cuh
  p.robot_keepout = (float)c->robot_keepout; p.zone_keepout = (float)c->zone_keepout; p.extent = (float)c->extent;
  p.pose = reinterpret_cast<float4*>(st->pose); p.aux = reinterpret_cast<float4*>(st->aux);
  p.zone_xy = reinterpret_cast<float2*>(st->zone_xy); p.zone_tmax = st->zone_tmax;
  p.cooldown = reinterpret_cast<uint2*>(st->cooldown);
  p.seed = reinterpret_cast<long long*>(st->seed); p.episode = st->episode;
  p.origin = reinterpret_cast<float4*>(st->origin); p.counters = st->counters;
  // optional prefetch planes: all present or none
  if (st->next_ready) {
    if (!st->next_zone_xy || !st->next_origin || !st->next_seed || (c->task != CRL_TASK_TSP && !st->next_task))
      return CRL_ERR_NULL;
    if (!aligned16(st->next_origin) || !aligned16(st->next_zone_xy)) return CRL_ERR_ALIGN;
    p.next_zone_xy = reinterpret_cast<float2*>(st->next_zone_xy); p.next_task = st->next_task;
    p.next_origin = reinterpret_cast<float4*>(st->next_origin);
    p.next_seed = reinterpret_cast<long long*>(st->next_seed); p.next_ready = st->next_ready;
  }
  if (st->fixed_layout) {
    if (!aligned16(st->fixed_layout)) return CRL_ERR_ALIGN;
    p.fixed = reinterpret_cast<const float4*>(st->fixed_layout);
  }
  p.init_hi = c->task == CRL_TASK_CM ? 0u : c->initial_visited;
  p.walled = c->walled;
  p.stamp = st->stamp;
  p.act_count = st->stamp ? st->stamp + 2 * (size_t)((c->num_envs + 31) / 32) : nullptr;
  p.epoch = st->prefetch_epoch;
  if (p.next_ready && !p.epoch) return CRL_ERR_NULL;
  p.row_list = st->row_list;
  p.goal = st->goal;
  if (st->bank_zone_xy || st->bank_origin || st->bank_task) {
    if (!st->bank_zone_xy || !st->bank_origin || (c->task != CRL_TASK_TSP && !st->bank_task)) return CRL_ERR_NULL;
    if (c->max_seed < c->min_seed) return CRL_ERR_CONFIG;              // the bank is indexed by seed - min_seed
    if (!aligned16(st->bank_origin) || (reinterpret_cast<uintptr_t>(st->bank_zone_xy) & 7u)) return CRL_ERR_ALIGN;
    p.bank_zone_xy = reinterpret_cast<const float2*>(st->bank_zone_xy);
    p.bank_origin = reinterpret_cast<const float4*>(st->bank_origin);
    p.bank_task = st->bank_task;
  }
  if (out) {
    if (!out->obs || !out->result) return CRL_ERR_NULL;     // zone_obs: checked by the callers that write it
    if (!aligned16(out->obs) || !aligned16(out->zone_obs)) return CRL_ERR_ALIGN;
    p.obs = reinterpret_cast<float4*>(out->obs); p.zone_obs = out->zone_obs;
    p.result = reinterpret_cast<unsigned long long*>(out->result);
    p.shaped = out->shaped_reward;
  }
  return CRL_OK;
}

static int launch_status() { return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH; }

// (task, N) pairs with compiled kernels
#define CRL_DISPATCH(task, n, CALL)                                              \
  do {                                                                           \
    if ((task) == CRL_TASK_TSP && (n) == 15) { CALL(CRL_TASK_TSP, 15); }         \
    else if ((task) == CRL_TASK_TSP && (n) == 5) { CALL(CRL_TASK_TSP, 5); }      \
    else if ((task) == CRL_TASK_TTSP && (n) == 15) { CALL(CRL_TASK_TTSP, 15); }  \
    else if ((task) == CRL_TASK_TTSP && (n) == 5) { CALL(CRL_TASK_TTSP, 5); }    \
    else if ((task) == CRL_TASK_CM && (n) == 6) { CALL(CRL_TASK_CM, 6); }        \
    else return CRL_ERR_UNSUPPORTED;                                             \
  } while (0)

// The step kernel of a configuration.  Fixed placements (CrlState.fixed_layout) have kernels for the
// 15-zone TSP only -- the hard instances PointTSP-v4 / v5 and their goal-conditioned flavours.
template <int T, int NN>
static void (*pick_step_kernel(bool ext, bool fixed))(const KParams) {
  if (fixed) {
    if constexpr (T == CRL_TASK_TSP && NN == 15) return ext ? step_kernel<T, NN, true, true> : step_kernel<T, NN, false, true>;
    else return nullptr;
  }
  return ext ? step_kernel<T, NN, true> : step_kernel<T, NN, false>;
}

// opt in to > 48 KB dynamic shared memory once per kernel
static int set_smem(void (*kernel)(const KParams), size_t bytes) {
  static void (*done_for[32])(const KParams) = {nullptr};
  if (bytes <= 48 * 1024) return CRL_OK;
  for (int i = 0; i < 32; ++i) {
    if (done_for[i] == kernel) return CRL_OK;
    if (done_for[i] == nullptr) {
      if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
        return CRL_ERR_DEVICE;
      done_for[i] = kernel;
      return CRL_OK;
    }
  }
  return CRL_ERR_DEVICE;
}

}  // namespace crl

using namespace crl;

extern "C" {

int crl_abi_version(void) { return CRL_ABI_VERSION; }

const char* crl_strerror(int code) {
  switch (code) {
    case CRL_OK: return "ok";
    case CRL_ERR_NULL: return "a required pointer is NULL";
    case CRL_ERR_CONFIG: return "CrlConfig out of range";
    case CRL_ERR_ALIGN: return "a float4 plane is not 16-byte aligned";
    case CRL_ERR_UNSUPPORTED: return "no kernel compiled for this (task, num_zones)";
    case CRL_ERR_LAUNCH: return "CUDA launch failed";
    case CRL_ERR_DEVICE: return "CUDA device/runtime error";
    default: return "unknown error";
  }
}

int crl_plane_bytes(const CrlConfig* c, int64_t* out_bytes, int32_t n) {
  int rc = check_config(c);
  if (rc) return rc;
  if (!out_bytes) return CRL_ERR_NULL;
  if (n < 0) return CRL_ERR_CONFIG;
  int64_t o[CRL_NUM_PLANES];
  const int64_t B = c->num_envs, N = c->num_zones, Z = zone_dim(c->task);
  o[0] = 16 * B; o[1] = 16 * B; o[2] = 8 * N * B;
  o[3] = c->task == CRL_TASK_TTSP ? 4 * ((N + 1) / 2) * B : 0;
  o[4] = c->task == CRL_TASK_CM ? 8 * B : 0;
  o[5] = 8 * B; o[6] = 4 * B; o[7] = 16 * B; o[8] = 8 * 8;
  o[9] = 2 * 8 * N * B;
  o[10] = 2 * (c->task == CRL_TASK_TTSP ? 4 * ((N + 1) / 2) * B : (c->task == CRL_TASK_CM ? 4 * B : 0));
  o[11] = 2 * 16 * B; o[12] = 2 * 8 * B; o[13] = 2 * 4 * B;
  o[14] = 32 * B; o[15] = 4 * N * Z * B; o[16] = 8 * B;
  o[17] = 3 * 4 * ((B + 31) / 32);
  o[18] = 16 * (1 + 2 * B);
  o[19] = 16;      /* row_list */
  o[20] = 4 * B;   /* goal */
  o[21] = 4 * B;   /* shaped_reward */
  o[22] = 16;      /* prefetch_epoch */
  for (int i = 0; i < n && i < CRL_NUM_PLANES; ++i) out_bytes[i] = o[i];
  return CRL_OK;
}

int crl_step_bytes(const CrlConfig* c, int64_t* rd, int64_t* wr) {
  int rc = check_config(c);
  if (rc) return rc;
  if (!rd || !wr) return CRL_ERR_NULL;
  const int64_t N = c->num_zones, Z = zone_dim(c->task);
  int64_t r = 8 /*action*/ + 32 /*pose+aux*/ + 8 * N, w = 32 + 8 /*result*/ + 32 /*obs*/ + 4 * N * Z;
  if (c->task == CRL_TASK_TTSP) r += 4 * ((N + 1) / 2);
  if (c->task == CRL_TASK_CM) { r += 8; w += 8; }
  *rd = r; *wr = w;
  return CRL_OK;
}

static int step_launch(const CrlConfig* c, const CrlState* st, const float* actions, const CrlOut* out,
                       uint32_t flags, uint64_t action_seed, uint64_t step_index, float* zone_obs_host, void* stream,
                       CrlResult* result_dev = nullptr) {
  KParams p;
  if (!out) return CRL_ERR_NULL;
  int rc = fill_params(c, st, out, p);
  if (rc) return rc;
  p.zone_obs_host = zone_obs_host;
  p.result_dev = reinterpret_cast<unsigned long long*>(result_dev);
  if (result_dev && (!zone_obs_host || !p.row_list)) return CRL_ERR_CONFIG;
  if (actions && (reinterpret_cast<uintptr_t>(actions) & 7u)) return CRL_ERR_ALIGN;
  p.actions = reinterpret_cast<const float2*>(actions);
  p.flags = flags; p.action_seed = action_seed; p.step_index = step_index;
  const bool ticketed = (flags & (CRL_STEP_CHAINED | CRL_STEP_CHAIN_START)) != 0u;
  if (ticketed && !p.stamp) return CRL_ERR_NULL;
  if ((flags & CRL_STEP_TRACK_ROWS) && !p.row_list) return CRL_ERR_NULL;
  if ((flags & CRL_STEP_GOALS) && (!p.goal || !p.shaped)) return CRL_ERR_NULL;
  if ((flags & CRL_STEP_ACTION_COUNTER) && !p.act_count) return CRL_ERR_NULL;
  if (!(flags & CRL_STEP_NO_ZONE_OBS) && !p.zone_obs) return CRL_ERR_NULL;
  if ((flags & CRL_STEP_NO_ZONE_OBS) && (zone_obs_host || (flags & CRL_STEP_TRACK_ROWS))) return CRL_ERR_CONFIG;
  if ((flags & CRL_STEP_HOST_PLANES) && (!zone_obs_host || c->task != CRL_TASK_TTSP)) return CRL_ERR_CONFIG;
  // the walls live in the EXT kernels only (the plain rollout kernels keep their register allocation)
  const bool ext = (flags & (CRL_STEP_GOALS | CRL_STEP_WAIT)) != 0u || c->walled != 0u;
  if ((flags & CRL_STEP_ZONE_OBS_DELTA) && (ext || zone_obs_host || (flags & CRL_STEP_NO_ZONE_OBS))) return CRL_ERR_CONFIG;
  // every TimedTSP row changes every step (time left): the flag would only add the per-row predicate to the step
  if (c->task == CRL_TASK_TTSP) p.flags &= ~CRL_STEP_ZONE_OBS_DELTA;
  // Programmatic launch (this grid may start while its predecessor drains) is safe when the
  // kernel then waits for the whole predecessor (plain, chain start) or for its own previous
  // step (chained).  After a CHAINED launch, though, "the predecessor is complete" no longer
  // implies that everything before it is: a step that is not itself chained is then launched
  // without the attribute, i.e. with full stream ordering.
  static std::atomic<void*> last_chained_stream{reinterpret_cast<void*>(-1)};
  const bool after_chained = last_chained_stream.load(std::memory_order_relaxed) == stream;
  const bool programmatic = (flags & CRL_STEP_CHAINED) || !after_chained;
  last_chained_stream.store((flags & CRL_STEP_CHAINED) ? stream : reinterpret_cast<void*>(-1), std::memory_order_relaxed);
  const int blocks = (p.B + kThreads - 1) / kThreads;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CRL_CALL_STEP(T, NN)                                                        \
  {                                                                                 \
    const size_t sm = (size_t)kThreads * NN * ZoneDim<T>::Z * 4;                    \
    void (*kern)(const KParams) = pick_step_kernel<T, NN>(ext, p.fixed != nullptr); \
    if (!kern) return CRL_ERR_UNSUPPORTED;                                          \
    rc = set_smem(kern, sm);                                                        \
    if (rc) return rc;                                                              \
    cudaLaunchConfig_t lc = {};                                                     \
    lc.gridDim = dim3(blocks); lc.blockDim = dim3(kThreads);                        \
    lc.dynamicSmemBytes = sm; lc.stream = s;                                        \
    cudaLaunchAttribute at[1];                                                      \
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                  \
    at[0].val.programmaticStreamSerializationAllowed = 1;                           \
    lc.attrs = at; lc.numAttrs = programmatic ? 1 : 0;                              \
    if (cudaLaunchKernelEx(&lc, kern, p) != cudaSuccess) {                          \
      (void)cudaGetLastError();                                                     \
      return CRL_ERR_LAUNCH;                                                        \
    }                                                                               \
  }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_STEP);
  return launch_status();
}

int crl_step(const CrlConfig* c, const CrlState* st, const float* actions, const CrlOut* out,
             uint32_t flags, uint64_t action_seed, uint64_t step_index, void* stream) {
  return step_launch(c, st, actions, out, flags, action_seed, step_index, nullptr, stream);
}

int crl_reset(const CrlConfig* c, const CrlState* st, const CrlOut* out, const uint8_t* mask, void* stream) {
  KParams p;
  if (!out || !out->zone_obs) return CRL_ERR_NULL;
  int rc = fill_params(c, st, out, p);
  if (rc) return rc;
  p.mask = mask;
  const int blocks = (p.B + kThreads - 1) / kThreads;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CRL_CALL_RESET(T, NN)                                                       \
  {                                                                                 \
    const size_t sm = (size_t)kThreads * NN * ZoneDim<T>::Z * 4;                    \
    rc = set_smem(reset_kernel<T, NN>, sm);                                         \
    if (rc) return rc;                                                              \
    reset_kernel<T, NN><<<blocks, kThreads, sm, s>>>(p);                            \
  }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_RESET);
  return launch_status();
}

int crl_reset_from_layout(const CrlConfig* c, const CrlState* st, const CrlOut* out, const CrlLayoutIn* lay,
                          const int32_t* env_ids, int32_t n, void* stream) {
  KParams p;
  if (!out || !out->zone_obs || !lay || !lay->xy0 || !lay->rot0 || !lay->zone_xy) return CRL_ERR_NULL;
  int rc = fill_params(c, st, out, p);
  if (rc) return rc;
  if (c->task == CRL_TASK_TTSP && !lay->zone_max_steps) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_CM && !lay->colours) return CRL_ERR_NULL;
  if (n < 0 || n > c->num_envs) return CRL_ERR_CONFIG;
  if (n == 0) return CRL_OK;
  LayoutParams L{lay->xy0, lay->rot0, lay->zone_xy, lay->zone_max_steps, lay->colours, env_ids, n};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CRL_CALL_LAYOUT(T, NN) { reset_from_layout_kernel<T, NN><<<(n + 127) / 128, 128, 0, s>>>(p, L); }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_LAYOUT);
  return launch_status();
}

int crl_prefetch_layouts(const CrlConfig* c, const CrlState* st, int32_t warps_per_sm, uint32_t round, void* stream) {
  KParams p;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  if (!p.next_ready || !st->prefetch_work || !p.epoch) return CRL_ERR_NULL;
  if (round > 0xffffff00u) return CRL_ERR_CONFIG;
  p.round = round;
  if (!aligned16(st->prefetch_work)) return CRL_ERR_ALIGN;
  if (warps_per_sm <= 0) warps_per_sm = 2;
  if (warps_per_sm > 32) warps_per_sm = 32;
  WorkItem* work = reinterpret_cast<WorkItem*>(st->prefetch_work);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(work, 0, sizeof(WorkHeader), s) != cudaSuccess) return CRL_ERR_DEVICE;
  // (0) empty slots -> dense work list
  // every sampler kernel runs in small CTAs (<= 64 registers x 32 or 64 threads): they fit into the registers
  // the step kernel leaves free on each SM (MaxRegs) instead of displacing one of its CTAs
  const int blocks_0 = min((p.B + 63) / 64, 148 * 8);
#define CRL_CALL_PREFETCH_0(T, NN) { prefetch_scan_kernel<NN><<<blocks_0, 64, 0, s>>>(p, work); }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_PREFETCH_0);
  // (A) layouts: persistent lanes, one layout each; a few warps per SM share it with the steps
  const int blocks_a = min((2 * p.B + 31) / 32, 148 * warps_per_sm);
  const uint32_t done_state = c->task == CRL_TASK_TSP ? kSlotReady + round : kSlotLayoutDone;
#define CRL_CALL_PREFETCH_A(T, NN) { prefetch_layout_kernel<NN><<<blocks_a, 32, 0, s>>>(p, work, done_state); }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_PREFETCH_A);
  rc = launch_status();
  if (rc || c->task == CRL_TASK_TSP) return rc;
  // (B) task draws for the same work list
  const int blocks_b = min((2 * p.B + 1) / 2, 148 * 4);
#define CRL_CALL_PREFETCH_B(T, NN) { prefetch_task_kernel<T, NN><<<blocks_b, 32, 0, s>>>(p, work); }
  CRL_DISPATCH(c->task, c->num_zones, CRL_CALL_PREFETCH_B);
  return launch_status();
}

int crl_prefetch_publish(const CrlState* st, uint32_t round, void* stream) {
  if (!st || !st->prefetch_epoch) return CRL_ERR_NULL;
  publish_epoch_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(st->prefetch_epoch, round);
  return launch_status();
}

int crl_set_goal(const CrlConfig* c, const CrlState* st, const int32_t* goals, void* stream) {
  KParams p;
  if (!goals) return CRL_ERR_NULL;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  if (!p.goal) return CRL_ERR_NULL;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int blocks = (p.B + 255) / 256;
  if (c->task == CRL_TASK_CM) set_goal_kernel<CRL_TASK_CM><<<blocks, 256, 0, s>>>(p, goals, c->num_zones);
  else set_goal_kernel<CRL_TASK_TSP><<<blocks, 256, 0, s>>>(p, goals, c->num_zones);
  return launch_status();
}

int crl_goal_query(const CrlConfig* c, const CrlState* st, float* goal_xy, uint8_t* needs_goal,
                   uint8_t* available, void* stream) {
  KParams p;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  if (!p.goal) return CRL_ERR_NULL;
  if (goal_xy && (reinterpret_cast<uintptr_t>(goal_xy) & 7u)) return CRL_ERR_ALIGN;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int blocks = (p.B + 255) / 256;
  float2* gx = reinterpret_cast<float2*>(goal_xy);
  if (c->task == CRL_TASK_CM) goal_query_kernel<CRL_TASK_CM><<<blocks, 256, 0, s>>>(p, gx, needs_goal, available, c->num_zones);
  else goal_query_kernel<CRL_TASK_TSP><<<blocks, 256, 0, s>>>(p, gx, needs_goal, available, c->num_zones);
  return launch_status();
}

int crl_set_qpos_qvel(const CrlConfig* c, const CrlState* st, const double* qpos, const double* qvel,
                      const int32_t* env_ids, int32_t n, void* stream) {
  KParams p;
  if (!qpos || !qvel) return CRL_ERR_NULL;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  if (n <= 0) return n == 0 ? CRL_OK : CRL_ERR_CONFIG;
  set_qpos_qvel_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(p, qpos, qvel, env_ids, n);
  return launch_status();
}

int crl_get_qpos_qvel(const CrlConfig* c, const CrlState* st, double* qpos, double* qvel,
                      const int32_t* env_ids, int32_t n, void* stream) {
  KParams p;
  if (!qpos || !qvel) return CRL_ERR_NULL;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  if (n <= 0) return n == 0 ? CRL_OK : CRL_ERR_CONFIG;
  get_qpos_qvel_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(p, qpos, qvel, env_ids, n);
  return launch_status();
}

int crl_step_host(const CrlConfig* c, const CrlState* st, const float* actions_host, float* actions_dev,
                  const CrlOut* out, const CrlOut* host_out, uint32_t flags, void* stream) {
  if (!c || !actions_host || !actions_dev || !out || !host_out || !host_out->obs || !host_out->zone_obs ||
      !host_out->result)
    return CRL_ERR_NULL;
  int rc = check_config(c);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t B = c->num_envs, N = c->num_zones, Z = zone_dim(c->task);
  if (cudaMemcpyAsync(actions_dev, actions_host, B * 8, cudaMemcpyHostToDevice, s) != cudaSuccess) return CRL_ERR_DEVICE;
  rc = crl_step(c, st, actions_dev, out, flags, 0, 0, stream);
  if (rc) return rc;
  if (cudaMemcpyAsync(host_out->obs, out->obs, B * 32, cudaMemcpyDeviceToHost, s) != cudaSuccess) return CRL_ERR_DEVICE;
  if (cudaMemcpyAsync(host_out->zone_obs, out->zone_obs, B * N * Z * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess)
    return CRL_ERR_DEVICE;
  if (cudaMemcpyAsync(host_out->result, out->result, B * 8, cudaMemcpyDeviceToHost, s) != cudaSuccess)
    return CRL_ERR_DEVICE;
  if ((flags & CRL_STEP_GOALS) && host_out->shaped_reward &&
      cudaMemcpyAsync(host_out->shaped_reward, out->shaped_reward, B * 4, cudaMemcpyDeviceToHost, s) != cudaSuccess)
    return CRL_ERR_DEVICE;
  if (cudaStreamSynchronize(s) != cudaSuccess) return CRL_ERR_DEVICE;
  return CRL_OK;
}

// device-side alias of a page-locked, device-mapped host pointer (NULL if it is not one); a small per-thread cache:
// a caller rotating a few action buffers must not evict the fixed ones
static void* mapped_alias(const void* h) {
  struct Mapped { const void* host; void* dev; };
  static thread_local Mapped cache[64] = {};
  static thread_local int next = 0;
  if (!h) return nullptr;
  for (auto& m : cache) if (m.host == h) return m.dev;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, h) != cudaSuccess || a.type != cudaMemoryTypeHost || !a.devicePointer) {
    (void)cudaGetLastError();
    return nullptr;
  }
  cache[next] = Mapped{h, a.devicePointer};
  next = (next + 1) % 64;
  return a.devicePointer;
}

// crl_host_call_*: the zero-copy host step with everything but the actions resolved once
struct CrlHostCall {
  const CrlConfig* cfg;
  const CrlState* st;
  CrlOut direct;               // obs / result / shaped_reward: device aliases of the caller's host buffers
  float* zone_obs_host;        // device alias of the caller's host zone_obs
  CrlResult* result_dev;       // the device copy of the result records
  uint32_t flags;
  const void* act_host[8];     // the caller's action buffers seen so far
  const float* act_dev[8];
  int act_next;
};

int crl_host_call_create(const CrlConfig* c, const CrlState* st, const CrlOut* out, const CrlOut* host_out, uint32_t flags,
                         CrlHostCall** call) {
  if (!c || !st || !out || !host_out || !host_out->obs || !host_out->zone_obs || !host_out->result || !st->row_list || !call)
    return CRL_ERR_NULL;
  int rc = check_config(c);
  if (rc) return rc;
  CrlHostCall h{};
  if (!out->result) return CRL_ERR_NULL;
  h.cfg = c; h.st = st; h.direct = *out; h.flags = flags | CRL_STEP_TRACK_ROWS; h.result_dev = out->result;
  h.direct.obs = static_cast<float*>(mapped_alias(host_out->obs));
  h.direct.result = static_cast<CrlResult*>(mapped_alias(host_out->result));
  h.zone_obs_host = static_cast<float*>(mapped_alias(host_out->zone_obs));
  if ((flags & CRL_STEP_GOALS) && host_out->shaped_reward)
    h.direct.shaped_reward = static_cast<float*>(mapped_alias(host_out->shaped_reward));
  if (!h.direct.obs || !h.direct.result || !h.zone_obs_host || ((flags & CRL_STEP_GOALS) && !h.direct.shaped_reward))
    return CRL_ERR_CONFIG;
  *call = new CrlHostCall(h);
  return CRL_OK;
}

int crl_host_call_step(CrlHostCall* h, const float* actions_host, void* stream) {
  if (!h || !actions_host) return CRL_ERR_NULL;
  const float* act = nullptr;
  for (int i = 0; i < 8; ++i) if (h->act_host[i] == actions_host) { act = h->act_dev[i]; break; }
  if (!act) {
    act = static_cast<const float*>(mapped_alias(actions_host));
    if (!act) return CRL_ERR_CONFIG;
    h->act_host[h->act_next] = actions_host; h->act_dev[h->act_next] = act;
    h->act_next = (h->act_next + 1) % 8;
  }
  int rc = step_launch(h->cfg, h->st, act, &h->direct, h->flags, 0, 0, h->zone_obs_host, stream, h->result_dev);
  if (rc) return rc;
  if (cudaStreamSynchronize(static_cast<cudaStream_t>(stream)) != cudaSuccess) return CRL_ERR_DEVICE;
  return CRL_OK;
}

void crl_host_call_destroy(CrlHostCall* h) { delete h; }

int crl_gae(const CrlResult* results, const float* reward_override, const float* values, const float* next_value,
            double discount, double gae_lambda, int32_t num_frames, int32_t num_envs, float* advantages,
            float* returns, void* stream) {
  if (!results || !values || !next_value || !advantages) return CRL_ERR_NULL;
  if (num_frames <= 0 || num_envs <= 0) return CRL_ERR_CONFIG;
  if (reinterpret_cast<uintptr_t>(results) & 7u) return CRL_ERR_ALIGN;
  // torch rounds the Python doubles `discount` and `discount * gae_lambda` to float32 when they
  // meet a float32 tensor
  const float g = (float)discount, gl = (float)(discount * gae_lambda);
  gae_kernel<<<(num_envs + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const unsigned long long*>(results), reward_override, values, next_value, g, gl, num_frames,
      num_envs, advantages, returns);
  return launch_status();
}

int crl_frame_capture(const CrlConfig* c, const CrlState* st, const CrlResult* result, int32_t initial, CrlFrame* frames_t,
                      float* layout_xy, uint32_t* layout_tmax, uint32_t capacity, uint32_t* fill, void* stream) {
  const int rc = check_config(c);
  if (rc) return rc;
  if (!st || !st->aux || !st->zone_xy || !frames_t || !layout_xy || !fill || (!initial && !result)) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_TTSP && (!st->zone_tmax || !layout_tmax)) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_CM && !st->cooldown) return CRL_ERR_NULL;
  if (capacity == 0u) return CRL_ERR_CONFIG;
  if (!aligned16(st->aux) || !aligned16(frames_t) || (reinterpret_cast<uintptr_t>(layout_xy) & 7u) ||
      (reinterpret_cast<uintptr_t>(result) & 7u) || (reinterpret_cast<uintptr_t>(fill) & 3u))
    return CRL_ERR_ALIGN;
  CaptureParams p;
  p.aux = reinterpret_cast<const float4*>(st->aux);
  p.zone_xy = reinterpret_cast<const float2*>(st->zone_xy);
  p.zone_tmax = c->task == CRL_TASK_TTSP ? st->zone_tmax : nullptr;
  p.cooldown = c->task == CRL_TASK_CM ? reinterpret_cast<const uint2*>(st->cooldown) : nullptr;
  p.result = reinterpret_cast<const unsigned long long*>(result);
  p.frames = reinterpret_cast<uint4*>(frames_t);
  p.layout_xy = reinterpret_cast<float2*>(layout_xy);
  p.layout_tmax = c->task == CRL_TASK_TTSP ? layout_tmax : nullptr;
  p.fill = fill; p.capacity = capacity;
  p.B = c->num_envs; p.N = c->num_zones; p.initial = initial != 0;
  frame_capture_kernel<<<(p.B + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  return launch_status();
}

// crl_copy_envs: the state planes of one side, checked as fill_params checks them (the counters are not copied and
// not needed).
static int copy_state_side(const CrlConfig* c, const CrlState* st, const int32_t* ids, CopySide& side) {
  if (!st || !st->pose || !st->aux || !st->zone_xy || !st->seed || !st->episode || !st->origin) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_TTSP && !st->zone_tmax) return CRL_ERR_NULL;
  if (c->task == CRL_TASK_CM && !st->cooldown) return CRL_ERR_NULL;
  if (!aligned16(st->pose) || !aligned16(st->aux) || !aligned16(st->zone_xy) || !aligned16(st->origin) ||
      (reinterpret_cast<uintptr_t>(st->seed) & 7u) || (reinterpret_cast<uintptr_t>(st->cooldown) & 7u))
    return CRL_ERR_ALIGN;
  side.pose = reinterpret_cast<float4*>(st->pose); side.aux = reinterpret_cast<float4*>(st->aux);
  side.zone_xy = reinterpret_cast<float2*>(st->zone_xy);
  side.zone_tmax = c->task == CRL_TASK_TTSP ? st->zone_tmax : nullptr;
  side.cooldown = c->task == CRL_TASK_CM ? reinterpret_cast<uint2*>(st->cooldown) : nullptr;
  side.seed = reinterpret_cast<long long*>(st->seed); side.episode = st->episode;
  side.origin = reinterpret_cast<float4*>(st->origin);
  side.ids = ids; side.B = c->num_envs;
  return CRL_OK;
}

// the two configs describe the same task instance: every field but the batch's size, place and seed range
static bool same_task_config(const CrlConfig* a, const CrlConfig* b) {
  CrlConfig x = *a, y = *b;
  for (CrlConfig* c : {&x, &y}) { c->num_envs = 0; c->env_offset = 0; c->seed_mode = 0; c->min_seed = 0; c->max_seed = 0; }
  return memcmp(&x, &y, sizeof(CrlConfig)) == 0;
}

int crl_copy_envs(const CrlConfig* dst_cfg, const CrlState* dst, const CrlOut* dst_out, const int32_t* dst_ids,
                  const CrlConfig* src_cfg, const CrlState* src, const CrlOut* src_out, const int32_t* src_ids,
                  int32_t n, uint32_t* rejected, void* stream) {
  int rc = check_config(dst_cfg);
  if (rc) return rc;
  if ((rc = check_config(src_cfg))) return rc;
  if (!same_task_config(dst_cfg, src_cfg)) return CRL_ERR_CONFIG;
  if (n < 0) return CRL_ERR_CONFIG;
  CopyParams p;
  memset(&p, 0, sizeof(p));
  if ((rc = copy_state_side(dst_cfg, dst, dst_ids, p.dst))) return rc;
  if ((rc = copy_state_side(src_cfg, src, src_ids, p.src))) return rc;
  if (dst->goal && src->goal) { p.dst.goal = dst->goal; p.src.goal = src->goal; }
  if (!dst_out != !src_out) return CRL_ERR_NULL;
  if (dst_out) {
    if (!dst_out->obs != !src_out->obs || !dst_out->zone_obs != !src_out->zone_obs ||
        !dst_out->result != !src_out->result || !dst_out->shaped_reward != !src_out->shaped_reward)
      return CRL_ERR_NULL;
    if (!aligned16(dst_out->obs) || !aligned16(src_out->obs) || (reinterpret_cast<uintptr_t>(dst_out->result) & 7u) ||
        (reinterpret_cast<uintptr_t>(src_out->result) & 7u) || (reinterpret_cast<uintptr_t>(dst_out->zone_obs) & 3u) ||
        (reinterpret_cast<uintptr_t>(src_out->zone_obs) & 3u))
      return CRL_ERR_ALIGN;
    p.dst.obs = reinterpret_cast<float4*>(dst_out->obs); p.src.obs = reinterpret_cast<float4*>(src_out->obs);
    p.dst.zone_obs = dst_out->zone_obs; p.src.zone_obs = src_out->zone_obs;
    p.dst.result = reinterpret_cast<unsigned long long*>(dst_out->result);
    p.src.result = reinterpret_cast<unsigned long long*>(src_out->result);
    p.dst.shaped = dst_out->shaped_reward; p.src.shaped = src_out->shaped_reward;
  }
  if ((reinterpret_cast<uintptr_t>(rejected) & 3u) || (reinterpret_cast<uintptr_t>(dst_ids) & 3u) ||
      (reinterpret_cast<uintptr_t>(src_ids) & 3u))
    return CRL_ERR_ALIGN;
  p.next_ready = dst->next_ready;
  p.rejected = rejected;
  p.n = n;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CRL_CALL_COPY(T, NN) { if (n > 0) copy_envs_kernel<T, NN><<<(n + 255) / 256, 256, 0, s>>>(p); }
  CRL_DISPATCH(dst_cfg->task, dst_cfg->num_zones, CRL_CALL_COPY);
  return n > 0 ? launch_status() : CRL_OK;
}

int crl_check_state(const CrlConfig* c, const CrlState* st, uint64_t* violations, void* stream) {
  KParams p;
  if (!violations) return CRL_ERR_NULL;
  int rc = fill_params(c, st, nullptr, p);
  if (rc) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(violations, 0, 8 * sizeof(uint64_t), s) != cudaSuccess) return CRL_ERR_DEVICE;
  check_state_kernel<<<(p.B + 255) / 256, 256, 0, s>>>(p, c->task, c->num_zones,
                                                       reinterpret_cast<unsigned long long*>(violations));
  return launch_status();
}

int crl_counters_read(const CrlState* st, double out[8], void* stream) {
  if (!st || !st->counters || !out) return CRL_ERR_NULL;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cudaMemcpyAsync(out, st->counters, 8 * sizeof(double), cudaMemcpyDeviceToHost, s) != cudaSuccess)
    return CRL_ERR_DEVICE;
  if (cudaStreamSynchronize(s) != cudaSuccess) return CRL_ERR_DEVICE;
  return CRL_OK;
}

}  // extern "C"
