// crl_encode.cu -- the consumer side of the observation: ZoneEnvModel's per-zone network and
// mean-pool (main/src/env_model.py:56-78), fused into one sm_100a kernel (SURVEY.md 8f rank 2).
//
//   zone_emb[e] = 1/N * sum_z  L3( relu( L2( relu( L1( [obs[e], zone_obs[e][z]] ))))),   L_i = nn.Linear
//               = L3( pooled[e] ),   pooled[e] = 1/N * sum_z relu( L2( relu( L1( . ))))    (L3 is affine)
//
// The reference materialises three (B*N, h) activations (h = 185 by default,
// main/scripts/train_ppo.py:66).  Here the kernel produces `pooled` (B, h) and nothing else; the
// mean is taken BEFORE the third Linear, which turns L3 from a (B N, h) x (h, h) GEMM into a
// (B, h) x (h, h) one (a third of the tensor work gone): L3 and combine_net_ (env_model.py:79) stay
// plain fp32 library GEMMs on the caller's side.
//
// The two wide GEMMs run TRANSPOSED on the 5th-gen tensor cores: H^T = W X^T, i.e. the weights are
// the A operand (M = hidden units, in blocks of 128 = the TMEM lanes) and a tile of 128 (env, zone) rows
// -- 8 envs of 16 zone slots, or 16 envs of 8 slots when N <= 8; slots beyond N are padding -- is the N
// dimension (TMEM columns).
// tcgen05.mma.cta_group::1.kind::f16: bf16 operands, fp32 accumulators in TMEM, M = 128, N = 128,
// K = 16 per instruction.  Why transposed: an accumulator row lives in ONE thread's registers after
// tcgen05.ld, so with the 16 zone slots of an env on consecutive COLUMNS the mean over zones is 15
// register adds per env -- no shuffles -- and lane j stores hidden unit j, i.e. coalesced rows of the
// output.  (The first version had rows = (env, zone) on the lanes: half of its instructions were a
// shuffle butterfly.)  W1 / W2 stay resident in shared memory for the whole persistent kernel.
//
// Epilogues are the bottleneck of such a narrow MLP (K <= 192 gives the tensor pipe ~1,700 cycles per
// tile while 2 x 96 KB of accumulator come back through registers), so they are minimal:
//  * the BIASES ARE FOLDED INTO THE GEMMS -- the K dimension carries constant-1 entries (layer 1:
//    input columns in_dim, in_dim + 1; layer 2: hidden rows h, h + 1, produced by two "generator" rows
//    of W1) that multiply the bias split into a bf16 high and low part;
//  * epilogue 1 = one cvt.rn.relu.bf16x2.f32 per pair of values + 16-byte stores: 8 consecutive rows m of
//    one hidden unit j are exactly one 16-byte unit of the layer-2 B operand in MN-major layout;
//  * epilogue 2 = one max per value (NaN-propagating) + the register adds + two coalesced stores per 32 values.
// A padding row is all zeros including its ones, hence stays exactly zero through both layers and
// drops out of the mean by itself.
//
// A CTA = two independent groups of 256 threads, each walking its own sequence of tiles with its own
// accumulators, operand buffers and mbarrier: while one group is in an epilogue (CUDA cores) the other
// group's MMAs occupy the tensor pipe.  Warp w of a group owns TMEM lane quadrant w % 4 of M-block
// w / 4.  The next tile's inputs are prefetched into registers.  Every wait is bounded.
//
// A separate translation unit on purpose: nothing here can move the register allocation of the
// step kernels (crl_kernels.cu; see profiles/r01_notes.md on how easily that happens).
//
// Shared-memory operand images (no swizzle; canonical layouts of cute::UMMA, mma_traits_sm100.hpp), all
// made of 8 x 8 core matrices of 128 contiguous bytes:
//  K-major (W1, W2 as A; the input rows X as B of layer 1): element (r, k) of an R x K matrix at
//      (r % 8) * 16 + (r / 8) * (16 K) + (k / 8) * 128 + (k % 8) * 2      LBO = 128 (next core matrix along K),
//                                                                         SBO = 16 K (next 8 rows)
//  MN-major (the layer-1 activations H1 as B of layer 2, N = row m, K = hidden unit j): element (m, j) at
//      (j % 8) * 16 + (j / 8) * 2048 + (m / 8) * 128 + (m % 8) * 2        LBO = 2048 (next 8 j), SBO = 128 (next 8 m)
// One tcgen05.mma consumes K = 16 = two core matrices along K.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/crl_b200.h"
#include "crl_core.cuh"

namespace crl_enc {

constexpr int kRows = 128;          // (env, zone) rows of a tile = the N of every MMA = accumulator columns
constexpr int kGroupThreads = 256;  // 8 warps: one per (M-block, TMEM lane quadrant)
constexpr int kGroups = 2;          // independent groups per CTA
// an env owns S = 8 (N <= 8) or 16 consecutive row slots of a tile; the slots beyond N are padding rows
__host__ __device__ inline int slots_per_env(int n_zones) { return n_zones <= 8 ? 8 : 16; }
// padded input width of layer 1: the per-env features (obs, and goal / one-hot skill for the reference's
// ZoneEnvGoalModel / ZoneEnvSkillModel, which the caller concatenates to obs), the zone row and at
// least one ones column; one or two K = 16 steps
__host__ __device__ inline int padded_k1(int in_dim) { return in_dim + 1 <= 16 ? 16 : 32; }
constexpr uint32_t kTmemCols = 512; // two M-blocks x 128 columns per group; the CTA owns the SM
constexpr uint32_t kSpinLimit = 1u << 24;

// K of layer 2: the h hidden units plus the two ones rows, multiple of 16
__host__ __device__ inline int padded_k(int h) { return (h + 2 + 15) & ~15; }
// M of both layers: blocks of 128 lanes covering padded_k (the ones rows are outputs of layer 1)
__host__ __device__ inline int padded_m(int h) { return (padded_k(h) + 127) & ~127; }

// byte offset of element (r, k) in the K-major image of a matrix with K columns
__host__ __device__ inline uint32_t canon(int r, int k, int K) {
  return (uint32_t)((r & 7) * 16 + (r >> 3) * (16 * K) + (k >> 3) * 128 + (k & 7) * 2);
}

struct Offsets {   // byte offsets: packed weight buffer == start of shared memory; then per-group buffers
  uint32_t w2, w1, packed_end, group0, h1, xbuf, bar, group_bytes, tmem_slot, smem_end;
};
__host__ __device__ inline Offsets offsets(int h, int in_dim) {
  const int KP = padded_k(h), MP = padded_m(h), kK1 = padded_k1(in_dim);
  Offsets o;
  o.w2 = 0;
  o.w1 = o.w2 + (uint32_t)MP * KP * 2;
  o.packed_end = o.w1 + (uint32_t)MP * kK1 * 2;
  o.group0 = (o.packed_end + 127u) & ~127u;
  o.h1 = 0;                                              // relative to the group's base
  o.xbuf = o.h1 + (uint32_t)KP * kRows * 2;
  o.bar = o.xbuf + (uint32_t)kRows * kK1 * 2;
  o.group_bytes = (o.bar + 40 + 127u) & ~127u;           // five mbarriers per slot (kBarBytes)
  o.tmem_slot = o.group0 + kGroups * o.group_bytes;    // + 8: the mbarrier of the weights' bulk copy
  o.smem_end = o.tmem_slot + 16;
  return o;
}

// ---- packing: torch-layout fp32 weights -> the shared-memory image -------------------------
struct PackArgs {
  const float *w1, *b1, *w2, *b2;
  uint8_t* out;
  int in_dim, h;
};

__global__ void pack_kernel(const PackArgs a) {
  const Offsets o = offsets(a.h, a.in_dim);
  const int KP = padded_k(a.h), MP = padded_m(a.h), kK1 = padded_k1(a.in_dim);
  const int n_w = MP * KP, n_w1 = MP * kK1;
  const int total = n_w + n_w1;
  // bias = hi + lo with hi = bf16(bias), lo = bf16(bias - hi): entry `ones` of the K dimension carries 1
  // and multiplies hi, entry `ones + 1` multiplies lo (layer 1 has the second one only if in_dim < 15)
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const bool second = i < n_w;
    const int K = second ? KP : kK1, ones = second ? a.h : a.in_dim;
    const int j = second ? i : i - n_w, row = j / K, k = j % K;
    // image row -> hidden unit: M-block 1 holds units 128 .. 191 in its UPPER 64 rows (lane quadrants 2 and 3), so that
    // its accumulators are drained by warps on the two schedulers that M-block 0 loads least; its lower rows are zero
    const int n = row < 128 ? row : (row >= 192 ? row - 64 : 1 << 20);
    const float* w = second ? a.w2 : a.w1;
    const float* b = second ? a.b2 : a.b1;
    float v = 0.f;
    if (n < a.h) {
      if (k < ones) v = w[(size_t)n * ones + k];
      else if (k == ones) v = __bfloat162float(__float2bfloat16_rn(b[n]));
      else if (k == ones + 1) v = b[n] - __bfloat162float(__float2bfloat16_rn(b[n]));
    } else if (!second && (n == a.h || n == a.h + 1) && k == ones) {
      v = 1.f;                                   // generator rows of W1: layer 2's ones entries h, h + 1
    }
    *reinterpret_cast<__nv_bfloat16*>(a.out + (second ? o.w2 : o.w1) + canon(row, k, K)) = __float2bfloat16_rn(v);
  }
}

// ---- PTX helpers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor: start address, LBO, SBO, version 1 (sm_100), no swizzle
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32) | (1ull << 46);
}

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32, issued by one thread
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(bar) : "memory");
}
// bounded wait on an mbarrier phase: returns false if it never completed (the caller reports it)
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t it = 0; it < kSpinLimit; ++it) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return true;
#ifdef CRL_ENC_DIAG_SLEEP                                       // timing diagnostic: how much do the polling warps cost the MMAs' operand reads
    __nanosleep(CRL_ENC_DIAG_SLEEP);
#endif
  }
  return false;
}
// this warp's 32 lanes x 32 consecutive fp32 columns of TMEM -> 32 registers per thread.  Asynchronous:
// tmem_ld_wait(v) before v is read (several loads may be in flight).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
// the registers are in/out operands so that no use of them can be scheduled above the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
      : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
        "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
        "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
        "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
      :: "memory");
}
// barrier over the 256 threads of one group (barrier 0 is __syncthreads)
__device__ __forceinline__ void group_sync(int group) { asm volatile("bar.sync %0, 256;" :: "r"(group + 1) : "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);   // .x (low half) = lo
  return *reinterpret_cast<const uint32_t*>(&t);
}
// {bf16(max(lo, 0)), bf16(max(hi, 0))} in one instruction (the first source lands in the upper half)
__device__ __forceinline__ uint32_t relu_pack_bf16(uint32_t lo_bits, uint32_t hi_bits) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(__uint_as_float(hi_bits)), "f"(__uint_as_float(lo_bits)));
  return d;
}

struct EncArgs {
  const float* obs;        // [B][obs_dim]
  const float* zone_obs;   // [B][N][Z]
  const uint8_t* packed;
  float* out;              // [B][h]: pooled hidden activation
  // crl_encoder_forward: instead of `out`, the kernel writes the head kernel's layer-input image directly -- per tile of
  // 128 envs the canonical K-major bf16 operand [obs, pooled, 1, 1, 0..] (head_k columns) -- so that the head's staging is
  // one bulk copy per tile and `pooled` never exists in fp32 (the head rounds it to bf16 anyway: identical results)
  uint8_t* xhead;
  int KH;                  // head_k(obs_dim, h)
  int* status;             // device int: set to 1 if a tensor-core wait expired
  int B, N, Z, obs_dim, h, n_tiles, S;   // S = slots_per_env(N)
  // crl_zone_encode_state: the zone part of the input rows is built from the STATE planes instead of being read
  // from a materialised zone_obs (aux != nullptr selects it; zone_obs is then not touched)
  const float4* aux;           // float4[B]: .w = steps | visited mask / colour codes << 16
  const float2* zone_xy;       // float2[N][B]
  const uint32_t* zone_tmax;   // uint32[ceil(N/2)][B] (TimedTSP)
  const uint2* cooldown;       // uint2[B] (ColourMatch)
  int task, num_steps;
  crl::DivConst div_steps, div_cd;
  // crl_zone_encode_frames / crl_frames_zone_obs: the zone part is built from a CrlFrame per row and the layout table
  const uint4* frames;         // CrlFrame[B]: bits, layout, cooldown
  const float2* layout_xy;     // float2[capacity][N]
  const uint32_t* layout_tmax; // uint32[capacity][ceil(N/2)] (TimedTSP)
};

// where the zone part of a layer-1 input row comes from
enum RowSrc : int { kSrcZoneObs = 0, kSrcState = 1, kSrcFrames = 2 };

// The features of zone `slot`: EXACTLY what step_kernel's zone_row writes to zone_obs[e][slot] (crl_kernels.cu;
// tests/test_gpu_encode.py and tests/test_gpu_rollout_frames.py compare bit for bit): x/3, y/3, r, g, b, 0.25
// [, time left | cooldown / max_cooldown], from the zone centre c, the state word aux.w and -- loaded only by the task
// that needs it -- the TimedTSP timeout word (tmax_word()) or the ColourMatch cooldown bytes (cooldown()).
template <class TmaxWord, class Cooldown>
__device__ __forceinline__ void zone_features(int task, const crl::DivConst& div_steps, const crl::DivConst& div_cd,
                                              float2 c, uint32_t bits, int slot, TmaxWord tmax_word, Cooldown cooldown,
                                              float (&z)[7]) {
  const int steps = (int)(bits & 0xffffu);
  const uint32_t hi = bits >> 16;
  const float third = 1.0f / 3.0f;
  z[0] = c.x * third; z[1] = c.y * third; z[5] = 0.25f; z[6] = 0.f;
  if (task == CRL_TASK_CM) {
    const uint32_t col = (hi >> (2 * slot)) & 3u;               // 0 B, 1 G, 2 R
    z[2] = col == 2u ? 1.f : 0.f; z[3] = col == 1u ? 1.f : 0.f; z[4] = col == 0u ? 1.f : 0.f;
    const uint2 cd = cooldown();
    const uint32_t w = slot < 4 ? cd.x : cd.y;
    z[6] = crl::div_const((float)((w >> (8 * (slot & 3))) & 0xffu), div_cd);
  } else {
    const bool v = (hi >> slot) & 1u;                          // Yellow (1,1,0) visited / Cyan (0,1,1)
    z[2] = v ? 1.f : 0.f; z[3] = 1.f; z[4] = v ? 0.f : 1.f;
    if (task == CRL_TASK_TTSP) {
      const uint32_t w = tmax_word();
      const int tm = (int)((w >> (16 * (slot & 1))) & 0xffffu);
      z[6] = v ? 1.0f : crl::div_const((float)(tm - steps), div_steps);
    }
  }
}

// ... of env e, from the state planes
__device__ __forceinline__ void zone_features_from_state(const EncArgs& a, int e, int slot, float (&z)[7]) {
  const float2 c = __ldg(a.zone_xy + (size_t)slot * a.B + e);
  const uint32_t bits = (uint32_t)__float_as_int(__ldg(reinterpret_cast<const float*>(a.aux + e) + 3));
  zone_features(a.task, a.div_steps, a.div_cd, c, bits, slot,
                [&] { return __ldg(a.zone_tmax + (size_t)(slot >> 1) * a.B + e); }, [&] { return __ldg(a.cooldown + e); }, z);
}

// ... of row e, from its CrlFrame and the layout table; a record without a layout entry (the table overflowed) gives NaN
__device__ __forceinline__ void zone_features_from_frame(const EncArgs& a, int e, int slot, float (&z)[7]) {
  const uint4 f = __ldg(a.frames + e);                         // bits, layout, cooldown.x, cooldown.y
  if (f.y == CRL_FRAME_NO_LAYOUT) {
#pragma unroll
    for (int j = 0; j < 7; ++j) z[j] = __int_as_float(0x7fc00000);
    return;
  }
  const float2 c = __ldg(a.layout_xy + (size_t)f.y * a.N + slot);
  zone_features(a.task, a.div_steps, a.div_cd, c, f.x, slot,
                [&] { return __ldg(a.layout_tmax + (size_t)f.y * ((a.N + 1) >> 1) + (slot >> 1)); },
                [&] { return make_uint2(f.z, f.w); }, z);
}

// eight consecutive values (k = 8 kc .. 8 kc + 7) of row (e, slot) of the layer-1 input
// [obs[e], zone_obs[e][slot], 1, 1, 0...]; all zeros -- the ones included -- for a padding row.
// SRC (RowSrc): kSrcState / kSrcFrames build the zone part from the state planes / from a CrlFrame (obs_dim == 8, so
// chunk 1 is exactly the zone features + ones); a template parameter so that the materialised path compiles exactly as
// it did without them.
template <int SRC>
__device__ __forceinline__ void load_half_row(const EncArgs& a, int tile, int m, int kc, float (&x)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) x[j] = 0.f;
  const int sh = a.S == 16 ? 4 : 3;                          // S is 8 or 16: no runtime division on this path
  const int e = (tile << (7 - sh)) + (m >> sh), slot = m & (a.S - 1);
  if (tile < a.n_tiles && e < a.B && slot < a.N) {
    const float* ob = a.obs + (size_t)e * a.obs_dim;
    if (SRC != kSrcZoneObs) {
      if (kc == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = __ldg(ob + j);
      } else {
        float z[7];
        if (SRC == kSrcState) zone_features_from_state(a, e, slot, z);
        else zone_features_from_frame(a, e, slot, z);
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = j < 7 && j < a.Z ? z[j < 7 ? j : 0] : (j <= a.Z + 1 ? 1.f : 0.f);
      }
    } else {
      const float* zo = a.zone_obs + ((size_t)e * a.N + slot) * a.Z;
      const int in_dim = a.obs_dim + a.Z;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int k = 8 * kc + j;
        if (k < a.obs_dim) x[j] = __ldg(ob + k);
        else if (k < in_dim) x[j] = __ldg(zo + (k - a.obs_dim));
        else if (k <= in_dim + 1) x[j] = 1.f;
      }
    }
  }
}

// max(v, 0) that passes a NaN on, as epilogue 1's cvt.rn.relu does (fmaxf would turn it into 0): a non-finite input row
// must give a non-finite `pooled` for its env, not a finite wrong one.  Same bits as fmaxf for every other v.
__device__ __forceinline__ float relu_nan(float v) {
  float r;
  asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(v));
  return r;
}

// relu of 32 consecutive rows m of this thread's hidden unit -> bf16 -> four 16-byte units of H1
__device__ __forceinline__ void relu_to_h1(const uint32_t (&v)[32], uint8_t* h1_row, int c, bool in_range) {
#ifdef CRL_ENC_DIAG_NO_H1_STORE                                 // timing diagnostic (wrong results): epilogue 1 without its shared-memory stores
  if (v[0] != 0x7fc12345u) return;
#endif
  if (!in_range) return;                                     // hidden rows >= KP do not exist in H1 (the X buffer follows it)
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    *reinterpret_cast<uint4*>(h1_row + (uint32_t)((c * 4 + q) * 128)) =
        make_uint4(relu_pack_bf16(v[q * 8 + 0], v[q * 8 + 1]), relu_pack_bf16(v[q * 8 + 2], v[q * 8 + 3]),
                   relu_pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), relu_pack_bf16(v[q * 8 + 6], v[q * 8 + 7]));
  }
}

// 32 consecutive rows m = the zone slots of envs e0 .. e0 + 32 / S - 1: relu, sum in registers, store column j.
// `col` = out + j (this thread's column of the output); `full`: every env of the tile exists and j < h, so the stores
// need no predicates (their address chains were a third of epilogue 2's time).
// relu + mean over the 16 zone slots of the two envs whose rows are the 32 columns of v
__device__ __forceinline__ void relu_pool16(const uint32_t (&v)[32], float inv_n, float& r0, float& r1) {
  float q[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float s[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      s[i] = relu_nan(__uint_as_float(v[8 * g + 2 * i])) + relu_nan(__uint_as_float(v[8 * g + 2 * i + 1]));
    q[g] = (s[0] + s[1]) + (s[2] + s[3]);
  }
  r0 = (q[0] + q[1]) * inv_n;
  r1 = (q[2] + q[3]) * inv_n;
}

// 8 x 8 transpose inside each group of 8 lanes: element i of lane r <-> element r of lane i (three exchange stages)
__device__ __forceinline__ void transpose8(float (&a)[8], int lane) {
#pragma unroll
  for (int d = 4; d >= 1; d >>= 1) {
    const bool up = (lane & d) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i & d) continue;                                     // pairs (i, i + d) with bit d of i clear
      const float send = up ? a[i] : a[i + d];
      const float got = __shfl_xor_sync(0xffffffffu, send, d);
      if (up) a[i] = got; else a[i + d] = got;
    }
  }
}

template <bool XHEAD = false>
__device__ __forceinline__ void relu_pool_store(const uint32_t (&v)[32], float* col, int h, int B, int S, int e0, bool full,
                                                bool j_ok, float inv_n, uint8_t* xh_unit = nullptr, int KH = 0) {
  float q[4];                                                 // sums of 8 consecutive rows
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float s[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      s[i] = relu_nan(__uint_as_float(v[8 * g + 2 * i])) + relu_nan(__uint_as_float(v[8 * g + 2 * i + 1]));
    q[g] = (s[0] + s[1]) + (s[2] + s[3]);
  }
  if (XHEAD) {                                               // crl_encoder_forward: bf16 into the head's operand image
    // xh_unit: this thread's unit in the image row of the zone tile's FIRST env.  The tile's 8 (S = 16) or 16 (S = 8) envs
    // are consecutive rows of one or two 8-row groups of the same head tile: env i of the tile at
    // + (i & 7) * 16 + (i >> 3) * 16 KH -- no per-store index arithmetic
    if (!j_ok) return;
    const int i0 = e0 & (S == 16 ? 7 : 15);
    if (S == 16) {
      if (e0 < B) *reinterpret_cast<__nv_bfloat16*>(xh_unit + i0 * 16) = __float2bfloat16_rn((q[0] + q[1]) * inv_n);
      if (e0 + 1 < B) *reinterpret_cast<__nv_bfloat16*>(xh_unit + (i0 + 1) * 16) = __float2bfloat16_rn((q[2] + q[3]) * inv_n);
    } else {
#pragma unroll
      for (int g = 0; g < 4; ++g)
        if (e0 + g < B)
          *reinterpret_cast<__nv_bfloat16*>(xh_unit + ((i0 + g) & 7) * 16 + ((i0 + g) >> 3) * (16 * KH)) = __float2bfloat16_rn(q[g] * inv_n);
    }
    return;
  }
  float* p = col + (size_t)e0 * (size_t)h;
  if (S == 16) {
    const float r0 = (q[0] + q[1]) * inv_n, r1 = (q[2] + q[3]) * inv_n;
    if (full) { p[0] = r0; p[h] = r1; }
    else if (j_ok) {
      if (e0 < B) p[0] = r0;
      if (e0 + 1 < B) p[h] = r1;
    }
  } else {
    if (full) {
#pragma unroll
      for (int g = 0; g < 4; ++g) p[(size_t)g * h] = q[g] * inv_n;
    } else if (j_ok) {
#pragma unroll
      for (int g = 0; g < 4; ++g)
        if (e0 + g < B) p[(size_t)g * h] = q[g] * inv_n;
    }
  }
}

// The pipeline (round 2).  17 warps: two GROUPS of 8 epilogue warps, each owning one tile slot (256 TMEM columns = two
// M-blocks of accumulators, an H1 buffer, an X buffer), and ONE issuing warp whose lane 0 issues every tcgen05.mma of
// both slots.  Nothing meets at a CTA / group barrier any more; five mbarriers per slot carry the dependencies:
//   full_x   (8 warp arrivals)  the slot's next input rows are staged AND its accumulators have been drained  -> L1 may go
//   full_h1  (8 warp arrivals)  epilogue 1 has written H1 (and read the layer-1 accumulators)                 -> L2 may go
//   l1_done  (tcgen05.commit)   layer 1 has completed                                                         -> epilogue 1
//   l2_done[b] (commit)         M-block b of layer 2 has completed                                            -> epilogue 2 of b
// Tensor-pipe order in steady state: L2 of slot g (24 MMAs) with the OTHER slot's next L1 inserted after the first few
// of them -- by then that slot's epilogue 2 (which started when ITS L2 completed, i.e. when this one began) has freed
// its accumulators -- so that slot's epilogue 1 runs under the rest of this L2 and its own L2 is ready to issue the
// moment this one ends: the pipe always has queued work, and each epilogue has a whole L2 (~1,500 cycles) to hide in.
// The issuing warp is warp 4 of group 0: an (M-block 1, lane quadrant 0) warp, which has no accumulator rows to drain
// (M-block 1's real rows sit in quadrants 2, 3).  Its share of the input staging goes to its neighbour, warp 5, which
// drains nothing either.  A 17th warp would cap the kernel at 96 registers per thread (five warps on one scheduler);
// with 16 warps it has 128 and no spills.
constexpr int kIssuerWarp = 4;
constexpr int kEncThreads = kGroupThreads * kGroups;
#ifndef CRL_ENC_INSERT_AFTER
#define CRL_ENC_INSERT_AFTER 12    // MMAs of an L2 issued before the issuer BLOCKS for the other slot's L1 (earlier if ready)
#endif
enum { kBarFullX = 0, kBarFullH1 = 8, kBarL1Done = 16, kBarL2Done = 24 /* + 8 b */, kBarBytes = 40 };

// one lane of a converged warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0u;
}
// Resident weights: global -> shared memory by the bulk-copy engine (cp.async.bulk, UBLKCP in SASS), completion counted
// in bytes on an mbarrier.  One thread issues it; nobody waits until the first MMA needs the image, so the copy runs
// under the first tiles' input staging (the register round trip it replaces took 13 passes of the whole CTA).
__device__ __forceinline__ void bulk_load_weights(uint32_t bar, uint32_t smem_dst, const uint8_t* src, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
  for (uint32_t off = 0; off < bytes; off += 32768u) {
    const uint32_t n = bytes - off < 32768u ? bytes - off : 32768u;
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_dst + off), "l"(src + off), "r"(n), "r"(bar) : "memory");
  }
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0u;
}

#ifdef CRL_ENC_TIMELINE   // diagnostic build: clock64 stamps of the first 64 tiles of every slot (tools/enc_timeline.py)
__device__ long long g_timeline[148 * 2 * 64 * 16];
#define CRL_TL(g, k, i) do { if ((k) < 64 && blockIdx.x < 148) g_timeline[((blockIdx.x * 2 + (g)) * 64 + (k)) * 16 + (i)] = clock64(); } while (0)
#else
#define CRL_TL(g, k, i) do { } while (0)
#endif

// XHEAD: the output goes into the head kernel's operand image (crl_encoder_forward) instead of `out`; a template
// parameter so that the plain kernels carry none of it (with a run-time test they lost 8 % to register pressure)
// WIDE: the layer-1 input takes two K steps (obs_dim + zone_dim + 1 > 16: ZoneEnvGoalModel / ZoneEnvSkillModel); a template
// parameter because the second prefetched chunk costs the one-step kernels eight registers they do not have (96 per thread)
template <int SRC, bool XHEAD, bool WIDE = false>
__global__ void __launch_bounds__(kEncThreads, 1) zone_encode_kernel(const EncArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const Offsets o = offsets(a.h, a.obs_dim + a.Z);
  const int KP = padded_k(a.h), MP = padded_m(a.h), kK1 = padded_k1(a.obs_dim + a.Z);
  const int n_mblocks = MP / 128;
  const int warp_idx = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform, and the compiler knows it
  const bool issuer = warp_idx == kIssuerWarp;
  const int group = warp_idx / (kGroupThreads / 32);          // 0 / 1 (the issuing warp: 0)
  const int t = threadIdx.x % kGroupThreads;
  const int m = t & (kRows - 1), half = t >> 7;               // input row / half of it this thread stages
  const int warp = t >> 5, lane = t & 31;
  const int mblock = warp >> 2, quad = warp & 3;              // accumulator rows this warp drains
  // hidden unit of this thread's accumulator row: M-block 1 keeps units 128 .. 191 in lane quadrants 2, 3 (pack_kernel)
  const int j0 = mblock == 0 ? quad * 32 : (quad >= 2 ? 128 + (quad - 2) * 32 : 1 << 20);
  const int j = j0 + lane;
  uint8_t* gbase = smem + o.group0 + (uint32_t)group * o.group_bytes;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + o.tmem_slot);
  const uint32_t bar0 = smem_u32(smem + o.group0 + o.bar);    // slot g's barriers at bar0 + g * group_bytes

  // ---- one-time setup: barriers, TMEM, resident weights ------------------------------------
  if (threadIdx.x == 0) {
    for (int g = 0; g < kGroups; ++g) {
      const uint32_t b = bar0 + (uint32_t)g * o.group_bytes;
      mbar_init(b + kBarFullX, kGroupThreads / 32 - (g == 0 ? 1 : 0));     // group 0 lends a warp to the issue loop
      mbar_init(b + kBarFullH1, kGroupThreads / 32 - (g == 0 ? 1 : 0));
      mbar_init(b + kBarL1Done, 1);
      mbar_init(b + kBarL2Done, 1);
      mbar_init(b + kBarL2Done + 8, 1);
    }
    mbar_init(smem_u32(tmem_slot) + 8u, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    bulk_load_weights(smem_u32(tmem_slot) + 8u, smem_u32(smem), a.packed, o.packed_end);
  }
  if (threadIdx.x < 32) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // crl_encoder_forward launches the head kernel with programmatic stream serialization: its CTAs may take over an SM the
  // moment this kernel's CTA there has exited (set up their barriers, TMEM and weights), and wait for the whole grid
  // -- griddepcontrol.wait -- only before they touch the operand images this kernel writes
  if (XHEAD) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // instruction descriptors: D fp32, A and B bf16, M = 128, N = 128; layer 1: both K-major; layer 2: B MN-major
  const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kRows >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t idesc2 = idesc1 | (1u << 16);
  const int tile_stride = kGroups * gridDim.x;
  bool healthy = true;

  if (issuer) {
    // ================= the issuing warp feeds the tensor pipe for both slots =================
    // All 32 lanes run this code CONVERGED and every value in it is warp-uniform (kernel parameters, blockIdx, vote
    // results), so the descriptors live in uniform registers; only the tcgen05 instructions themselves are executed by
    // one elected lane.  (The first version ran the loop in a single thread: ptxas then keeps everything in vector
    // registers, and each MMA cost six R2UR moves, a waterfall loop and ~100 instructions -- 300 cycles per MMA against
    // the 64 the tensor pipe needs; profiles/r02_notes.md.)
    const uint32_t tm = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t w1_addr = smem_u32(smem + o.w1), w2_addr = smem_u32(smem + o.w2);
    const uint32_t slot0 = smem_u32(smem + o.group0);
    const int n_s = KP / 16;
    const bool leader = elect_one();                          // the same lane issues every MMA and commit
    int n[kGroups], l1i[kGroups] = {0, 0}, l2i[kGroups] = {0, 0};
    for (int g = 0; g < kGroups; ++g) {
      const int first = kGroups * (int)blockIdx.x + g;
      n[g] = first < a.n_tiles ? (a.n_tiles - first + tile_stride - 1) / tile_stride : 0;
    }
    healthy = mbar_wait(smem_u32(tmem_slot) + 8u, 0u) && healthy;     // the resident weights have landed
    __syncwarp();
    // descriptors differ between MMAs only in their start-address field (bits 0..13, in 16-byte units)
    const uint64_t a1_desc = smem_desc(w1_addr, 128u, 16 * kK1), a2_desc = smem_desc(w2_addr, 128u, 16 * KP);
    const uint64_t x_desc = smem_desc(slot0 + o.xbuf, 128u, 16 * kK1), h1_desc = smem_desc(slot0 + o.h1, 2048u, 128u);
    const uint32_t slot_units = o.group_bytes >> 4;
    auto ready = [&](uint32_t bar, uint32_t parity) {          // warp-uniform poll
      return __shfl_sync(0xffffffffu, (int)mbar_test(bar, parity), 0) != 0;
    };
    // layer 1 of slot g's next tile: H1^T[128 b ..][m] = W1[128 b ..][kK1] X^T
    auto issue_l1 = [&](int g) {
      const uint32_t bars = bar0 + (uint32_t)g * o.group_bytes;
      healthy = mbar_wait(bars + kBarFullX, (uint32_t)l1i[g] & 1u) && healthy;
      __syncwarp();
      tc_fence_after();
      for (int b = 0; b < n_mblocks; ++b)
        for (int s2 = 0; s2 < kK1 / 16; ++s2) {
          const uint64_t ad = a1_desc + (uint64_t)(uint32_t)(b * 16 * kK1 + 16 * s2);
          const uint64_t bd = x_desc + (uint64_t)((uint32_t)g * slot_units + 16u * (uint32_t)s2);
          if (leader) mma_bf16(tm + (uint32_t)(g * 256 + b * 128), ad, bd, idesc1, s2 > 0);
        }
      if (leader) mma_commit(bars + kBarL1Done);
      CRL_TL(g, l1i[g], 0);                                    // layer 1 issued
      ++l1i[g];
    };
    // K steps [s_from, s_to) of M-block b of slot g's layer 2: H2^T[128 b ..][m] = W2[128 b ..][KP] H1^T
    auto issue_l2 = [&](int g, int b, int s_from, int s_to) {
      const uint32_t acc = tm + (uint32_t)(g * 256 + b * 128);
      uint64_t ad = a2_desc + (uint64_t)(uint32_t)(b * 16 * KP + 16 * s_from);
      uint64_t bd = h1_desc + (uint64_t)((uint32_t)g * slot_units + 256u * (uint32_t)s_from);
#pragma unroll 4
      for (int s2 = s_from; s2 < s_to; ++s2, ad += 16u, bd += 256u)
        if (leader) mma_bf16(acc, ad, bd, idesc2, s2 > 0);
      if (s_from < s_to && s_to == n_s && leader) mma_commit(bar0 + (uint32_t)g * o.group_bytes + kBarL2Done + 8u * (uint32_t)b);
    };
    for (int k = 0; k < n[0]; ++k) {
      for (int g = 0; g < kGroups; ++g) {
        if (k >= n[g]) continue;
        if (l1i[g] <= k) issue_l1(g);                         // the first tile; a CTA whose other slot has no tiles
        const int og = g ^ 1;
        const uint32_t bars = bar0 + (uint32_t)g * o.group_bytes, obars = bar0 + (uint32_t)og * o.group_bytes;
        // the other slot's next L1 rides inside this L2 -- unless that slot still owes the L2 before it
        bool need = l1i[og] < n[og] && l1i[og] <= l2i[og];
        for (uint32_t it = 0;; ++it) {                         // wait for H1 of (g, k); meanwhile serve the other slot
          if (need && ready(obars + kBarFullX, (uint32_t)l1i[og] & 1u)) { issue_l1(og); need = false; }
          if (ready(bars + kBarFullH1, (uint32_t)k & 1u)) break;
          if (it >= kSpinLimit) { healthy = false; break; }
        }
        tc_fence_after();
        CRL_TL(g, k, 1);                                       // H1 seen by the issuer
        int done = 0;
        if (need) {                                            // the insert point: inside M-block 0
          done = n_s < CRL_ENC_INSERT_AFTER ? n_s : CRL_ENC_INSERT_AFTER;
          issue_l2(g, 0, 0, done);
          issue_l1(og);                                        // blocks until that slot's epilogue 2 is over
        }
        issue_l2(g, 0, done, n_s);
        for (int b = 1; b < n_mblocks; ++b) issue_l2(g, b, 0, n_s);
        CRL_TL(g, k, 2);                                       // layer 2 issued
        ++l2i[g];
      }
    }
  } else {
    // ================= the two groups: stage X, epilogue 1 (-> H1), epilogue 2 (-> pooled) =================
    const uint32_t bars = bar0 + (uint32_t)group * o.group_bytes;
    const uint32_t my_acc = tmem_base + (uint32_t)group * 256u + (uint32_t)(mblock * 128) + ((uint32_t)(quad * 32) << 16);
    uint8_t* h1buf = gbase + o.h1;
    uint8_t* xbuf = gbase + o.xbuf;
    const uint32_t x_off = (uint32_t)((m & 7) * 16 + (m >> 3) * (16 * kK1) + half * 128);
    const uint32_t h1_off = (uint32_t)((j & 7) * 16 + (j >> 3) * 2048);
    const bool drains1 = mblock < n_mblocks && j0 < KP;       // layer 2 reads hidden rows < KP
    const uint32_t l2_bar = bars + kBarL2Done + 8u * (uint32_t)(mblock < n_mblocks ? mblock : n_mblocks - 1);
    const float inv_n = 1.0f / (float)a.N;
    const int log2_s = a.S == 16 ? 4 : 3, per_chunk = 32 >> log2_s;   // envs per 32 accumulator columns (a runtime
    int tile = kGroups * blockIdx.x + group;                           // division here cost epilogue 2 ~800 cycles per tile)
    float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, x2[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // 16-byte units `half` and, for 32-wide inputs, `half + 2`
    // group 0's warp 5 also stages the rows of warp 4 (the issuing warp): rows m - 32, same half
    const bool dual = group == 0 && warp == kIssuerWarp + 1;
    float y[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, y2[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int md = m - 32;
    const uint32_t y_off = (uint32_t)((md & 7) * 16 + (md >> 3) * (16 * kK1) + half * 128);
    auto stage_x = [&](int tl) {                               // this thread's part of the slot's layer-1 B operand
      const uint4 xv = make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
      *reinterpret_cast<uint4*>(xbuf + x_off) = xv;
      if (dual) {
        *reinterpret_cast<uint4*>(xbuf + y_off) =
            make_uint4(pack_bf16(y[0], y[1]), pack_bf16(y[2], y[3]), pack_bf16(y[4], y[5]), pack_bf16(y[6], y[7]));
        if (WIDE)
          *reinterpret_cast<uint4*>(xbuf + y_off + 256) =
              make_uint4(pack_bf16(y2[0], y2[1]), pack_bf16(y2[2], y2[3]), pack_bf16(y2[4], y2[5]), pack_bf16(y2[6], y2[7]));
      }
      if (XHEAD) {
        // an env's first row: its obs chunk (half 0: the same eight bf16 values) and its ones / zero padding behind the
        // pooled units (half 1) go into the head operand image
        auto image_row = [&](int mr, const uint4& v) {
          if ((mr & (a.S - 1)) != 0) return;
          const int e = (tl << (7 - (a.S == 16 ? 4 : 3))) + (mr >> (a.S == 16 ? 4 : 3));
          if (tl >= a.n_tiles || e >= a.B) return;
          const int mh = e & (kRows - 1);
          uint8_t* row = a.xhead + (size_t)(e >> 7) * (size_t)(kRows * a.KH * 2) + (uint32_t)((mh & 7) * 16 + (mh >> 3) * (16 * a.KH));
          if (half == 0) {
            *reinterpret_cast<uint4*>(row) = v;
          } else {
            for (int k = 8 + a.h; k < a.KH; ++k)
              *reinterpret_cast<__nv_bfloat16*>(row + (uint32_t)((k >> 3) * 128 + (k & 7) * 2)) =
                  __float2bfloat16_rn(k <= 8 + a.h + 1 ? 1.f : 0.f);
          }
        };
        image_row(m, xv);
        if (dual) image_row(md, xv);                           // (half 1: the value is not used)
      }
      if (WIDE)
        *reinterpret_cast<uint4*>(xbuf + x_off + 256) =
            make_uint4(pack_bf16(x2[0], x2[1]), pack_bf16(x2[2], x2[3]), pack_bf16(x2[4], x2[5]), pack_bf16(x2[6], x2[7]));
      fence_async_smem();
    };
    auto fetch_x = [&](int tl) {
      load_half_row<SRC>(a, tl, m, half, x);
      if (WIDE) load_half_row<SRC>(a, tl, m, half + 2, x2);
      if (dual) {
        load_half_row<SRC>(a, tl, md, half, y);
        if (WIDE) load_half_row<SRC>(a, tl, md, half + 2, y2);
      }
    };
    fetch_x(tile);
    stage_x(tile);
    __syncwarp();
    if (lane == 0) mbar_arrive(bars + kBarFullX);
    fetch_x(tile + tile_stride);                               // in flight until the first epilogue 1 is over
    uint32_t parity = 0u;
    for (int k = 0; tile < a.n_tiles; tile += tile_stride, parity ^= 1u, ++k) {
      // ---- epilogue 1: hidden unit j, rows m = 32 c .. 32 c + 31 -> relu -> bf16 -> four 16-byte units of H1 ----
      healthy = mbar_wait(bars + kBarL1Done, parity) && healthy;
      tc_fence_after();
      if (t == 0) CRL_TL(group, k, 3);                         // layer 1 done, seen by warp 0
      if (drains1) {
#ifdef CRL_ENC_DIAG_HALF_DRAIN                                // timing diagnostic (wrong results): half of epilogue 1's TMEM reads
        const int c_stop = kRows / 64;
#else
        const int c_stop = kRows / 32;
#endif
#pragma unroll 1
        for (int c = 0; c < c_stop; c += 2) {                 // two TMEM loads in flight
          uint32_t v0[32], v1[32];
          tmem_ld32(my_acc + (uint32_t)(c * 32), v0);
          tmem_ld32(my_acc + (uint32_t)(c * 32 + 32), v1);
          tmem_ld_wait(v0);
          relu_to_h1(v0, h1buf + h1_off, c, j < KP);
          tmem_ld_wait(v1);
          relu_to_h1(v1, h1buf + h1_off, c + 1, j < KP);
        }
      }
      fence_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + kBarFullH1);
      if (t == 0) CRL_TL(group, k, 4);                         // epilogue 1 over (warp 0)
      // ---- the next tile's input rows (layer 1 of this tile has completed: the X buffer is free) ----
      stage_x(tile + tile_stride);
      fetch_x(tile + 2 * tile_stride);
      // ---- epilogue 2: ReLU, mean over each env's zone slots (register adds), coalesced stores ----
      if (t == 0) CRL_TL(group, k, 5);                         // next rows staged (warp 0)
      if (XHEAD) {
      // (the image-writing variants keep one warp per (M-block, quadrant): their 16-byte stores want all 8 envs of a unit
      // group in one warp; with the column split below they measured 16 % slower)
      const bool drains2 = mblock < n_mblocks && j0 < a.h;      // the output has h columns
      float* const out_col = a.out + j;
      uint8_t* const xh_unit = a.xhead + (uint32_t)(((8 + j) >> 3) * 128 + ((8 + j) & 7) * 2);   // column 8 + j of an image row
      healthy = mbar_wait(l2_bar, parity) && healthy;
      tc_fence_after();
      if (t == 0) CRL_TL(group, k, 6);                         // layer 2 (M-block 0) done, seen by warp 0
      if (drains2) {
        const bool full = j < a.h && ((tile + 1) << (7 - log2_s)) <= a.B;
        // the image row of the tile's first env (its 8 / 16 envs share a head tile and start an 8-row group)
        const int et = tile << (7 - log2_s);
        uint8_t* const xh_tile = XHEAD ? xh_unit + (size_t)(et >> 7) * (size_t)(kRows * a.KH * 2) + (uint32_t)(((et & (kRows - 1)) >> 3) * (16 * a.KH))
                                       : nullptr;
        if (XHEAD && a.S == 16) {
          // 16 zone slots per env: the tile is 8 envs = ONE 8-row group of the head image.  Collect the eight pooled
          // values of this thread's unit, transpose 8 x 8 inside each group of 8 lanes (lane r then holds units
          // 8 g .. 8 g + 7 of env r) and write ONE 16-byte piece per lane instead of eight 2-byte ones.
          float pv[8];
#pragma unroll
          for (int c = 0; c < kRows / 32; c += 2) {
            uint32_t v0[32], v1[32];
            tmem_ld32(my_acc + (uint32_t)(c * 32), v0);
            tmem_ld32(my_acc + (uint32_t)(c * 32 + 32), v1);
            tmem_ld_wait(v0);
            relu_pool16(v0, inv_n, pv[2 * c], pv[2 * c + 1]);
            tmem_ld_wait(v1);
            relu_pool16(v1, inv_n, pv[2 * c + 2], pv[2 * c + 3]);
          }
          // units >= h of the image row: the head's ones (h, h + 1), then zeros
#pragma unroll
          for (int i = 0; i < 8; ++i) pv[i] = j < a.h ? pv[i] : (j <= a.h + 1 ? 1.f : 0.f);
          transpose8(pv, lane);
          const int r = lane & 7;
          if (et + r < a.B && ((8 + j) >> 3) < (a.KH >> 3))     // (a warp's last 8-unit groups can lie beyond the image's width)
            *reinterpret_cast<uint4*>(xh_tile - (uint32_t)(((8 + j) & 7) * 2) + (uint32_t)(r * 16)) =      // chunk (8 + j) / 8, row r
                make_uint4(pack_bf16(pv[0], pv[1]), pack_bf16(pv[2], pv[3]), pack_bf16(pv[4], pv[5]), pack_bf16(pv[6], pv[7]));
        } else
#pragma unroll 1
        for (int c = 0; c < kRows / 32; c += 2) {             // two TMEM loads in flight
          uint32_t v0[32], v1[32];
          tmem_ld32(my_acc + (uint32_t)(c * 32), v0);
          tmem_ld32(my_acc + (uint32_t)(c * 32 + 32), v1);
          tmem_ld_wait(v0);
          if (t == 0) CRL_TL(group, k, 8 + 2 * c);               // 8 / 12: a pair of TMEM loads has arrived
          const int e0 = (tile << (7 - log2_s)) + c * per_chunk;
          relu_pool_store<XHEAD>(v0, out_col, a.h, a.B, a.S, e0, full, j < a.h, inv_n, xh_tile, a.KH);
          tmem_ld_wait(v1);
          relu_pool_store<XHEAD>(v1, out_col, a.h, a.B, a.S, e0 + per_chunk, full, j < a.h, inv_n, xh_tile, a.KH);
          if (t == 0) CRL_TL(group, k, 9 + 2 * c);               // 9 / 13: pooled and stored
        }
      }
      } else {
      // Who drains what: in lane quadrants 0, 1 only M-block 0 has rows, and its warp takes all 128 columns; in quadrants
      // 2, 3 BOTH M-blocks have rows and the quadrant's two warps split the COLUMNS of both (warp w / 4 takes half w / 4):
      // M-block 0 completes 12 MMAs before M-block 1, so this way both warps work on it at once and the tail after the
      // last MMA is half of M-block 1, not all of it.
      bool waited = false;
#pragma unroll 1
      for (int b = 0; b < n_mblocks; ++b) {
        const bool split = quad >= 2;
        const bool mine = split ? true : (mblock == 0 && b == 0);
        const int jb0 = b == 0 ? quad * 32 : 128 + (quad - 2) * 32, jb = jb0 + lane;   // this thread's unit in M-block b
        if (!mine || jb0 >= a.h) continue;                     // the output has h columns
        healthy = mbar_wait(bars + kBarL2Done + 8u * (uint32_t)b, parity) && healthy;
        tc_fence_after();
        waited = true;
        if (t == 0 && b == 0) CRL_TL(group, k, 6);             // layer 2 (M-block 0) done, seen by warp 0
        const int c_lo = split ? 2 * mblock : 0, c_hi = split ? c_lo + 2 : kRows / 32;   // 32-column chunks
        const uint32_t acc_b = tmem_base + (uint32_t)group * 256u + (uint32_t)(b * 128) + ((uint32_t)(quad * 32) << 16);
        const bool full = jb < a.h && ((tile + 1) << (7 - log2_s)) <= a.B;
        // the image row of the tile's first env (its 8 / 16 envs share a head tile and start an 8-row group)
        const int et = tile << (7 - log2_s);
        uint8_t* const xh_tile = XHEAD ? a.xhead + (uint32_t)(((8 + jb) >> 3) * 128 + ((8 + jb) & 7) * 2) +
                                             (size_t)(et >> 7) * (size_t)(kRows * a.KH * 2) + (uint32_t)(((et & (kRows - 1)) >> 3) * (16 * a.KH))
                                       : nullptr;
        float* const out_b = a.out + jb;
        if (XHEAD && a.S == 16) {
          // 16 zone slots per env: the tile is 8 envs = ONE 8-row group of the head image.  Collect the pooled values of
          // this thread's unit (envs 2 c, 2 c + 1 from chunk c; zeros for the chunks of the other warp), transpose 8 x 8
          // inside each group of 8 lanes (lane r then holds units 8 g .. 8 g + 7 of env r) and write ONE 16-byte piece per
          // lane and env of this warp's columns instead of eight 2-byte ones.
          float pv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int c = 0; c < kRows / 32; c += 2) {
            if (c < c_lo || c >= c_hi) continue;
            uint32_t v0[32], v1[32];
            tmem_ld32(acc_b + (uint32_t)(c * 32), v0);
            tmem_ld32(acc_b + (uint32_t)(c * 32 + 32), v1);
            tmem_ld_wait(v0);
            relu_pool16(v0, inv_n, pv[2 * c], pv[2 * c + 1]);
            tmem_ld_wait(v1);
            relu_pool16(v1, inv_n, pv[2 * c + 2], pv[2 * c + 3]);
          }
          // units >= h of the image row: the head's ones (h, h + 1), then zeros
#pragma unroll
          for (int i = 0; i < 8; ++i) pv[i] = jb < a.h ? pv[i] : (jb <= a.h + 1 ? 1.f : 0.f);
          transpose8(pv, lane);
          const int r = lane & 7;                              // the env of the tile this lane now holds
          if (r >= 2 * c_lo && r < 2 * c_hi && et + r < a.B && ((8 + jb) >> 3) < (a.KH >> 3))
            *reinterpret_cast<uint4*>(xh_tile - (uint32_t)(((8 + jb) & 7) * 2) + (uint32_t)(r * 16)) =      // chunk (8 + jb) / 8, row r
                make_uint4(pack_bf16(pv[0], pv[1]), pack_bf16(pv[2], pv[3]), pack_bf16(pv[4], pv[5]), pack_bf16(pv[6], pv[7]));
        } else {
#pragma unroll 1
          for (int c = c_lo; c < c_hi; c += 2) {               // two TMEM loads in flight
            uint32_t v0[32], v1[32];
            tmem_ld32(acc_b + (uint32_t)(c * 32), v0);
            tmem_ld32(acc_b + (uint32_t)(c * 32 + 32), v1);
            tmem_ld_wait(v0);
            if (t == 0) CRL_TL(group, k, 8 + 2 * c);             // 8 / 12: a pair of TMEM loads has arrived
            const int e0 = (tile << (7 - log2_s)) + c * per_chunk;
            relu_pool_store<XHEAD>(v0, out_b, a.h, a.B, a.S, e0, full, jb < a.h, inv_n, xh_tile, a.KH);
            tmem_ld_wait(v1);
            relu_pool_store<XHEAD>(v1, out_b, a.h, a.B, a.S, e0 + per_chunk, full, jb < a.h, inv_n, xh_tile, a.KH);
            if (t == 0) CRL_TL(group, k, 9 + 2 * c);             // 9 / 13: pooled and stored
          }
        }
      }
      if (!waited) {                                           // a warp without rows still orders itself behind layer 2
        healthy = mbar_wait(l2_bar, parity) && healthy;
        tc_fence_after();
      }
      }
      // accumulators drained + next rows staged: the issuer may overwrite both with the slot's next layer 1
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + kBarFullX);
      if (t == 0) CRL_TL(group, k, 7);                         // epilogue 2 over (warp 0)
    }
  }
  if (!healthy && a.status) atomicExch(a.status, 1);
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ---- the head: forward() = combine_net_([obs, L3(pooled)]) (env_model.py:79) as ONE more tcgen05 GEMM ----------
// Both Linears are affine, so  out[e] = Wc [obs[e], W3 pooled[e] + b3] + bc = W' [obs[e], pooled[e], 1, 1]  with
// W' = [Wc_obs | Wc_emb W3 | bias hi | bias lo] folded once on the host side (encoder.py).  The same transposed
// formulation as above: out^T[j][e] = W'[j][:] X^T, the folded weights resident in shared memory as the A operand
// (M = output units in blocks of 128 = TMEM lanes), a tile of 128 ENVS the N dimension, K = obs_dim + h + 2 padded to
// 16.  After tcgen05.ld lane j holds unit j of 32 consecutive envs: 32 coalesced 128-byte stores per load.  4.7 GFLOP
// at 65,536 envs and h = 185: the kernel is bound by reading (obs, pooled) and writing out once (~100 MB), not by the
// tensor pipe -- the library fp32 GEMM it replaces took longer than the whole fused zone kernel (profiles/r01_notes.md).
__host__ __device__ inline int head_k(int obs_dim, int h) { return (obs_dim + h + 2 + 15) & ~15; }

struct HeadOffsets { uint32_t w, packed_end, group0, xbuf, bar, group_bytes, tmem_slot, smem_end; };
__host__ __device__ inline HeadOffsets head_offsets(int obs_dim, int h) {
  const int KH = head_k(obs_dim, h), MP = padded_m(h);
  HeadOffsets o;
  o.w = 0;
  o.packed_end = (uint32_t)MP * KH * 2;
  o.group0 = (o.packed_end + 127u) & ~127u;
  o.xbuf = 0;
  o.bar = (uint32_t)kRows * KH * 2;                      // + 8: the mbarrier of the tile's bulk copy (PACKED)
  o.group_bytes = (o.bar + 16 + 127u) & ~127u;
  o.tmem_slot = o.group0 + kGroups * o.group_bytes;
  o.smem_end = o.tmem_slot + 16;
  return o;
}

struct HeadPackArgs { const float *w, *b; uint8_t* out; int obs_dim, h; };

// W' rows n < h: [w[n][0 .. obs_dim + h), bf16(b[n]), b[n] - bf16(b[n]), 0...]; rows >= h: zeros
__global__ void head_pack_kernel(const HeadPackArgs a) {
  const int KH = head_k(a.obs_dim, a.h), MP = padded_m(a.h), in = a.obs_dim + a.h;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < MP * KH; i += gridDim.x * blockDim.x) {
    const int n = i / KH, k = i % KH;
    float v = 0.f;
    if (n < a.h) {
      if (k < in) v = a.w[(size_t)n * in + k];
      else if (k == in) v = __bfloat162float(__float2bfloat16_rn(a.b[n]));
      else if (k == in + 1) v = a.b[n] - __bfloat162float(__float2bfloat16_rn(a.b[n]));
    }
    *reinterpret_cast<__nv_bfloat16*>(a.out + canon(n, k, KH)) = __float2bfloat16_rn(v);
  }
}

struct HeadArgs {
  const float* obs;      // [B][obs_dim]
  const float* pooled;   // [B][h]
  const uint8_t* packed;
  float* out;            // [B][h]
  int* status;
  int B, obs_dim, h, n_tiles;
  const uint8_t* xhead;  // PACKED: the operand images the zone kernel wrote (crl_encoder_forward); obs / pooled unused
};

// unit j of 32 consecutive envs e0 ..: one base pointer, constant strides; predicates only on the batch's last tile
__device__ __forceinline__ void head_store(const uint32_t (&v)[32], float* col, int h, int B, int e0, bool j_ok) {
  if (!j_ok) return;
  float* p = col + (size_t)e0 * (size_t)h;
  if (e0 + 32 <= B) {
#pragma unroll
    for (int i = 0; i < 32; ++i) p[(size_t)i * h] = __uint_as_float(v[i]);
  } else {
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (e0 + i < B) p[(size_t)i * h] = __uint_as_float(v[i]);
  }
}

template <bool PACKED>
__global__ void __launch_bounds__(kGroupThreads * kGroups, 1) encoder_head_kernel(const HeadArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const HeadOffsets o = head_offsets(a.obs_dim, a.h);
  const int KH = head_k(a.obs_dim, a.h), MP = padded_m(a.h), in = a.obs_dim + a.h;
  const int n_mblocks = MP / 128, chunks = KH / 8;
  const int group = threadIdx.x / kGroupThreads, t = threadIdx.x % kGroupThreads;
  const int warp = t >> 5, lane = t & 31, mblock = warp >> 2, quad = warp & 3;
  const int j = mblock * 128 + quad * 32 + lane;              // output unit (accumulator row) of this thread
  uint8_t* gbase = smem + o.group0 + (uint32_t)group * o.group_bytes;
  uint8_t* xbuf = gbase + o.xbuf;
  uint64_t* bar = reinterpret_cast<uint64_t*>(gbase + o.bar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + o.tmem_slot);
  const uint32_t bar_addr = smem_u32(bar);
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar_addr) : "memory");
    mbar_init(bar_addr + 8u, 1);
    if (group == 0) mbar_init(smem_u32(tmem_slot) + 8u, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (group == 0) bulk_load_weights(smem_u32(tmem_slot) + 8u, smem_u32(smem), a.packed, o.packed_end);
  }
  if (threadIdx.x < 32) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t acc = tmem_base + (uint32_t)group * 256u;
  const uint32_t my_acc = acc + (uint32_t)(mblock * 128) + ((uint32_t)(quad * 32) << 16);
  const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kRows >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  bool weights_in = false;
  const uint32_t tile_bytes = (uint32_t)(kRows * KH * 2);
  uint32_t xparity = 0u;
  if (PACKED) asm volatile("griddepcontrol.wait;" ::: "memory");   // the zone kernel's images are complete and visible
  if (PACKED && t == 0) {                                      // the first tile's operand image: one bulk copy
    const int tile0 = kGroups * blockIdx.x + group;
    if (tile0 < a.n_tiles) bulk_load_weights(bar_addr + 8u, smem_u32(xbuf), a.xhead + (size_t)tile0 * tile_bytes, tile_bytes);
  }
  const uint32_t x_addr = smem_u32(xbuf), w_addr = smem_u32(smem + o.w);
  const bool drains = mblock < n_mblocks && mblock * 128 + quad * 32 < a.h;
  uint32_t parity = 0u;
  bool healthy = true;
  for (int tile = kGroups * blockIdx.x + group; tile < a.n_tiles; tile += kGroups * gridDim.x) {
    // ---- B operand: the tile's 128 rows [obs, pooled, 1, 1, 0..] as bf16, K-major.
    if (PACKED) {
      // already in shared memory, or on its way (issued a tile ago); only the MMA-issuing thread waits for it
    } else if (a.obs_dim == 8 && chunks <= 32) {
      // ZoneEnvModel's shape: chunk 0 of a row is exactly obs[e] (two 16-byte loads), chunk c >= 1 is
      // pooled[e][8 (c - 1) ..].  A warp takes a row at a time, lane c its chunk c -- no index arithmetic, no address
      // selects (the general loop below spends ~10 instructions per element on them) -- four rows per iteration so that
      // 32 loads per lane are in flight.
#pragma unroll 1
      for (int m0 = warp; m0 < kRows; m0 += 4 * (kGroupThreads / 32)) {
        float x[4][8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + i * (kGroupThreads / 32), e = tile * kRows + m;
          const size_t e_ok = (size_t)(e < a.B ? e : 0);
          if (lane == 0) {
            const float4 lo = __ldg(reinterpret_cast<const float4*>(a.obs + e_ok * 8));
            const float4 hi = __ldg(reinterpret_cast<const float4*>(a.obs + e_ok * 8) + 1);
            x[i][0] = lo.x; x[i][1] = lo.y; x[i][2] = lo.z; x[i][3] = lo.w;
            x[i][4] = hi.x; x[i][5] = hi.y; x[i][6] = hi.z; x[i][7] = hi.w;
          } else {
            const float* src = a.pooled + e_ok * a.h;
            const int k0 = 8 * (lane - 1);
#pragma unroll
            for (int q = 0; q < 8; ++q) x[i][q] = __ldg(src + (k0 + q < a.h ? k0 + q : 0));
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + i * (kGroupThreads / 32), e = tile * kRows + m;
          if (lane >= chunks) continue;
          if (lane > 0) {
            const int k0 = 8 * (lane - 1);
#pragma unroll
            for (int q = 0; q < 8; ++q) x[i][q] = k0 + q < a.h ? x[i][q] : (k0 + q <= a.h + 1 ? 1.f : 0.f);
          }
          if (e >= a.B) {
#pragma unroll
            for (int q = 0; q < 8; ++q) x[i][q] = 0.f;
          }
          *reinterpret_cast<uint4*>(xbuf + (uint32_t)((m & 7) * 16 + (m >> 3) * (16 * KH) + lane * 128)) =
              make_uint4(pack_bf16(x[i][0], x[i][1]), pack_bf16(x[i][2], x[i][3]), pack_bf16(x[i][4], x[i][5]),
                         pack_bf16(x[i][6], x[i][7]));
        }
      }
    } else
    // the general shape (per-env features wider than 8: ZoneEnvGoalModel / ZoneEnvSkillModel): consecutive threads take

    // consecutive 8-value chunks of one env (coalesced reads); a row beyond the batch is all zeros.  Four chunks
    // per iteration with UNCONDITIONAL loads from clamped addresses (the selects come after), so that 32 loads
    // are in flight per thread: this kernel is bound by how fast it reads (obs, pooled), not by the tensor pipe.
    for (int u0 = t; u0 < kRows * chunks; u0 += 4 * kGroupThreads) {
      float x[4][8];
      int mm[4], cc[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int u = u0 + i * kGroupThreads;
        const int m = u / chunks, c = u - m * chunks, e = tile * kRows + m;
        mm[i] = m; cc[i] = u < kRows * chunks ? c : -1;
        const size_t e_ok = (size_t)(e < a.B ? e : 0);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int k = 8 * c + q;
          const float* src = k < a.obs_dim ? a.obs + e_ok * a.obs_dim + k
                                           : a.pooled + e_ok * a.h + (k < in ? k - a.obs_dim : 0);
          x[i][q] = __ldg(src);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (cc[i] < 0) continue;
        const int e = tile * kRows + mm[i];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int k = 8 * cc[i] + q;
          x[i][q] = e < a.B ? (k < in ? x[i][q] : (k <= in + 1 ? 1.f : 0.f)) : 0.f;
        }
        *reinterpret_cast<uint4*>(xbuf + (uint32_t)((mm[i] & 7) * 16 + (mm[i] >> 3) * (16 * KH) + cc[i] * 128)) =
            make_uint4(pack_bf16(x[i][0], x[i][1]), pack_bf16(x[i][2], x[i][3]), pack_bf16(x[i][4], x[i][5]),
                       pack_bf16(x[i][6], x[i][7]));
      }
    }
    fence_async_smem();
    tc_fence_before();
    group_sync(group);
    if (t == 0) {
      if (!weights_in) { weights_in = true; healthy = mbar_wait(smem_u32(tmem_slot) + 8u, 0u) && healthy; }
      if (PACKED) { healthy = mbar_wait(bar_addr + 8u, xparity) && healthy; xparity ^= 1u; }
      tc_fence_after();
      for (int b = 0; b < n_mblocks; ++b)
        for (int s = 0; s < KH / 16; ++s)
          mma_bf16(acc + (uint32_t)(b * 128), smem_desc(w_addr + (uint32_t)(b * 16 * 16 * KH) + 256u * s, 128u, 16 * KH),
                   smem_desc(x_addr + 256u * s, 128u, 16 * KH), idesc, s > 0);
      mma_commit(bar_addr);
    }
    healthy = mbar_wait(bar_addr, parity) && healthy;
    parity ^= 1u;
    tc_fence_after();
    if (PACKED && t == 0) {                                    // the MMAs have read the operand buffer: fetch the next image
      const int next = tile + kGroups * (int)gridDim.x;       // under this tile's epilogue
      if (next < a.n_tiles) bulk_load_weights(bar_addr + 8u, smem_u32(xbuf), a.xhead + (size_t)next * tile_bytes, tile_bytes);
    }
    if (drains) {
#pragma unroll 1
      for (int c = 0; c < kRows / 32; c += 2) {               // two TMEM loads in flight
        uint32_t v0[32], v1[32];
        tmem_ld32(my_acc + (uint32_t)(c * 32), v0);
        tmem_ld32(my_acc + (uint32_t)(c * 32 + 32), v1);
        tmem_ld_wait(v0);
        head_store(v0, a.out + j, a.h, a.B, tile * kRows + c * 32, j < a.h);
        tmem_ld_wait(v1);
        head_store(v1, a.out + j, a.h, a.B, tile * kRows + (c + 1) * 32, j < a.h);
      }
    }
    // the next tile's MMAs overwrite the accumulators and the operand buffer: ordered after these loads by the
    // fence and the group barrier that precede them
    tc_fence_before();
  }
  if (!healthy && a.status) atomicExch(a.status, 1);
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ================= the PRECISE mode: the same two layers with fp32-level accuracy =================================
// The fast kernels multiply bf16-rounded operands (relative error 2^-9 per operand, 3-5e-3 of the largest output
// against the fp32 reference module).  Here every operand is split into two bf16 terms, x = x_hi + x_lo (residual
// 2^-18 |x|), and every product is three MMAs, W_hi X_hi + W_lo X_hi + W_hi X_lo (the dropped W_lo X_lo term is 2^-18
// relative), accumulated in fp32 in TMEM; the biases are added in fp32 in the epilogues.  Measured against the REAL
// module's fp32 output: <= 1e-4 of the largest value (tests/test_gpu_encode.py), i.e. like for like with the reference.
// Twice the operand bytes do not fit an SM beside a tile's activations, so a CTA holds ONE M-block of W2 (hi + lo,
// 96 KB) and computes that block's 128 output units for its tiles; layer 1 (all hidden units: they are layer 2's K)
// is computed by both CTAs of a pair -- it is 6 of 42 MMAs.  One tile in flight per CTA: this is the validation /
// like-for-like mode, ~7x the fast kernel's time (620 us at 65,536 PointTSP envs; torch fp32 eager: 7.3 ms).
__host__ __device__ inline int precise_k(int h) { return (h + 15) & ~15; }

struct PreciseOffsets {      // bytes; `g_*` in the packed global buffer, `s_*` in shared memory
  uint32_t g_w1, g_w2, g_w2_block, g_bias, g_end;
  uint32_t s_w1, s_w2, s_h1hi, s_h1lo, s_xhi, s_xlo, s_bar, s_wbar, s_tmem, s_end;
};
__host__ __device__ inline PreciseOffsets precise_offsets(int h) {
  const uint32_t KP = (uint32_t)precise_k(h), MP = (KP + 127u) & ~127u;
  PreciseOffsets o;
  o.g_w1 = 0;                                   // W1 hi | W1 lo: MP x 16 bf16 each
  o.g_w2 = 2u * MP * 16u * 2u;                  // per M-block: W2 hi | W2 lo, 128 x KP bf16 each
  o.g_w2_block = 2u * 128u * KP * 2u;
  o.g_bias = o.g_w2 + (MP / 128u) * o.g_w2_block;   // float b1[MP] | float b2[MP]
  o.g_end = o.g_bias + 2u * MP * 4u;
  o.s_w1 = 0;
  o.s_w2 = o.g_w2;
  o.s_h1hi = o.s_w2 + o.g_w2_block;
  o.s_h1lo = o.s_h1hi + KP * kRows * 2u;
  o.s_xhi = o.s_h1lo + KP * kRows * 2u;
  o.s_xlo = o.s_xhi + kRows * 16u * 2u;
  o.s_bar = o.s_xlo + kRows * 16u * 2u;
  o.s_wbar = o.s_bar + 8u;
  o.s_tmem = o.s_wbar + 8u;
  o.s_end = o.s_tmem + 16u;
  return o;
}

struct PrecisePackArgs { const float *w1, *b1, *w2, *b2; uint8_t* out; int in_dim, h; };

__global__ void pack_precise_kernel(const PrecisePackArgs a) {
  const PreciseOffsets o = precise_offsets(a.h);
  const int KP = precise_k(a.h), MP = (KP + 127) & ~127;
  const int n1 = MP * 16, n2 = MP * KP, total = n1 + n2 + 2 * MP;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    if (i >= n1 + n2) {                                        // biases, fp32
      const int r = i - n1 - n2, n = r % MP;
      reinterpret_cast<float*>(a.out + o.g_bias)[r] = n < a.h ? (r < MP ? a.b1[n] : a.b2[n]) : 0.f;
      continue;
    }
    const bool second = i >= n1;
    const int K = second ? KP : 16, lim = second ? a.h : a.in_dim;
    const int q = second ? i - n1 : i, n = q / K, k = q % K;
    const float v = (n < a.h && k < lim) ? (second ? a.w2[(size_t)n * a.h + k] : a.w1[(size_t)n * a.in_dim + k]) : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v), lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    uint8_t *phi, *plo;
    if (second) {
      uint8_t* blk = a.out + o.g_w2 + (uint32_t)(n >> 7) * o.g_w2_block;
      phi = blk + canon(n & 127, k, KP);
      plo = blk + 128u * KP * 2u + canon(n & 127, k, KP);
    } else {
      phi = a.out + o.g_w1 + canon(n, k, 16);
      plo = a.out + o.g_w1 + (uint32_t)MP * 32u + canon(n, k, 16);
    }
    *reinterpret_cast<__nv_bfloat16*>(phi) = hi;
    *reinterpret_cast<__nv_bfloat16*>(plo) = lo;
  }
}

__device__ __forceinline__ void split_bf16(float v, float& hi, float& lo) {
  hi = __bfloat162float(__float2bfloat16_rn(v));
  lo = v - hi;                                                 // exact; rounded to bf16 when packed
}

__global__ void __launch_bounds__(kGroupThreads, 1) zone_encode_precise_kernel(const EncArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const PreciseOffsets o = precise_offsets(a.h);
  const int KP = precise_k(a.h), MP = (KP + 127) & ~127, n_mblocks = MP / 128;
  const int t = threadIdx.x, lane = t & 31;
  const int warp = __shfl_sync(0xffffffffu, t >> 5, 0);       // warp-uniform, and the compiler knows it
  const bool leader = elect_one();                            // of each warp; warp 0's issues the MMAs
  const int m = t & (kRows - 1), half = t >> 7;
  const int my_block = (int)blockIdx.x % n_mblocks;            // the M-block of layer 2 this CTA owns
  const uint32_t bar = smem_u32(smem + o.s_bar), wbar = smem_u32(smem + o.s_wbar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + o.s_tmem);
  if (t == 0) {
    mbar_init(bar, 1);
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(wbar), "r"(o.g_w2 + o.g_w2_block) : "memory");
    const uint8_t* src2 = a.packed + o.g_w2 + (uint32_t)my_block * o.g_w2_block;
    for (uint32_t off = 0; off < o.g_w2; off += 16384u)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   :: "r"(smem_u32(smem + o.s_w1) + off), "l"(a.packed + off), "r"(o.g_w2 - off < 16384u ? o.g_w2 - off : 16384u), "r"(wbar) : "memory");
    for (uint32_t off = 0; off < o.g_w2_block; off += 16384u)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   :: "r"(smem_u32(smem + o.s_w2) + off), "l"(src2 + off), "r"(o.g_w2_block - off < 16384u ? o.g_w2_block - off : 16384u), "r"(wbar) : "memory");
  }
  if (t < 32) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t acc1 = tmem_base, acc2 = tmem_base + 256u;    // layer 1: two M-blocks x 128 columns; layer 2: one
  const uint32_t idesc1 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kRows >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t idesc2 = idesc1 | (1u << 16);
  const float* bias = reinterpret_cast<const float*>(a.packed + o.g_bias);
  // epilogue 1: warp = (M-block, lane quadrant) of layer 1's accumulators
  const int mb1 = warp >> 2, q1 = warp & 3, j1 = mb1 * 128 + q1 * 32 + lane;
  const bool drains1 = mb1 < n_mblocks && mb1 * 128 + q1 * 32 < KP;
  const float b1v = drains1 ? __ldg(bias + j1) : 0.f;
  // epilogue 2: warp = (lane quadrant, column half) of this CTA's layer-2 accumulators
  const int q2 = warp & 3, ch = warp >> 2, j2 = my_block * 128 + q2 * 32 + lane;
  const bool drains2 = my_block * 128 + q2 * 32 < a.h;
  const float b2v = j2 < a.h ? __ldg(bias + MP + j2) : 0.f;
  const float inv_n = 1.0f / (float)a.N;
  const int log2_s = a.S == 16 ? 4 : 3;
  uint32_t parity = 0u;
  bool healthy = true, weights_in = false;
  float x[8];
  load_half_row<kSrcZoneObs>(a, (int)blockIdx.x / n_mblocks, m, half, x);
  for (int tile = (int)blockIdx.x / n_mblocks; tile < a.n_tiles; tile += (int)gridDim.x / n_mblocks) {
    // ---- the tile's input rows (prefetched a tile ago), split ----
    float xh[8], xl[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) split_bf16(x[i], xh[i], xl[i]);
    const uint32_t x_off = (uint32_t)((m & 7) * 16 + (m >> 3) * 256 + half * 128);
    *reinterpret_cast<uint4*>(smem + o.s_xhi + x_off) =
        make_uint4(pack_bf16(xh[0], xh[1]), pack_bf16(xh[2], xh[3]), pack_bf16(xh[4], xh[5]), pack_bf16(xh[6], xh[7]));
    *reinterpret_cast<uint4*>(smem + o.s_xlo + x_off) =
        make_uint4(pack_bf16(xl[0], xl[1]), pack_bf16(xl[2], xl[3]), pack_bf16(xl[4], xl[5]), pack_bf16(xl[6], xl[7]));
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    load_half_row<kSrcZoneObs>(a, tile + (int)gridDim.x / n_mblocks, m, half, x);   // the next tile's rows travel under this tile
    // MMAs are issued by warp 0 with all its lanes CONVERGED (uniform descriptors; one elected lane executes the
    // tcgen05 instructions): from a single-thread branch every MMA costs ~300 cycles of issue (see zone_encode_kernel)
    if (warp == 0) {
      if (!weights_in) healthy = mbar_wait(wbar, 0u) && healthy;
      __syncwarp();
      tc_fence_after();
      const uint32_t tmu = __shfl_sync(0xffffffffu, acc1, 0);
      const uint32_t w1hi = smem_u32(smem + o.s_w1), w1lo = w1hi + (uint32_t)MP * 32u;
      const uint32_t xhi = smem_u32(smem + o.s_xhi), xlo = smem_u32(smem + o.s_xlo);
      for (int b = 0; b < n_mblocks; ++b) {
        const uint32_t d = tmu + (uint32_t)(b * 128), wo = (uint32_t)(b * 128 * 32);
        const uint64_t ahi = smem_desc(w1hi + wo, 128u, 256u), alo = smem_desc(w1lo + wo, 128u, 256u);
        const uint64_t bhi = smem_desc(xhi, 128u, 256u), blo = smem_desc(xlo, 128u, 256u);
        if (leader) mma_bf16(d, ahi, bhi, idesc1, 0u);
        if (leader) mma_bf16(d, alo, bhi, idesc1, 1u);
        if (leader) mma_bf16(d, ahi, blo, idesc1, 1u);
      }
      if (leader) mma_commit(bar);
    }
    weights_in = true;
    healthy = mbar_wait(bar, parity) && healthy;
    parity ^= 1u;
    tc_fence_after();
    // ---- epilogue 1: + bias, relu, split, two MN-major images of H1 ----
    if (drains1) {
      const uint32_t h1_off = (uint32_t)((j1 & 7) * 16 + (j1 >> 3) * 2048);
      const uint32_t my_acc = acc1 + (uint32_t)(mb1 * 128) + ((uint32_t)(q1 * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < kRows / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(my_acc + (uint32_t)(c * 32), v);
        tmem_ld_wait(v);
        if (j1 < KP) {
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            float hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) split_bf16(relu_nan(__uint_as_float(v[u * 8 + i]) + b1v), hi[i], lo[i]);
            const uint32_t at = h1_off + (uint32_t)((c * 4 + u) * 128);
            *reinterpret_cast<uint4*>(smem + o.s_h1hi + at) =
                make_uint4(pack_bf16(hi[0], hi[1]), pack_bf16(hi[2], hi[3]), pack_bf16(hi[4], hi[5]), pack_bf16(hi[6], hi[7]));
            *reinterpret_cast<uint4*>(smem + o.s_h1lo + at) =
                make_uint4(pack_bf16(lo[0], lo[1]), pack_bf16(lo[2], lo[3]), pack_bf16(lo[4], lo[5]), pack_bf16(lo[6], lo[7]));
          }
        }
      }
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    // ---- layer 2, this CTA's M-block: three MMAs per K step ----
    if (warp == 0) {
      tc_fence_after();
      const uint32_t d2 = __shfl_sync(0xffffffffu, acc2, 0);
      const uint32_t w2hi = smem_u32(smem + o.s_w2), w2lo = w2hi + 128u * (uint32_t)KP * 2u;
      const uint32_t hhi = smem_u32(smem + o.s_h1hi), hlo = smem_u32(smem + o.s_h1lo);
      uint64_t ahi = smem_desc(w2hi, 128u, 16 * KP), alo = smem_desc(w2lo, 128u, 16 * KP);
      uint64_t bhi = smem_desc(hhi, 2048u, 128u), blo = smem_desc(hlo, 2048u, 128u);
#pragma unroll 2
      for (int s2 = 0; s2 < KP / 16; ++s2, ahi += 16u, alo += 16u, bhi += 256u, blo += 256u) {
        if (leader) mma_bf16(d2, ahi, bhi, idesc2, s2 > 0);
        if (leader) mma_bf16(d2, alo, bhi, idesc2, 1u);
        if (leader) mma_bf16(d2, ahi, blo, idesc2, 1u);
      }
      if (leader) mma_commit(bar);
    }
    healthy = mbar_wait(bar, parity) && healthy;
    parity ^= 1u;
    tc_fence_after();
    // ---- epilogue 2: + bias, relu, mean over each env's REAL zone slots (a padding row is relu(bias) here, not 0) ----
    if (drains2) {
      const uint32_t my_acc = acc2 + ((uint32_t)(q2 * 32) << 16) + (uint32_t)(ch * 64);
#pragma unroll 1
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld32(my_acc + (uint32_t)(c * 32), v);
        tmem_ld_wait(v);
        const int row0 = ch * 64 + c * 32;                     // tile row of v[0]
        if (j2 < a.h) {
          float sum = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int slot = (row0 + i) & (a.S - 1);
            if (slot < a.N) sum += relu_nan(__uint_as_float(v[i]) + b2v);
            if (slot == a.S - 1) {
              const int e = (tile << (7 - log2_s)) + ((row0 + i) >> log2_s);
              if (e < a.B) a.out[(size_t)e * a.h + j2] = sum * inv_n;
              sum = 0.f;
            }
          }
        }
      }
    }
    tc_fence_before();       // the next tile's MMAs overwrite the accumulators after the barrier at the loop's top
  }
  if (!healthy && a.status) atomicExch(a.status, 1);
  tc_fence_before();
  __syncthreads();
  if (t < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
}

// ---- backward: dL/d(W1, b1, W2, b2) of pooled, given g = dL/dpooled (crl_zone_encode_backward) ------------------
// One persistent CTA per SM walks tiles of kBwdRows = 64 (env, zone-slot) rows (4 envs x 16 slots or 8 x 8; padding slots
// are all-zero rows as in the forward, so they contribute exact zeros) and, per tile, on the tensor cores:
//   L1   H1^T  = W1 X^T                 (recomputed exactly as the forward: same image, folded biases)  -> bf16 relu H1
//   L2   A2^T  = W2 H1^T                                                                                   -> dH2
//        dH2[m][i] = acc2 > 0 ? bf16(g[e(m)][i] * fp32(1/N)) : 0        (select: a masked NaN g gives 0)
//   dH1  D^T   = W2^T dH2^T             (the W2 image read through an MN-major descriptor)
//        dH1[m][j] = H1[m][j] > 0 ? bf16(D[m][j]) : 0                   (written over H1 in place)
//   dW2 += dH2^T H1   (M = W2 image row, N = H1 row incl. the ones row h: column h is db2)
//   dW1 += dH1^T X    (M = hidden unit, N = input column incl. the ones column in_dim: column in_dim is db1)
// dW2 / dW1 stay in TMEM for the CTA's whole life (2 x 192 + 2 x 32 columns); the per-tile accumulators take the last
// 64 columns, one M-block at a time.  At the end every CTA writes its fp32 partial to the workspace and
// encoder_bwd_reduce_kernel sums the partials in a fixed order in fp64: no float atomics, bit-identical from run to run.
// Operand images (no swizzle, kBwdRows = R = 64): H1 / dH1 element (m, j) at (j % 8) 16 + (j / 8) 16 R + (m / 8) 128 +
// (m % 8) 2 -- MN-major B of L2 (LBO 16 R, SBO 128) and K-major A / B of the weight gradients (LBO 128, SBO 16 R);
// dH2 the same keyed by the W2 image row r; X as in the forward, which read along m is the MN-major B of dW1.
constexpr int kBwdRows = 64;
constexpr int kBwdThreads = 256;                    // 8 warps: (TMEM lane quadrant, half of the 64 row columns)
constexpr uint32_t kBwdW2Col = 0, kBwdW2Stride = 192, kBwdW1Col = 384, kBwdScratchCol = 448;

struct BwdOffsets { uint32_t h1, dh2, x, x_bytes, bar, tmem_slot, smem_end; };
__host__ __device__ inline BwdOffsets bwd_offsets(int h, int in_dim) {
  const Offsets f = offsets(h, in_dim);             // the resident weight image is the forward's, at the same place
  BwdOffsets o;
  o.h1 = (f.packed_end + 127u) & ~127u;
  o.dh2 = o.h1 + (uint32_t)padded_k(h) * kBwdRows * 2;
  o.x = o.dh2 + (uint32_t)padded_m(h) * kBwdRows * 2;
  o.x_bytes = (uint32_t)kBwdRows * padded_k1(in_dim) * 2;
  o.bar = o.x + 2 * o.x_bytes;                        // two X buffers: the next tile is staged while dW1 reads this one
  o.tmem_slot = o.bar + 16;                           // mbarriers: MMA completion, weights' bulk copy
  o.smem_end = o.tmem_slot + 16;
  return o;
}
// floats of one CTA's partial: dW2 | db2 as [h + 1][h] (column j of the torch layout is row j here), then dW1 | db1 as
// [in_dim + 1][h]
__host__ __device__ inline int64_t bwd_partial_floats(int h, int in_dim) { return (int64_t)(h + 1 + in_dim + 1) * h; }

struct BwdArgs {
  const float *obs, *zone_obs, *g;
  const uint8_t* packed;
  float* part;
  int* status;
  int B, N, Z, obs_dim, h, n_tiles, S;
};
// kSrcFrames: plus the frames source of the forward (frames, layout table, task, divisors); a type of its own so that the
// kernel of materialised rows keeps its parameter block
struct BwdFramesArgs : BwdArgs { EncArgs rows; };

// eight consecutive values (k = 8 kc ..) of row m of a backward tile; zeros for padding rows and rows beyond the batch.
// SRC: where the zone part comes from, as for load_half_row (kSrcFrames: obs_dim == 8, chunk 1 = zone features + ones)
template <int SRC, class Args>
__device__ __forceinline__ void bwd_load_chunk(const Args& a, int tile, int m, int kc, float (&x)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) x[j] = 0.f;
  const int sh = a.S == 16 ? 4 : 3;
  const int e = tile * (kBwdRows >> sh) + (m >> sh), slot = m & (a.S - 1);
  const int in_dim = a.obs_dim + a.Z;
  if (tile < a.n_tiles && e < a.B && slot < a.N && 8 * kc < padded_k1(in_dim)) {
    const float* ob = a.obs + (size_t)e * a.obs_dim;
    if constexpr (SRC == kSrcFrames) {
      if (kc == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = __ldg(ob + j);
      } else {
        float z[7];
        zone_features_from_frame(a.rows, e, slot, z);
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = j < 7 && j < a.Z ? z[j < 7 ? j : 0] : (j <= a.Z + 1 ? 1.f : 0.f);
      }
      return;
    }
    const float* zo = a.zone_obs + ((size_t)e * a.N + slot) * a.Z;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = 8 * kc + j;
      if (k < a.obs_dim) x[j] = __ldg(ob + k);
      else if (k < in_dim) x[j] = __ldg(zo + (k - a.obs_dim));
      else if (k <= in_dim + 1) x[j] = 1.f;
    }
  }
}

__device__ __forceinline__ float bf16_bits_to_float(uint32_t b) { return __uint_as_float(b << 16); }

template <int SRC, class Args>
__global__ void __launch_bounds__(kBwdThreads, 1) zone_encode_backward_kernel(const Args a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int in_dim = a.obs_dim + a.Z;
  const Offsets fo = offsets(a.h, in_dim);
  const BwdOffsets o = bwd_offsets(a.h, in_dim);
  const int KP = padded_k(a.h), MP = padded_m(a.h), kK1 = padded_k1(in_dim), n_mb = MP / 128;
  const int t = threadIdx.x, lane = t & 31;
  const int warp = __shfl_sync(0xffffffffu, t >> 5, 0);
  const int q = warp & 3, ch = warp >> 2;                     // lane quadrant, rows m = 32 ch .. 32 ch + 31
  const bool leader = elect_one();
  const uint32_t bar = smem_u32(smem + o.bar), wbar = bar + 8u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + o.tmem_slot);
  if (t == 0) {
    mbar_init(bar, 1);
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    bulk_load_weights(wbar, smem_u32(smem), a.packed, fo.packed_end);
  }
  if (t < 32) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
  const uint32_t scratch = tmem_base + kBwdScratchCol;
  // instruction descriptors (D fp32, A / B bf16, M = 128): bit 15 = A MN-major, bit 16 = B MN-major
  const uint32_t id_base = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 4) << 24);
  const uint32_t id_rows = id_base | ((uint32_t)(kBwdRows >> 3) << 17);               // N = 64 rows
  const uint32_t id_l2 = id_rows | (1u << 16), id_dh1 = id_rows | (1u << 15) | (1u << 16);
  const uint32_t id_dw2 = id_base | ((uint32_t)(KP >> 3) << 17);                       // N = H1 rows
  const uint32_t id_dw1 = id_base | ((uint32_t)(kK1 >> 3) << 17) | (1u << 16);          // N = input columns
  const uint32_t w1_addr = smem_u32(smem + fo.w1), w2_addr = smem_u32(smem + fo.w2);
  const uint32_t h1_addr = smem_u32(smem + o.h1), dh2_addr = smem_u32(smem + o.dh2);
  uint8_t* h1buf = smem + o.h1;
  uint8_t* dh2buf = smem + o.dh2;
  const float inv_n = 1.0f / (float)a.N;
  const int sh = a.S == 16 ? 4 : 3;
  uint32_t parity = 0u;
  bool healthy = true;
  // issue (warp 0, converged; one elected lane executes) + commit, then everyone waits for completion
  auto mma_phase = [&](auto&& issue) {
    if (warp == 0) {
      tc_fence_after();
      issue();
      if (leader) mma_commit(bar);
      __syncwarp();
    }
    healthy = mbar_wait(bar, parity) && healthy;
    parity ^= 1u;
    tc_fence_after();
  };
  auto phase_end = [&]() {                                    // smem written for the tensor pipe / TMEM read: next phase may go
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
  };
  // hidden unit of W2 / W1 image row r (pack_kernel's row map: M-block 1 keeps units 128 .. 191 in its upper 64 rows)
  auto unit_of_row = [](int r) { return r < 128 ? r : (r >= 192 ? r - 64 : -1); };

  const int m_st = t & (kBwdRows - 1), kc_st = t >> 6;        // the 16-byte unit of X this thread stages
  const uint32_t x_off = (uint32_t)((m_st & 7) * 16 + (m_st >> 3) * (16 * kK1) + kc_st * 128);
  float x[8];
  int tile = (int)blockIdx.x;
  bwd_load_chunk<SRC>(a, tile, m_st, kc_st, x);
  for (int k = 0; tile < a.n_tiles; tile += (int)gridDim.x, ++k) {
    const uint32_t xb = o.x + (uint32_t)(k & 1) * o.x_bytes;
    if (kc_st < kK1 / 8)
      *reinterpret_cast<uint4*>(smem + xb + x_off) =
          make_uint4(pack_bf16(x[0], x[1]), pack_bf16(x[2], x[3]), pack_bf16(x[4], x[5]), pack_bf16(x[6], x[7]));
    phase_end();
    bwd_load_chunk<SRC>(a, tile + (int)gridDim.x, m_st, kc_st, x);  // the next tile's rows travel under this one
    const uint32_t x_addr = smem_u32(smem + xb);
    if (k == 0 && warp == 0) { healthy = mbar_wait(wbar, 0u) && healthy; __syncwarp(); }
    // ---- L1, one M-block at a time, -> H1 (bf16 relu), keyed by hidden unit (ones rows h, h + 1 included) ----
    for (int b = 0; b < n_mb; ++b) {
      mma_phase([&] {
        for (int s = 0; s < kK1 / 16; ++s)
          if (leader) mma_bf16(scratch, smem_desc(w1_addr + (uint32_t)(b * 16 * 16 * kK1 + 256 * s), 128u, 16 * kK1),
                               smem_desc(x_addr + 256u * s, 128u, 16 * kK1), id_rows, s > 0);
      });
      const int u = unit_of_row(128 * b + 32 * q + lane);
      uint32_t v[32];
      tmem_ld32(scratch + lane_addr + (uint32_t)(32 * ch), v);
      tmem_ld_wait(v);
      if (u >= 0) relu_to_h1(v, h1buf + (uint32_t)((u & 7) * 16 + (u >> 3) * (16 * kBwdRows)), ch, u < KP);
      phase_end();
    }
    // ---- L2, one M-block at a time, -> dH2 keyed by W2 image row ----
    for (int b = 0; b < n_mb; ++b) {
      mma_phase([&] {
        for (int s = 0; s < KP / 16; ++s)
          if (leader) mma_bf16(scratch, smem_desc(w2_addr + (uint32_t)(b * 16 * 16 * KP + 256 * s), 128u, 16 * KP),
                               smem_desc(h1_addr + (uint32_t)(2 * 16 * kBwdRows * s), 16 * kBwdRows, 128u), id_l2, s > 0);
      });
      const int r = 128 * b + 32 * q + lane, u = unit_of_row(r);
      uint32_t v[32];
      tmem_ld32(scratch + lane_addr + (uint32_t)(32 * ch), v);
      tmem_ld_wait(v);
      if (u >= 0) {
        // this thread's 32 rows are the slots of 32 / S envs
        const int e0 = tile * (kBwdRows >> sh) + ((32 * ch) >> sh);
        float d[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int e = e0 + i;
          const float gv = (i < (32 >> sh) && u < a.h && e < a.B) ? __ldg(a.g + (size_t)e * a.h + u) : 0.f;
          d[i] = __bfloat162float(__float2bfloat16_rn(__fmul_rn(gv, inv_n)));
        }
        uint8_t* row = dh2buf + (uint32_t)((r & 7) * 16 + (r >> 3) * (16 * kBwdRows));
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          float w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int mi = 8 * qq + i, ei = mi >> sh;
            const float dv = ei == 0 ? d[0] : (ei == 1 ? d[1] : (ei == 2 ? d[2] : d[3]));
            w[i] = __uint_as_float(v[mi]) > 0.f ? dv : 0.f;
          }
          *reinterpret_cast<uint4*>(row + (uint32_t)((ch * 4 + qq) * 128)) =
              make_uint4(pack_bf16(w[0], w[1]), pack_bf16(w[2], w[3]), pack_bf16(w[4], w[5]), pack_bf16(w[6], w[7]));
        }
      }
      phase_end();
    }
    // ---- dW2 += dH2^T H1 (both M-blocks), and dH1^T = W2^T dH2^T one M-block at a time -> dH1 over H1 ----
    for (int b = 0; b < n_mb; ++b) {
      mma_phase([&] {
        if (b == 0)
          for (int bb = 0; bb < n_mb; ++bb)
            for (int s = 0; s < kBwdRows / 16; ++s)
              if (leader) mma_bf16(tmem_base + kBwdW2Col + (uint32_t)bb * kBwdW2Stride,
                                   smem_desc(dh2_addr + (uint32_t)(bb * 16 * 16 * kBwdRows + 256 * s), 128u, 16 * kBwdRows),
                                   smem_desc(h1_addr + 256u * s, 128u, 16 * kBwdRows), id_dw2, (k > 0 || s > 0) ? 1u : 0u);
        bool first = true;
        for (int s = 0; s < MP / 16; ++s) {
          if (s >= 8 && s < 12) continue;                    // image rows 128 .. 191: zero rows of W2
          if (leader) mma_bf16(scratch, smem_desc(w2_addr + (uint32_t)(b * 16 * 128 + 2 * 16 * KP * s), 16 * KP, 128u),
                               smem_desc(dh2_addr + (uint32_t)(2 * 16 * kBwdRows * s), 16 * kBwdRows, 128u), id_dh1, first ? 0u : 1u);
          first = false;
        }
      });
      const int j = 128 * b + 32 * q + lane;
      uint32_t v[32];
      tmem_ld32(scratch + lane_addr + (uint32_t)(32 * ch), v);
      tmem_ld_wait(v);
      if (j < a.h) {
        uint8_t* row = h1buf + (uint32_t)((j & 7) * 16 + (j >> 3) * (16 * kBwdRows));
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
          uint4* p = reinterpret_cast<uint4*>(row + (uint32_t)((ch * 4 + qq) * 128));
          const uint4 hv = *p;
          const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w};
          float w[8];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            w[2 * i] = bf16_bits_to_float(hw[i] & 0xffffu) > 0.f ? __uint_as_float(v[8 * qq + 2 * i]) : 0.f;
            w[2 * i + 1] = bf16_bits_to_float(hw[i] >> 16) > 0.f ? __uint_as_float(v[8 * qq + 2 * i + 1]) : 0.f;
          }
          *p = make_uint4(pack_bf16(w[0], w[1]), pack_bf16(w[2], w[3]), pack_bf16(w[4], w[5]), pack_bf16(w[6], w[7]));
        }
      }
      phase_end();
    }
    // ---- dW1 += dH1^T X: completion is awaited by the next tile's first phase (before H1 / this X buffer are reused) ----
    if (warp == 0) {
      tc_fence_after();
      for (int b = 0; b < n_mb; ++b)
        for (int s = 0; s < kBwdRows / 16; ++s)
          if (leader) mma_bf16(tmem_base + kBwdW1Col + (uint32_t)(32 * b),
                               smem_desc(h1_addr + (uint32_t)(b * 16 * 16 * kBwdRows + 256 * s), 128u, 16 * kBwdRows),
                               smem_desc(x_addr + (uint32_t)(2 * 16 * kK1 * s), 16 * kK1, 128u), id_dw1, (k > 0 || s > 0) ? 1u : 0u);
      __syncwarp();
    }
  }
  // ---- the CTA's partial: TMEM -> workspace (transposed: consecutive lanes = consecutive hidden units, coalesced) ----
  mma_phase([&] {});                                           // every MMA issued so far has completed
  float* part = a.part + (size_t)blockIdx.x * (size_t)bwd_partial_floats(a.h, in_dim);
  for (int b = 0; b < n_mb; ++b) {
    const int u = unit_of_row(128 * b + 32 * q + lane);
    for (int c = ch; c * 32 <= a.h; c += 2) {                 // columns 0 .. h (h: the ones row -> db2)
      uint32_t v[32];
      tmem_ld32(tmem_base + lane_addr + kBwdW2Col + (uint32_t)b * kBwdW2Stride + (uint32_t)(32 * c), v);
      tmem_ld_wait(v);
      if (u >= 0 && u < a.h)
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (32 * c + i <= a.h) part[(size_t)(32 * c + i) * a.h + u] = __uint_as_float(v[i]);
    }
    if (ch == 0) {                                             // columns 0 .. in_dim (in_dim: the ones column -> db1)
      const int j = 128 * b + 32 * q + lane;
      uint32_t v[32];
      tmem_ld32(tmem_base + lane_addr + kBwdW1Col + (uint32_t)(32 * b), v);
      tmem_ld_wait(v);
      float* p1 = part + (size_t)(a.h + 1) * a.h;
      if (j < a.h)
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i <= in_dim) p1[(size_t)i * a.h + j] = __uint_as_float(v[i]);
    }
  }
  if (!healthy && a.status) atomicExch(a.status, 1);
  tc_fence_before();
  __syncthreads();
  if (t < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
}

// element i of the partials, summed over the n_part CTAs in index order in fp64 -> torch-layout fp32 outputs
struct BwdReduceArgs { const float* part; float *dw1, *db1, *dw2, *db2; int n_part, h, in_dim; };
__global__ void encoder_bwd_reduce_kernel(const BwdReduceArgs a) {
  const int64_t n = bwd_partial_floats(a.h, a.in_dim), e2 = (int64_t)(a.h + 1) * a.h;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int p = 0; p < a.n_part; ++p) s += (double)__ldg(a.part + (size_t)p * n + i);
    const float v = (float)s;
    if (i < e2) {
      const int col = (int)(i / a.h), u = (int)(i % a.h);
      if (col < a.h) a.dw2[(size_t)u * a.h + col] = v;
      else a.db2[u] = v;
    } else {
      const int col = (int)((i - e2) / a.h), u = (int)((i - e2) % a.h);
      if (col < a.in_dim) a.dw1[(size_t)u * a.in_dim + col] = v;
      else a.db1[u] = v;
    }
  }
}

static int check_shape(const CrlEncoderShape* s) {
  if (!s) return CRL_ERR_NULL;
  if (s->obs_dim <= 0 || s->zone_dim <= 0 || s->obs_dim + s->zone_dim + 1 > 32) return CRL_ERR_CONFIG;   // + a ones column
  if (s->num_zones <= 0 || s->num_zones > 16) return CRL_ERR_CONFIG;
  if (s->hidden <= 0) return CRL_ERR_CONFIG;
  if (padded_k(s->hidden) > 192) return CRL_ERR_UNSUPPORTED;   // resident W2 + two groups' operand buffers must fit an SM
  return CRL_OK;
}

}  // namespace crl_enc

using namespace crl_enc;

extern "C" {

#ifdef CRL_ENC_TIMELINE
int crl_debug_enc_timeline(long long* host, int64_t bytes) {
  return cudaMemcpyFromSymbol(host, g_timeline, (size_t)bytes < sizeof(g_timeline) ? (size_t)bytes : sizeof(g_timeline)) == cudaSuccess ? 0 : -1;
}
#endif

int crl_encoder_packed_bytes(const CrlEncoderShape* s, int64_t* bytes) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!bytes) return CRL_ERR_NULL;
  *bytes = (int64_t)offsets(s->hidden, s->obs_dim + s->zone_dim).packed_end;
  return CRL_OK;
}

int crl_encoder_pack(const CrlEncoderShape* s, const float* w1, const float* b1, const float* w2, const float* b2,
                     void* packed, void* stream) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!w1 || !b1 || !w2 || !b2 || !packed) return CRL_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(packed) & 15u) return CRL_ERR_ALIGN;
  PackArgs a{w1, b1, w2, b2, static_cast<uint8_t*>(packed), s->obs_dim + s->zone_dim, s->hidden};
  pack_kernel<<<148, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

// The frames source of crl_zone_encode_frames / crl_zone_encode_backward_frames / crl_frames_zone_obs
struct FrameRows { const CrlFrame* frames; const float* layout_xy; const uint32_t* layout_tmax; };

// the exact-division constants the step kernel uses (proven on the host once per divisor)
static crl::DivConst enc_div_const(int d, int lo, int hi) {
  static struct { int d, lo, hi; crl::DivConst k; } cache[8];
  static int used = 0;
  for (int i = 0; i < used; ++i)
    if (cache[i].d == d && cache[i].lo == lo && cache[i].hi == hi) return cache[i].k;
  const crl::DivConst k = crl::make_div_const(d, lo, hi);
  if (used < 8) { cache[used].d = d; cache[used].lo = lo; cache[used].hi = hi; cache[used].k = k; ++used; }
  return k;
}

// Rows built from frames: the env configuration (task, N, num_steps, max_cooldown; CRL_ERR_CONFIG for one no step
// accepts), the encoder shape (obs_dim 8: CRL_ERR_UNSUPPORTED otherwise; the task's zone_dim and num_zones:
// CRL_ERR_CONFIG otherwise) and the record / table pointers -> the frames fields of `a`.
static int frame_row_params(const CrlEncoderShape* s, const CrlConfig* cfg, const FrameRows& fr, EncArgs& a) {
  if (!cfg) return CRL_ERR_NULL;
  if (cfg->task < 0 || cfg->task > 2 || cfg->num_zones <= 0 || cfg->num_zones > (cfg->task == CRL_TASK_CM ? 7 : 15) ||
      cfg->num_steps <= 0 || cfg->num_steps > 65534 || cfg->max_cooldown < 0 || cfg->max_cooldown > 255)
    return CRL_ERR_CONFIG;
  if (s) {
    if (s->obs_dim != 8) return CRL_ERR_UNSUPPORTED;
    if (cfg->num_zones != s->num_zones || s->zone_dim != (cfg->task == CRL_TASK_TSP ? 6 : 7)) return CRL_ERR_CONFIG;
  }
  if (!fr.frames || !fr.layout_xy || (cfg->task == CRL_TASK_TTSP && !fr.layout_tmax)) return CRL_ERR_NULL;
  if ((reinterpret_cast<uintptr_t>(fr.frames) & 15u) || (reinterpret_cast<uintptr_t>(fr.layout_xy) & 7u) ||
      (reinterpret_cast<uintptr_t>(fr.layout_tmax) & 3u))
    return CRL_ERR_ALIGN;
  a.task = cfg->task; a.num_steps = cfg->num_steps; a.N = cfg->num_zones; a.Z = cfg->task == CRL_TASK_TSP ? 6 : 7;
  a.div_steps = enc_div_const(cfg->num_steps, -65535, 65535);
  a.div_cd = enc_div_const(cfg->max_cooldown > 0 ? cfg->max_cooldown : 1, 0, 255);
  if (!a.div_steps.exact || !a.div_cd.exact) return CRL_ERR_CONFIG;
  a.frames = reinterpret_cast<const uint4*>(fr.frames);
  a.layout_xy = reinterpret_cast<const float2*>(fr.layout_xy);
  a.layout_tmax = fr.layout_tmax;
  return CRL_OK;
}

static int zone_encode_launch(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* zone_obs,
                              const CrlConfig* cfg, const CrlState* st, const void* packed, float* pooled, int32_t* status,
                              void* stream, void* xhead = nullptr, const FrameRows* fr = nullptr) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!obs || (!zone_obs && !st && !fr) || !packed || (!pooled && !xhead)) return CRL_ERR_NULL;
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  if (reinterpret_cast<uintptr_t>(packed) & 15u) return CRL_ERR_ALIGN;
  if (fr) {                                                  // checked before any CUDA call
    if (xhead) return CRL_ERR_UNSUPPORTED;
    EncArgs probe{};
    const int rf = frame_row_params(s, cfg, *fr, probe);
    if (rf) return rf;
  }
  const Offsets o = offsets(s->hidden, s->obs_dim + s->zone_dim);
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess) return CRL_ERR_DEVICE;
  static bool attr_set[64] = {false};                       // per device: opt in to > 48 KB of dynamic shared memory
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(zone_encode_kernel<kSrcZoneObs, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_kernel<kSrcZoneObs, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_kernel<kSrcState, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_kernel<kSrcZoneObs, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_kernel<kSrcState, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_kernel<kSrcFrames, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return CRL_ERR_DEVICE;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  EncArgs a{};
  a.obs = obs; a.zone_obs = zone_obs; a.packed = static_cast<const uint8_t*>(packed); a.out = pooled; a.status = status;
  a.xhead = static_cast<uint8_t*>(xhead); a.KH = head_k(s->obs_dim, s->hidden);
  a.B = num_envs; a.N = s->num_zones; a.Z = s->zone_dim; a.obs_dim = s->obs_dim; a.h = s->hidden;
  a.S = slots_per_env(s->num_zones);
  a.n_tiles = (num_envs + kRows / a.S - 1) / (kRows / a.S);
  if (st) {
    // the zone features come from the state planes: the shapes must be the env's own
    if (!cfg || !st->aux || !st->zone_xy) return CRL_ERR_NULL;
    if (s->obs_dim != 8 || cfg->num_envs != num_envs || cfg->num_zones != s->num_zones || cfg->task < 0 || cfg->task > 2 ||
        s->zone_dim != (cfg->task == CRL_TASK_TSP ? 6 : 7) || cfg->num_steps <= 0 || cfg->num_steps > 65534 ||
        cfg->max_cooldown < 0 || cfg->max_cooldown > 255)
      return CRL_ERR_CONFIG;
    if (cfg->task == CRL_TASK_TTSP && !st->zone_tmax) return CRL_ERR_NULL;
    if (cfg->task == CRL_TASK_CM && !st->cooldown) return CRL_ERR_NULL;
    a.aux = reinterpret_cast<const float4*>(st->aux);
    a.zone_xy = reinterpret_cast<const float2*>(st->zone_xy);
    a.zone_tmax = st->zone_tmax;
    a.cooldown = reinterpret_cast<const uint2*>(st->cooldown);
    a.task = cfg->task; a.num_steps = cfg->num_steps;
    a.div_steps = enc_div_const(cfg->num_steps, -65535, 65535);
    a.div_cd = enc_div_const(cfg->max_cooldown > 0 ? cfg->max_cooldown : 1, 0, 255);
    if (!a.div_steps.exact || !a.div_cd.exact) return CRL_ERR_CONFIG;
  } else if (fr) {
    const int rf = frame_row_params(s, cfg, *fr, a);
    if (rf) return rf;
  }
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int want = (a.n_tiles + kGroups - 1) / kGroups;
  const int grid = want < sms ? want : sms;                   // persistent: one CTA per SM, weights loaded once
  const cudaStream_t cs = static_cast<cudaStream_t>(stream);
  if (st && xhead) zone_encode_kernel<kSrcState, true><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  else if (st) zone_encode_kernel<kSrcState, false><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  else if (fr) zone_encode_kernel<kSrcFrames, false><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  else if (xhead) zone_encode_kernel<kSrcZoneObs, true><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  else if (padded_k1(s->obs_dim + s->zone_dim) == 32) zone_encode_kernel<kSrcZoneObs, false, true><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  else zone_encode_kernel<kSrcZoneObs, false><<<grid, kEncThreads, o.smem_end, cs>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

int crl_zone_encode(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* zone_obs,
                    const void* packed, float* pooled, int32_t* status, void* stream) {
  if (!zone_obs) return CRL_ERR_NULL;
  return zone_encode_launch(s, num_envs, obs, zone_obs, nullptr, nullptr, packed, pooled, status, stream);
}

int crl_zone_encode_state(const CrlEncoderShape* s, const CrlConfig* cfg, const CrlState* st, const float* obs,
                          const void* packed, float* pooled, int32_t* status, void* stream) {
  if (!cfg || !st) return CRL_ERR_NULL;
  return zone_encode_launch(s, cfg->num_envs, obs, nullptr, cfg, st, packed, pooled, status, stream);
}

int crl_zone_encode_frames(const CrlEncoderShape* s, const CrlConfig* cfg, int32_t num_rows, const float* obs,
                           const CrlFrame* frames, const float* layout_xy, const uint32_t* layout_tmax, const void* packed,
                           float* pooled, int32_t* status, void* stream) {
  if (!cfg) return CRL_ERR_NULL;
  const FrameRows fr{frames, layout_xy, layout_tmax};
  return zone_encode_launch(s, num_rows, obs, nullptr, cfg, nullptr, packed, pooled, status, stream, nullptr, &fr);
}

// one thread per (row, zone): the Z features of zone_features_from_frame
__global__ void frames_zone_obs_kernel(const EncArgs a, float* zone_obs) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)a.B * a.N) return;
  const int e = (int)(i / a.N), slot = (int)(i % a.N);
  float z[7];
  zone_features_from_frame(a, e, slot, z);
  float* row = zone_obs + i * a.Z;
#pragma unroll
  for (int j = 0; j < 7; ++j)
    if (j < a.Z) row[j] = z[j];
}

int crl_frames_zone_obs(const CrlConfig* cfg, int32_t num_rows, const CrlFrame* frames, const float* layout_xy,
                        const uint32_t* layout_tmax, float* zone_obs, void* stream) {
  if (!cfg || !zone_obs) return CRL_ERR_NULL;
  if (num_rows <= 0) return CRL_ERR_CONFIG;
  EncArgs a{};
  const int rc = frame_row_params(nullptr, cfg, FrameRows{frames, layout_xy, layout_tmax}, a);
  if (rc) return rc;
  a.B = num_rows;
  const int64_t n = (int64_t)num_rows * a.N;
  frames_zone_obs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, zone_obs);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

int crl_encoder_head_packed_bytes(const CrlEncoderShape* s, int64_t* bytes) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!bytes) return CRL_ERR_NULL;
  const HeadOffsets o = head_offsets(s->obs_dim, s->hidden);
  if (o.smem_end > 227u * 1024u) return CRL_ERR_UNSUPPORTED;
  *bytes = (int64_t)o.packed_end;
  return CRL_OK;
}

int crl_encoder_pack_head(const CrlEncoderShape* s, const float* w, const float* b, void* packed, void* stream) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!w || !b || !packed) return CRL_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(packed) & 15u) return CRL_ERR_ALIGN;
  if (head_offsets(s->obs_dim, s->hidden).smem_end > 227u * 1024u) return CRL_ERR_UNSUPPORTED;
  HeadPackArgs a{w, b, static_cast<uint8_t*>(packed), s->obs_dim, s->hidden};
  head_pack_kernel<<<148, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

static int head_launch(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* pooled, const void* xhead,
                       const void* packed_head, float* out, int32_t* status, void* stream) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if ((!xhead && (!obs || !pooled)) || !packed_head || !out) return CRL_ERR_NULL;
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  if (reinterpret_cast<uintptr_t>(packed_head) & 15u) return CRL_ERR_ALIGN;
  const HeadOffsets o = head_offsets(s->obs_dim, s->hidden);
  if (o.smem_end > 227u * 1024u) return CRL_ERR_UNSUPPORTED;
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess) return CRL_ERR_DEVICE;
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(encoder_head_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(encoder_head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return CRL_ERR_DEVICE;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  HeadArgs a{obs, pooled, static_cast<const uint8_t*>(packed_head), out, status, num_envs, s->obs_dim, s->hidden, 0,
             static_cast<const uint8_t*>(xhead)};
  a.n_tiles = (num_envs + kRows - 1) / kRows;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int want = (a.n_tiles + kGroups - 1) / kGroups;
  const int grid = want < sms ? want : sms;
  if (xhead) {
    // programmatic launch behind the zone kernel (see there); without a programmatic predecessor it is an ordinary launch
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(kGroupThreads * kGroups);
    lc.dynamicSmemBytes = o.smem_end; lc.stream = static_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at; lc.numAttrs = 1;
    if (cudaLaunchKernelEx(&lc, encoder_head_kernel<true>, a) != cudaSuccess) { (void)cudaGetLastError(); return CRL_ERR_LAUNCH; }
    return CRL_OK;
  }
  encoder_head_kernel<false><<<grid, kGroupThreads * kGroups, o.smem_end, static_cast<cudaStream_t>(stream)>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

int crl_encoder_head(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* pooled,
                     const void* packed_head, float* out, int32_t* status, void* stream) {
  if (!obs || !pooled) return CRL_ERR_NULL;
  return head_launch(s, num_envs, obs, pooled, nullptr, packed_head, out, status, stream);
}

int crl_encoder_workspace_bytes(const CrlEncoderShape* s, int32_t num_envs, int64_t* bytes) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!bytes) return CRL_ERR_NULL;
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  if (s->obs_dim != 8 || padded_k1(s->obs_dim + s->zone_dim) != 16) return CRL_ERR_UNSUPPORTED;   // ZoneEnvModel's own shape
  *bytes = (int64_t)((num_envs + kRows - 1) / kRows) * kRows * head_k(s->obs_dim, s->hidden) * 2;
  return CRL_OK;
}

int crl_encoder_forward(const CrlEncoderShape* s, const CrlConfig* cfg, const CrlState* st, int32_t num_envs, const float* obs,
                        const float* zone_obs, const void* packed, const void* packed_head, void* workspace, float* out,
                        int32_t* status, void* stream) {
  int64_t need = 0;
  const int rc = crl_encoder_workspace_bytes(s, num_envs, &need);
  if (rc) return rc;
  if (!workspace || !out || !packed_head) return CRL_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(workspace) & 15u) return CRL_ERR_ALIGN;
  if (st ? (!cfg || cfg->num_envs != num_envs) : !zone_obs) return st ? CRL_ERR_CONFIG : CRL_ERR_NULL;
  const int rz = zone_encode_launch(s, num_envs, obs, st ? nullptr : zone_obs, st ? cfg : nullptr, st, packed, nullptr, status, stream,
                                    workspace);
  if (rz) return rz;
  return head_launch(s, num_envs, nullptr, nullptr, workspace, packed_head, out, status, stream);
}

// ---- precise mode (split-bf16 operands, fp32 biases; like for like with the fp32 reference module) ----
static int check_precise(const CrlEncoderShape* s) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (s->obs_dim + s->zone_dim > 16) return CRL_ERR_UNSUPPORTED;           // one K step of layer 1
  if (precise_offsets(s->hidden).s_end > 227u * 1024u) return CRL_ERR_UNSUPPORTED;
  return CRL_OK;
}

int crl_encoder_precise_packed_bytes(const CrlEncoderShape* s, int64_t* bytes) {
  const int rc = check_precise(s);
  if (rc) return rc;
  if (!bytes) return CRL_ERR_NULL;
  *bytes = (int64_t)precise_offsets(s->hidden).g_end;
  return CRL_OK;
}

int crl_encoder_pack_precise(const CrlEncoderShape* s, const float* w1, const float* b1, const float* w2, const float* b2,
                             void* packed, void* stream) {
  const int rc = check_precise(s);
  if (rc) return rc;
  if (!w1 || !b1 || !w2 || !b2 || !packed) return CRL_ERR_NULL;
  if (reinterpret_cast<uintptr_t>(packed) & 15u) return CRL_ERR_ALIGN;
  PrecisePackArgs a{w1, b1, w2, b2, static_cast<uint8_t*>(packed), s->obs_dim + s->zone_dim, s->hidden};
  pack_precise_kernel<<<148, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

int crl_zone_encode_precise(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* zone_obs,
                            const void* packed_precise, float* pooled, int32_t* status, void* stream) {
  const int rc = check_precise(s);
  if (rc) return rc;
  if (!obs || !zone_obs || !packed_precise || !pooled) return CRL_ERR_NULL;
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  if (reinterpret_cast<uintptr_t>(packed_precise) & 15u) return CRL_ERR_ALIGN;
  const PreciseOffsets o = precise_offsets(s->hidden);
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess) return CRL_ERR_DEVICE;
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(zone_encode_precise_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return CRL_ERR_DEVICE;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  EncArgs a{};
  a.obs = obs; a.zone_obs = zone_obs; a.packed = static_cast<const uint8_t*>(packed_precise); a.out = pooled; a.status = status;
  a.B = num_envs; a.N = s->num_zones; a.Z = s->zone_dim; a.obs_dim = s->obs_dim; a.h = s->hidden;
  a.S = slots_per_env(s->num_zones);
  a.n_tiles = (num_envs + kRows / a.S - 1) / (kRows / a.S);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int nb = ((precise_k(s->hidden) + 127) & ~127) / 128;
  const int want = a.n_tiles * nb, cap = sms / nb * nb;       // CTA c owns M-block c % nb of tiles c / nb, c / nb + grid / nb, ..
  const int grid = want < cap ? want : cap;
  zone_encode_precise_kernel<<<grid, kGroupThreads, o.s_end, static_cast<cudaStream_t>(stream)>>>(a);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

// ---- backward ----
// the launch rule: one partial per CTA, grid = min(tiles of kBwdRows rows, SMs of the current device)
static int bwd_grid(const CrlEncoderShape* s, int32_t num_envs, int* grid, int* n_tiles) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess) return CRL_ERR_DEVICE;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return CRL_ERR_DEVICE;
  const int per_tile = kBwdRows / slots_per_env(s->num_zones);
  *n_tiles = (int)(((int64_t)num_envs + per_tile - 1) / per_tile);
  *grid = *n_tiles < sms ? *n_tiles : sms;
  return CRL_OK;
}

int crl_encoder_backward_workspace_bytes(const CrlEncoderShape* s, int32_t num_envs, int64_t* bytes) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!bytes) return CRL_ERR_NULL;
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  int grid = 0, n_tiles = 0;
  const int rg = bwd_grid(s, num_envs, &grid, &n_tiles);
  if (rg) return rg;
  *bytes = (int64_t)grid * bwd_partial_floats(s->hidden, s->obs_dim + s->zone_dim) * 4;
  return CRL_OK;
}

static int zone_encode_backward_launch(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* zone_obs,
                                       const CrlConfig* cfg, const FrameRows* fr, const void* packed,
                                       const float* grad_pooled, void* workspace, float* dw1, float* db1, float* dw2,
                                       float* db2, int32_t* status, void* stream) {
  const int rc = check_shape(s);
  if (rc) return rc;
  if (!obs || (!zone_obs && !fr) || !packed || !grad_pooled || !workspace || !dw1 || !db1 || !dw2 || !db2) return CRL_ERR_NULL;
  BwdFramesArgs a{};
  if (fr) {
    const int rf = frame_row_params(s, cfg, *fr, a.rows);
    if (rf) return rf;
  }
  if (num_envs <= 0) return CRL_ERR_CONFIG;
  if ((reinterpret_cast<uintptr_t>(packed) | reinterpret_cast<uintptr_t>(workspace)) & 15u) return CRL_ERR_ALIGN;
  const BwdOffsets o = bwd_offsets(s->hidden, s->obs_dim + s->zone_dim);
  if (o.smem_end > 227u * 1024u) return CRL_ERR_UNSUPPORTED;
  int grid = 0, n_tiles = 0;
  const int rg = bwd_grid(s, num_envs, &grid, &n_tiles);
  if (rg) return rg;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return CRL_ERR_DEVICE;
  static bool attr_set[64] = {false};
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    if (cudaFuncSetAttribute(zone_encode_backward_kernel<kSrcZoneObs, BwdArgs>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(zone_encode_backward_kernel<kSrcFrames, BwdFramesArgs>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess)
      return CRL_ERR_DEVICE;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  a.obs = obs; a.zone_obs = zone_obs; a.g = grad_pooled; a.packed = static_cast<const uint8_t*>(packed);
  a.part = static_cast<float*>(workspace); a.status = status;
  a.B = num_envs; a.N = s->num_zones; a.Z = s->zone_dim; a.obs_dim = s->obs_dim; a.h = s->hidden;
  a.S = slots_per_env(s->num_zones); a.n_tiles = n_tiles;
  const cudaStream_t cs = static_cast<cudaStream_t>(stream);
  if (fr) zone_encode_backward_kernel<kSrcFrames, BwdFramesArgs><<<grid, kBwdThreads, o.smem_end, cs>>>(a);
  else zone_encode_backward_kernel<kSrcZoneObs, BwdArgs><<<grid, kBwdThreads, o.smem_end, cs>>>(static_cast<const BwdArgs&>(a));
  if (cudaGetLastError() != cudaSuccess) return CRL_ERR_LAUNCH;
  const BwdReduceArgs r{static_cast<const float*>(workspace), dw1, db1, dw2, db2, grid, s->hidden, s->obs_dim + s->zone_dim};
  const int64_t n = bwd_partial_floats(s->hidden, s->obs_dim + s->zone_dim);
  encoder_bwd_reduce_kernel<<<(int)((n + 255) / 256), 256, 0, cs>>>(r);
  return cudaGetLastError() == cudaSuccess ? CRL_OK : CRL_ERR_LAUNCH;
}

int crl_zone_encode_backward(const CrlEncoderShape* s, int32_t num_envs, const float* obs, const float* zone_obs,
                             const void* packed, const float* grad_pooled, void* workspace, float* dw1, float* db1,
                             float* dw2, float* db2, int32_t* status, void* stream) {
  if (!zone_obs) return CRL_ERR_NULL;
  return zone_encode_backward_launch(s, num_envs, obs, zone_obs, nullptr, nullptr, packed, grad_pooled, workspace, dw1, db1,
                                     dw2, db2, status, stream);
}

int crl_zone_encode_backward_frames(const CrlEncoderShape* s, const CrlConfig* cfg, int32_t num_rows, const float* obs,
                                    const CrlFrame* frames, const float* layout_xy, const uint32_t* layout_tmax,
                                    const void* packed, const float* grad_pooled, void* workspace, float* dw1, float* db1,
                                    float* dw2, float* db2, int32_t* status, void* stream) {
  if (!cfg) return CRL_ERR_NULL;
  const FrameRows fr{frames, layout_xy, layout_tmax};
  return zone_encode_backward_launch(s, num_rows, obs, nullptr, cfg, &fr, packed, grad_pooled, workspace, dw1, db1, dw2,
                                     db2, status, stream);
}

}  // extern "C"
