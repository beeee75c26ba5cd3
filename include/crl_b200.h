/*
 * crl_b200.h -- C ABI of the B200 batched simulator for the env.step() hot path
 * of PointTSP-v0 / PointTTSP-v0 / ColourMatch-v0.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  It replaces what sits
 * under the reference's vector env,
 *     main/src/torch_ac/torch_utils/penv.py:4-21   worker(): step / reset on done
 *     main/src/torch_ac/torch_utils/penv.py:46-66  ParallelEnv.reset/step/step_no_reset
 * i.e. N x { ZoneWrapper(FixedSeedsWrapper(TSPEnv|TimedTSPEnv|ColourMatchEnv)) }
 * (main/envs/make_env.py:3-51) each driving mujoco-py, by one call per batch.
 *
 * Rules of the boundary
 *  - plain C: pointers, sizes, PODs.  No C++ types, no torch types, no exceptions.
 *  - every pointer inside CrlState / CrlOut / CrlLayoutIn is DEVICE memory that the
 *    caller owns (torch allocates it); the library borrows it for the stream work
 *    it enqueues and allocates nothing itself.
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and
 *    does not synchronise, except crl_counters_read and crl_step_host, which say so.
 *  - return value 0 = OK; negative = CrlError.  Argument errors are detected on the
 *    host before anything is launched.  crl_strerror() names a code.
 *  - not re-entrant on the same CrlState; distinct states/devices may be driven
 *    from distinct host threads.
 *
 * Device layout (B = num_envs, N = num_zones, Z = zone_dim: 6 for TSP, 7 otherwise)
 *  state, structure-of-arrays, one 16-byte vector per env and plane:
 *    pose      float4[B]   (X, Y, phi, Vx)      world-frame position, heading in
 *                                                [-pi, pi], world-frame velocity
 *    aux       float4[B]   (Vy, omega, episode_return, bits)
 *                          bits (int32 reinterpret): steps in bits 0-15; bits 16-30 =
 *                          visited mask (TSP/TTSP, N <= 15) or 2-bit colour codes (ColourMatch,
 *                          N <= 7: 0 Blue, 1 Green, 2 Red); bit 31 = parity of `episode` (the
 *                          next-layout slot the env's next reset takes, known without a load)
 *    zone_xy   float2[N][B]                      zone centres, plane-major
 *    zone_tmax uint32[ceil(N/2)][B]              TimedTSP only: zone_max_steps, two
 *                                                uint16 per word (zone 2j low half)
 *    cooldown  uint2[B]                          ColourMatch only: one byte per zone
 *    seed      int64[B]    Engine._seed of each env (incremented by every reset)
 *    episode   uint32[B]   resets performed so far
 *    origin    float4[B]   (x0, y0, rot0, 0): the MuJoCo body frame of the episode,
 *                          kept only to convert to/from qpos/qvel
 *    counters  double[8]   sum of episode returns, episodes finished, successes
 *                          (goal_met), sum of episode lengths, resets served from a
 *                          prefetched layout, resets sampled inline, rejected crl_set_goal
 *                          requests, chained-step waits that gave up (must stay 0)
 *  optional next-layout planes (all NULL = no prefetch): the draws of each env's next TWO
 *  Engine.resets (reset number n parks in slot n & 1), made in the background by
 *  crl_prefetch_layouts so that an auto-reset inside crl_step is a copy instead of a
 *  rejection-sampling loop
 *    next_zone_xy float2[2][N][B], next_task uint32[2][ceil(N/2)][B] (TimedTSP timeouts) or
 *    uint32[2][B] (ColourMatch colour codes), next_origin float4[2][B], next_seed int64[2][B]
 *    (the seed the parked layout was drawn for), next_ready uint32[2][B] (0 = slot empty, 2 = layout
 *    parked and task draws pending, 3 = claimed by a running prefetch, 16 + r = ready, filled by
 *    sampler round r)
 *  optional stamp uint32[2][ceil(B/32)]: steps started / finished per group of 32 envs,
 *  see CRL_STEP_CHAINED
 *  optional row_list uint32[4] (CRL_STEP_TRACK_ROWS, crl_host_call_*; word 0 = zone_obs rows moved or counted,
 *  word 1 = result records moved by the host-direct step, words 2-3 unused) and goal int32[B]
 *  (goal-conditioned variants, CRL_STEP_GOALS): see CrlState
 *  outputs, the layout the reference's consumer builds (main/src/utils/format.py:27-28):
 *    obs       float[B][8]      remaining, pos/3 (2), dir (2), vel/1.5 (2), yaw rate/3
 *    zone_obs  float[B][N][Z]   x/3, y/3, r, g, b, 0.25 [, time left | cooldown/150]
 *    result    CrlResult[B]     reward, done, goal_met, integer reward component, need_next_goal
 *    shaped_reward float[B]     info['shaped_reward'] of the goal-conditioned variants
 */
#ifndef CRL_B200_H_
#define CRL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_ABI_VERSION 9
#define CRL_MAX_ZONES 16

/* task ids; reference classes: main/envs/TSP_env.py:11, TTSP_env.py:12, colour_match_env.py:11 */
enum CrlTask { CRL_TASK_TSP = 0, CRL_TASK_TTSP = 1, CRL_TASK_CM = 2 };

enum CrlError {
  CRL_OK = 0,
  CRL_ERR_NULL = -1,        /* a required pointer is NULL */
  CRL_ERR_CONFIG = -2,      /* task / sizes out of range */
  CRL_ERR_ALIGN = -3,       /* a vector plane is not 16-byte aligned */
  CRL_ERR_UNSUPPORTED = -4, /* (task, num_zones) has no compiled kernel */
  CRL_ERR_LAUNCH = -5,      /* CUDA reported an error at launch */
  CRL_ERR_DEVICE = -6       /* no sm_100 device / CUDA runtime failure */
};

/* flags for crl_step */
#define CRL_STEP_AUTO_RESET 1u   /* penv.py:9-10: finished envs restart inside the call */
#define CRL_STEP_PHYSICS_ONLY 2u /* debug/parity: integrate `frameskip` substeps, no task logic */
/* Back-to-back rollout steps.  CRL_STEP_CHAINED: the caller asserts that the kernel enqueued
 * immediately before this call on `stream` is a crl_step (of this or of another CrlState) that
 * did not produce this call's `actions`, and that the previous crl_step of THIS CrlState was
 * made with CRL_STEP_CHAINED or CRL_STEP_CHAIN_START and nothing else touched the state since.
 * The step then orders itself after the previous step of the same CrlState warp by warp
 * (CrlState.stamp: steps started / finished per group of 32 envs, release/acquire) instead of
 * waiting for the whole preceding grid, so the tail of one launch overlaps the head of the
 * next.  CRL_STEP_CHAIN_START: first step of such a run (ordinary whole-grid wait, but it
 * takes part in the stamp protocol).  Both need CrlState.stamp.  Safe inside CUDA graphs: the
 * counts live on the device, nothing per-launch comes from the host.  Steps without either
 * flag never touch the stamps. */
#define CRL_STEP_CHAINED 4u
#define CRL_STEP_CHAIN_START 8u
/* Needs CrlState.row_list.  The step adds to row_list[0] the number of envs whose zone_obs row
 * differs from the row the previous step left there (a zone fired, the env was reset, a
 * ColourMatch cooldown ticked; every TimedTSP env, whose time-left column moves each step).
 * The count is cumulative: the caller zeroes it when it wants a new one.  Implied by the
 * host-direct step (crl_host_call_*). */
#define CRL_STEP_TRACK_ROWS 16u
/* Goal-conditioned variants PointTSP-v3 / PointTTSP-v3 / ColourMatch-v3
 * (zone-goals/envs/TSP_next_city_env.py:52-75, TTSP_next_city_env.py:45-56,
 * colour_match_next_city_env.py:103-133): the step also reads CrlState.goal and writes
 * CrlOut.shaped_reward (distance to the goal zone before minus after the physics; 0 when the
 * goal zone fired; ColourMatch: minus 1 when another zone changed colour) and
 * CrlResult.need_next_goal (goal reached, or episode over), clearing the goal when set. */
#define CRL_STEP_GOALS 32u
/* WaitWrapper (main/envs/wrappers.py:29-54), for step_no_reset rollouts: an env whose episode
 * ends in a step without CRL_STEP_AUTO_RESET is parked; further steps of a parked env change
 * nothing and report an all-zero observation, reward 0, done = 1, until it is reset. */
#define CRL_STEP_WAIT 64u
/* With actions == NULL: the step index of the in-kernel Philox action draw is `step_index` PLUS the
 * number of CRL_STEP_ACTION_COUNTER steps the env's group of 32 has taken so far, kept on the device
 * (third plane of CrlState.stamp).  A launch captured in a CUDA graph and replayed then draws fresh
 * iid U(-1,1)^2 actions per (env, step) at every replay -- action_space.sample() of a random-action
 * rollout -- with nothing coming from the host.  Needs CrlState.stamp. */
#define CRL_STEP_ACTION_COUNTER 128u
/* The step does not build or write zone_obs (CrlOut.zone_obs may be NULL): for a consumer that derives the zone
 * rows from the state planes itself -- crl_zone_encode_state, the fused ZoneEnvModel encoder -- a rollout that only
 * needs the embedding never materialises 360 / 420 / 168 of the 584 / 676 / 336 bytes an env-step moves.  Not with
 * CRL_STEP_TRACK_ROWS or the host-direct step, crl_host_call_* (they ship zone_obs rows). */
#define CRL_STEP_NO_ZONE_OBS 512u
/* Host-direct step (crl_host_call_*), TimedTSP only: host_out->zone_obs is PLANE-major, float[Z][B][N] (the caller
 * views it as (B, N, Z) through strides).  TimedTSP's time-left column moves every step, so with a row-major mirror
 * every row would cross PCIe every step (420 B per env); plane-major, that column is one contiguous [B][N] plane the
 * step writes with coalesced stores (60 B per env), and only the rows of visits and resets touch the other six planes. */
#define CRL_STEP_HOST_PLANES 1024u
/* The step writes only the zone_obs rows whose bytes change -- the rows CRL_STEP_TRACK_ROWS counts: a zone fired, the env
 * was rebuilt by the auto-reset, a ColourMatch cooldown ticked, every TimedTSP row -- and leaves every other row of
 * CrlOut.zone_obs untouched.  PRECONDITION: out->zone_obs holds the rows of the state the step starts from, as a crl_reset
 * of all envs or a step that wrote zone_obs left them.  PointTSP then moves 224 instead of 584 bytes per env-step, plus a
 * row for each zone event and reset.  TimedTSP ignores the flag (its time-left column moves every step).  Not with
 * CRL_STEP_NO_ZONE_OBS, the host-direct step (crl_host_call_step) or the goal-conditioned / WaitWrapper / walled kernels
 * (CRL_STEP_GOALS, CRL_STEP_WAIT, CrlConfig.walled): CRL_ERR_CONFIG.  A library that ignores the bit writes every row:
 * the same bytes. */
#define CRL_STEP_ZONE_OBS_DELTA 2048u

/* how a reset chooses the episode's seed; wrappers.py:10-23 and Engine.seed/reset */
enum CrlSeedMode {
  CRL_SEED_INCREMENT = 0, /* make_test_env: seed once, every reset does _seed += 1 */
  CRL_SEED_FIXED_RANGE = 1 /* FixedSeedsWrapper: each reset re-seeds uniformly in [min_seed, max_seed] */
};

typedef struct CrlConfig {
  int32_t task;          /* CrlTask */
  int32_t num_envs;      /* B */
  int32_t num_zones;     /* N: 15 / 15 / 6 (main/envs/__init__.py:9,45) */
  int32_t num_steps;     /* 2000 (main/envs/__init__.py:13) */
  int32_t frameskip;     /* 10 (Engine frameskip_binom_n, p = 1) */
  int32_t max_cooldown;  /* 150 (colour_match_env.py:16) */
  int32_t seed_mode;     /* CrlSeedMode */
  int32_t env_offset;    /* global index of env 0 of this shard (multi-GPU: rank * B) */
  int64_t min_seed;      /* CRL_SEED_FIXED_RANGE bounds, inclusive */
  int64_t max_seed;
  double zone_size;      /* 0.2 (ZoneEnvBase.py:51) */
  double time_saved_reward; /* 0.01 (TSP_env.py:14) */
  double beta_a;         /* 3.0 (TTSP_env.py:13) */
  double beta_b;         /* 1.5 */
  double robot_keepout;  /* 0.4 (Engine default) */
  double zone_keepout;   /* 0.55 (ZoneEnvBase.py:50) */
  double extent;         /* 3.0 (ZoneEnvBase.py:41) */
  /* TSP / TimedTSP zones that START an episode visited (bit i = zone i): the hard instances
   * PointTSP-v4 / v5 (main/envs/TSP_hard_env.py:27-30, `zones_colours` of
   * main/envs/__init__.py:52-81: Cyan = a city, Yellow = a distractor that counts as visited).
   * 0 for every other registration.  Ignored by ColourMatch. */
  uint32_t initial_visited;
  /* 1: `walled=True` (main/envs/zone_envs/ZoneEnvBase.py:39,55-62): 244 box geoms of half-size 0.1 centred on the
   * square of half-width `extent` at every multiple of 0.1; the robot's sphere collides with them (soft contact,
   * normal rows only: PARITY UNPINNED and simplified -- DESIGN.md 4.9).  No registration of the reference sets it
   * (main/envs/__init__.py:7-50); 0 everywhere else.  A walled env steps through the EXT kernels. */
  uint32_t walled;
} CrlConfig;

typedef struct CrlState {
  float* pose;          /* float4[B] */
  float* aux;           /* float4[B] */
  float* zone_xy;       /* float2[N][B] */
  uint32_t* zone_tmax;  /* uint32[ceil(N/2)][B]; TTSP only */
  uint32_t* cooldown;   /* uint2[B]; ColourMatch only */
  int64_t* seed;        /* int64[B] */
  uint32_t* episode;    /* uint32[B] */
  float* origin;        /* float4[B] */
  double* counters;     /* double[8] */
  float* next_zone_xy;  /* float2[2][N][B]; optional (prefetch) */
  uint32_t* next_task;  /* TTSP: uint32[2][ceil(N/2)][B]; ColourMatch: uint32[2][B]; optional */
  float* next_origin;   /* float4[2][B]; optional */
  int64_t* next_seed;   /* int64[2][B]; optional */
  uint32_t* next_ready; /* uint32[2][B]; optional.  Zero it whenever CrlState.seed is rewritten */
  uint32_t* stamp;      /* uint32[3][ceil(B/32)]; optional, zero-initialised.  Steps started and
                           steps finished for each group of 32 envs (CRL_STEP_CHAINED), and the
                           in-kernel-action steps taken (CRL_STEP_ACTION_COUNTER) */
  uint32_t* prefetch_work; /* 16 (1 + 2 B) bytes, 16-byte aligned: work list of crl_prefetch_layouts
                              (needed with next_*) */
  uint32_t* row_list;   /* uint32[4]; optional (CRL_STEP_TRACK_ROWS, crl_host_call_*): word 0 = number
                           of envs whose zone_obs row changed (or, host-direct, moved), word 1 = result
                           records the host-direct step moved, both cumulative; words 2-3 unused */
  int32_t* goal;        /* int32[B]; optional (CRL_STEP_GOALS): goal_zone of each env, -1 = None.
                           Every reset clears it */
  /* optional LAYOUT BANK (all three NULL = none): the maps of the K = max_seed - min_seed + 1
   * seeds min_seed..max_seed, e.g. exported from the reference (make_train_env's
   * num_training_tasks maps, make_env.py:3-18; evaluate.py's seeds).  A reset that runs with a
   * seed s in that range COPIES entry s - min_seed instead of sampling (in either seed mode;
   * seeds outside the range are sampled as usual), so the device trains / evaluates on exactly
   * the reference's maps, and with CRL_SEED_FIXED_RANGE no sampler is needed at all. */
  const float* bank_zone_xy;   /* float2[K][N] zone centres */
  const float* bank_origin;    /* float4[K]: x0, y0, rot0, 0 */
  const uint32_t* bank_task;   /* TTSP: uint32[K][ceil(N/2)] timeouts packed like zone_tmax;
                                  ColourMatch: uint32[K] colour codes, 2 bits per zone; TSP: NULL */
  /* optional FIXED PLACEMENTS (NULL = none): float4[1 + N], entry 0 the robot, entry 1 + i zone i.
   * Engine's `robot_locations` / `zones_locations` / `robot_rot` (Safety Gym
   * placements_dict_from_object: an object with a location is drawn inside a 2e-9-wide box
   * around it -- here: AT it -- and still has to pass the keepout test against the objects
   * placed before it, else the layout attempt is abandoned), as the hard instances use them
   * (main/envs/__init__.py:52-81).  Entry 0 = (x, y, rot, f) with f = 1 position fixed, 2 heading
   * fixed, 3 both, 0 neither; entry 1 + i = (x, y, 0, f) with f = 1 fixed, 0 sampled.  Read by
   * every sampler (crl_reset, the auto-reset of crl_step, crl_prefetch_layouts); layout banks and
   * crl_reset_from_layout take their positions as given. */
  const float* fixed_layout;
  /* uint32[4], zero-initialised; needed with next_*.  Word 0 = the last sampler round whose parked
   * layouts crl_step / crl_reset may use (written by crl_prefetch_publish). */
  uint32_t* prefetch_epoch;
} CrlState;

typedef struct CrlResult {
  float reward;     /* float reward of the step (dense + time bonus) */
  uint8_t done;
  uint8_t goal_met; /* info['goal_met'] */
  int8_t event;     /* integer reward component: new_city in {0,1} or Hamming delta in {-2..1} */
  uint8_t need_next_goal; /* info['need_next_goal'] (CRL_STEP_GOALS), else 0 */
} CrlResult;

typedef struct CrlOut {
  float* obs;        /* float[B][8] */
  float* zone_obs;   /* float[B][N][Z] */
  CrlResult* result; /* [B] */
  float* shaped_reward; /* float[B]: info['shaped_reward']; optional (CRL_STEP_GOALS) */
} CrlOut;

/* Host-supplied-layout mode (equivalence testing): n layouts in the reference's own
 * units and frame, array-of-structures, fp64 like the reference. */
typedef struct CrlLayoutIn {
  const double* xy0;             /* [n][2]  layout['robot'] */
  const double* rot0;            /* [n]     world_config['robot_rot'] */
  const double* zone_xy;         /* [n][N][2] layout['zone{i}'] */
  const int32_t* zone_max_steps; /* [n][N]  TTSP (TTSP_env.py:19-21), else NULL */
  const int32_t* colours;        /* [n][N]  ColourMatch codes 0/1/2 (colour_match_env.py:57-68), else NULL */
} CrlLayoutIn;

int crl_abi_version(void);
const char* crl_strerror(int code);

/* Bytes the caller must allocate for each plane of CrlState / CrlOut, in the order
 * pose, aux, zone_xy, zone_tmax, cooldown, seed, episode, origin, counters, next_zone_xy,
 * next_task, next_origin, next_seed, next_ready, obs, zone_obs, result, stamp,
 * prefetch_work, row_list, goal, shaped_reward, prefetch_epoch (CRL_NUM_PLANES entries; 0 = plane unused by
 * this task).  Writes the first min(n, CRL_NUM_PLANES) entries of out_bytes. */
#define CRL_NUM_PLANES 23
int crl_plane_bytes(const CrlConfig* cfg, int64_t* out_bytes, int32_t n);

/* Algorithmic HBM bytes one env-step moves in this layout: read, written.  The written figure counts the whole zone_obs
 * row; a CRL_STEP_ZONE_OBS_DELTA step writes that row only when it changes. */
int crl_step_bytes(const CrlConfig* cfg, int64_t* bytes_read, int64_t* bytes_written);

/* Engine.reset() for the envs with mask[e] != 0 (all envs if mask == NULL): choose the
 * seed per cfg->seed_mode, draw timeouts / colours and the layout on the device with
 * Philox4x32-10, zero the physics state, write the first observation.
 * Replaces Engine.reset -> build_layout/sample_layout -> World.rebuild, and
 * TTSP_env.py:73-76 / colour_match_env.py:125-127. */
int crl_reset(const CrlConfig* cfg, const CrlState* st, const CrlOut* out,
              const uint8_t* mask, void* stream);

/* Fill the empty next-layout slots (see CrlState.next_*): for each env whose slot is
 * empty, draw its NEXT reset now.  Meant to be launched every few steps on a stream other
 * than the stepping one.  Hides Engine.build_layout's rejection sampling, which the reference
 * runs inside reset() (penv.py:9-10).  The sampler runs one lane per env on `warps_per_sm`
 * persistent warps per SM (0 = default 2: a background job beside the steps; up to 32 before a
 * full crl_reset, where nothing else is running).
 * ORDERING (ABI 6: stream order instead of acquire/release flags, so that the step's reset path is
 * one batch of plain loads).  `round` numbers the call, 1, 2, 3 ... per CrlState, increasing.
 *  - the call must be ordered AFTER the steps whose finished envs it is to serve (enqueue it on a
 *    stream that has waited for the stepping stream), and rounds of one CrlState must not overlap;
 *  - slots it fills are marked "ready, round r" and crl_step ignores them (samples inline, with the
 *    identical result) until crl_prefetch_publish(st, r, stepping_stream) has been enqueued on the
 *    stepping stream AFTER that stream waited for round r to finish.  Steps enqueued behind the
 *    publish see everything the round wrote by stream order.
 * The step never waits for the sampler as long as the caller publishes a round a few steps after
 * launching it (vec_env.ZoneVecEnv.tick publishes round r - 2 when it launches round r). */
int crl_prefetch_layouts(const CrlConfig* cfg, const CrlState* st, int32_t warps_per_sm,
                         uint32_t round, void* stream);
int crl_prefetch_publish(const CrlState* st, uint32_t round, void* stream);

/* The same reset with the layout handed in (device arrays, see CrlLayoutIn) for
 * envs env_ids[0..n) (env_ids == NULL: envs 0..n). */
int crl_reset_from_layout(const CrlConfig* cfg, const CrlState* st, const CrlOut* out,
                          const CrlLayoutIn* layout, const int32_t* env_ids, int32_t n,
                          void* stream);

/* One env.step() of every env: TSPEnv.step / TimedTSPEnv.step / ColourMatchEnv.step
 * over Engine.step (TSP_env.py:45-49, TTSP_env.py:62-71, colour_match_env.py:95-101).
 * actions: float[B][2] device, or NULL to draw U(-1,1)^2 in-kernel from
 * Philox(key = action_seed, counter = (global env, step_index)). */
int crl_step(const CrlConfig* cfg, const CrlState* st, const float* actions,
             const CrlOut* out, uint32_t flags, uint64_t action_seed,
             uint64_t step_index, void* stream);

/* crl_step with HOST buffers (pinned or pageable): copies actions host->device into
 * `actions_dev`, steps, copies obs / zone_obs / result (and, with CRL_STEP_GOALS, shaped_reward
 * if host_out has it) device->host into `host_out`, then synchronises the stream.  The reference-facing call ParallelEnv.step makes. */
int crl_step_host(const CrlConfig* cfg, const CrlState* st, const float* actions_host,
                  float* actions_dev, const CrlOut* out, const CrlOut* host_out,
                  uint32_t flags, void* stream);

/* The HOST-DIRECT step: crl_step_host for a caller that keeps its host observation buffers between calls (as
 * ParallelEnv's consumers do: the obs of step t is only read before step t+1), in ONE kernel and a stream synchronisation
 * per call.  No staging and no copy-engine transfers: the step kernel reads the actions from, and writes obs / result /
 * shaped_reward AND every zone_obs row it changed straight to, the caller's host buffers (actions_host and all of
 * host_out), which must be page-locked and device-mapped (cudaHostAlloc; CRL_ERR_CONFIG otherwise).  zone_obs is 60-90 %
 * of a step's output bytes and almost all of it repeats the previous step (zone centres never move inside an episode; a
 * colour changes only when a zone fires), so only the rows that CHANGED cross PCIe.  PRECONDITION: host_out->zone_obs
 * holds the device zone_obs as of the previous step (e.g. left there by crl_step_host or by a full copy after crl_reset).
 * Result records are treated like zone_obs rows: a record (all zeros except on an event, a done or a goal change) is
 * written to host_out->result only when it differs from the one there, which the kernel knows from the device copy
 * out->result (updated by every step) -- PRECONDITION: host_out->result holds out->result as of the previous step, as
 * crl_step_host leaves it.  What the caller sees is byte-identical to crl_step_host's.  Needs CrlState.row_list:
 * row_list[0] counts the zone_obs rows moved and row_list[1] the result records moved, cumulatively.  The device copies
 * CrlOut.obs / shaped_reward are NOT updated by such a call (zone_obs and result are).
 * The call is PREPARED: what ParallelEnv.step (penv.py:52-59) does once per frame with the same envs and the same buffers
 * is resolved once -- the device aliases of the caller's page-locked host buffers, the flags -- so that a per-frame call
 * carries three arguments (a ctypes / cgo / JNI binding pays per argument: 3.5 us for eleven against 0.9 us for three
 * through ctypes).  crl_host_call_create: `cfg` and `st` are kept BY POINTER (the caller keeps them alive and may change
 * their fields between steps); `out` and `host_out` are read now; `flags` as for crl_step (CRL_STEP_TRACK_ROWS implied;
 * CRL_STEP_HOST_PLANES for a plane-major TimedTSP mirror).  crl_host_call_step: one step; `actions_host` float[B][2],
 * page-locked and device-mapped (CRL_ERR_CONFIG otherwise); the stream is synchronised before it returns.  A call object
 * is used by one thread at a time; the host buffers it was created with (and the action buffers it has seen) stay
 * allocated and page-locked while it lives. */
typedef struct CrlHostCall CrlHostCall;
int crl_host_call_create(const CrlConfig* cfg, const CrlState* st, const CrlOut* out, const CrlOut* host_out,
                         uint32_t flags, CrlHostCall** call);
int crl_host_call_step(CrlHostCall* call, const float* actions_host, void* stream);
void crl_host_call_destroy(CrlHostCall* call);

/* Goal RPCs of the goal-conditioned variants, one call for the whole batch instead of one pipe
 * message per env (zone-goals/src/torch_ac/torch_utils/penv.py:18-25, 75-99).
 * crl_set_goal: env.set_goal(goals[e]) for every e with goals[e] >= 0 (device int32[B]); what
 * the reference asserts (index in range; TSP / TimedTSP: zone not yet visited) is checked on
 * the device: an invalid request leaves the goal unset and adds 1 to counters[6].
 * crl_goal_query: any of needs_goal uint8[B] (goal_zone is None), goal_xy float[B][2]
 * (get_goal: zone centre / 3; zeros where there is no goal), available uint8[B][N]
 * (get_available_goals); NULL = not wanted.  All device pointers. */
int crl_set_goal(const CrlConfig* cfg, const CrlState* st, const int32_t* goals, void* stream);
int crl_goal_query(const CrlConfig* cfg, const CrlState* st, float* goal_xy, uint8_t* needs_goal,
                   uint8_t* available, void* stream);

/* Physics state in the reference's own coordinates (sim.data.qpos / qvel, fp64, device
 * arrays [n][3]) for envs env_ids[0..n) (NULL: 0..n).  set: teacher forcing for the
 * per-substep parity tests; get: export. */
int crl_set_qpos_qvel(const CrlConfig* cfg, const CrlState* st, const double* qpos,
                      const double* qvel, const int32_t* env_ids, int32_t n, void* stream);
int crl_get_qpos_qvel(const CrlConfig* cfg, const CrlState* st, double* qpos, double* qvel,
                      const int32_t* env_ids, int32_t n, void* stream);

/* Advantages of one rollout, on the device, from the records crl_step wrote
 * (main/src/torch_ac/algos/base.py:195-205; SURVEY.md 8f rank 3).  A rollout of T frames keeps
 * T + 1 result slots [T+1][B]: slot t + 1 is CrlOut.result of step t (point CrlOut at the slot:
 * the step writes its outputs in place, nothing is copied), slot 0 is the last slot of the
 * previous rollout (zeros at first: no env finished yet).  reward[t] = slot[t+1].reward -- or
 * reward_override[(t+1) B + e] if not NULL (info['shaped_reward'], base.py:155-159) --,
 * masks[t] = 1 - slot[t].done, the mask after the last step = 1 - slot[T].done:
 *   delta = reward[t] + discount v[t+1] mask[t+1] - v[t]
 *   A[t]  = delta + discount gae_lambda A[t+1] mask[t+1],   v[T] = next_value, A[T] = 0
 * evaluated in float32 operation by operation as torch does, so the result is bit-identical to
 * the reference's.  values, advantages, returns (= values + advantages, may be NULL): float[T][B];
 * next_value: float[B].  All device pointers. */
int crl_gae(const CrlResult* results, const float* reward_override, const float* values,
            const float* next_value, double discount, double gae_lambda, int32_t num_frames,
            int32_t num_envs, float* advantages, float* returns, void* stream);

/* Failure detection: counts, per kind, the envs whose state planes violate an invariant that
 * only a stray write or a broken reset could violate.  violations: device uint64[8] =
 * {non-finite body state, heading outside [-pi, pi], step count above num_steps (and not the
 * parked sentinel), zone centre outside the placement extents, visited / colour / cooldown bits
 * out of range, next-layout flag out of range, goal outside [-1, N), TimedTSP timeout above
 * num_steps}.  All zeros = healthy.  Asynchronous on `stream`. */
int crl_check_state(const CrlConfig* cfg, const CrlState* st, uint64_t* violations, void* stream);

/* ---- the consumer of the observation: ZoneEnvModel's zone encoder (SURVEY.md 8f rank 2) ----
 * main/src/env_model.py:56-78: zone_net_ = Linear(obs_dim + Z, h), ReLU, Linear(h, h), ReLU, Linear(h, h)
 * applied to [obs[e], zone_obs[e][z]] for every zone, then the mean over the env's zones.  The third
 * Linear is affine, so the mean commutes with it:
 *     zone_emb = W3 pooled + b3,   pooled[e] = mean_z relu(W2 relu(W1 [obs[e], zone_obs[e][z]] + b1) + b2)
 * crl_zone_encode computes `pooled` in one fused kernel on the tensor cores (tcgen05, bf16 operands,
 * fp32 accumulation in TMEM; csrc/crl_encode.cu): the (B N, h) activations the reference materialises
 * never leave the SM, and the third Linear shrinks from B N to B rows -- it and combine_net_ stay
 * fp32 library GEMMs on the caller's side.  The rollout-time forward of BaseAlgo.collect_experiences
 * (base.py:133-140); crl_zone_encode_backward (below) is the training half.  hidden <= 190 (the default is 185,
 * scripts/train_ppo.py:66), obs_dim + zone_dim <= 31 (one K step up to 15, two beyond: ZoneEnvGoalModel /
 * ZoneEnvSkillModel, whose per-env goal / one-hot skill the caller concatenates to obs), num_zones <= 16. */
typedef struct CrlEncoderShape {
  int32_t obs_dim;    /* 8 */
  int32_t zone_dim;   /* Z */
  int32_t hidden;     /* h */
  int32_t num_zones;  /* N */
} CrlEncoderShape;
/* bytes of the packed-weights buffer (device, 16-byte aligned) */
int crl_encoder_packed_bytes(const CrlEncoderShape* shape, int64_t* bytes);
/* fp32 torch-layout weights of the first two Linears ([out][in], device) -> the bf16 shared-memory
 * image the kernel keeps resident */
int crl_encoder_pack(const CrlEncoderShape* shape, const float* w1, const float* b1, const float* w2,
                     const float* b2, void* packed, void* stream);
/* pooled float[B][h] (see above).  obs float[B][obs_dim], zone_obs float[B][N][Z] (CrlOut's layout),
 * all device.  status: optional device int32, set to 1 if a tensor-core completion wait expired
 * (results then undefined); the kernel never hangs. */
int crl_zone_encode(const CrlEncoderShape* shape, int32_t num_envs, const float* obs, const float* zone_obs,
                    const void* packed, float* pooled, int32_t* status, void* stream);
/* The same with the zone part of every input row BUILT FROM THE STATE PLANES (CrlState.aux, zone_xy, zone_tmax /
 * cooldown; cfg gives task, sizes, num_steps, max_cooldown) instead of read from a materialised zone_obs: bit for bit
 * the rows the step writes (main/envs obs_zones: x/3, y/3, r, g, b, 0.25 [, time left | cooldown / 150]), so
 * `pooled` is bit-identical to crl_zone_encode on the step's own zone_obs.  Reads 32 + 8 N (+ 4 ceil(N/2) | 8) + 4
 * bytes per env instead of 32 + 4 N Z; with CRL_STEP_NO_ZONE_OBS the step does not write zone_obs at all.
 * obs: the step's CrlOut.obs, float[B][obs_dim = 8]. */
int crl_zone_encode_state(const CrlEncoderShape* shape, const CrlConfig* cfg, const CrlState* st, const float* obs,
                          const void* packed, float* pooled, int32_t* status, void* stream);

/* The rest of ZoneEnvModel.forward (env_model.py:76-79): out = combine_net_([obs, L3(pooled)]).  Both Linears are
 * affine, so this is ONE GEMM  out[e] = W' [obs[e], pooled[e], 1]  with W' = [Wc_obs | Wc_emb W3], b' = Wc_emb b3 + bc
 * folded by the caller; crl_encoder_head runs it on the tensor cores as well (tcgen05, bf16 operands, fp32
 * accumulation, folded weights resident in shared memory; bound by reading (obs, pooled) and writing out once), so
 * the whole forward is two kernels of this library and no library GEMM.  With w = [0 | W3], b = b3 the same call
 * yields zone_emb = L3(pooled).  w: float[h][obs_dim + h] (torch layout), b: float[h], all device pointers. */
int crl_encoder_head_packed_bytes(const CrlEncoderShape* shape, int64_t* bytes);
int crl_encoder_pack_head(const CrlEncoderShape* shape, const float* w, const float* b, void* packed, void* stream);
int crl_encoder_head(const CrlEncoderShape* shape, int32_t num_envs, const float* obs, const float* pooled,
                     const void* packed_head, float* out, int32_t* status, void* stream);

/* The whole ZoneEnvModel.forward (env_model.py:66-79) in two launches with NO fp32 `pooled` in between: the zone kernel
 * writes the head kernel's input -- per tile of 128 envs the bf16 operand image [obs, pooled, 1, 1, 0..] -- into
 * `workspace` (crl_encoder_workspace_bytes; contents are scratch), and the head kernel fetches each tile with one bulk
 * copy.  Same result as crl_zone_encode + crl_encoder_head (the head rounds `pooled` to bf16 either way).  `st` != NULL:
 * the zone rows are built from the state planes (as crl_zone_encode_state; `cfg` is the env's, `zone_obs` unused);
 * `st` == NULL: from the materialised `zone_obs`.  Needs obs_dim == 8 and zone_dim <= 7 (ZoneEnvModel's own shape),
 * otherwise CRL_ERR_UNSUPPORTED: use the two calls. */
int crl_encoder_workspace_bytes(const CrlEncoderShape* shape, int32_t num_envs, int64_t* bytes);
int crl_encoder_forward(const CrlEncoderShape* shape, const CrlConfig* cfg, const CrlState* st, int32_t num_envs,
                        const float* obs, const float* zone_obs, const void* packed, const void* packed_head,
                        void* workspace, float* out, int32_t* status, void* stream);

/* PRECISE mode of the fused zone kernel: every operand split into two bf16 terms (x = hi + lo), every product three
 * tensor-core MMAs (hi hi + lo hi + hi lo), fp32 accumulation, fp32 biases in the epilogues -- `pooled` agrees with the
 * fp32 reference module (env_model.py:56-78) to ~1e-5 of its largest value instead of the fast kernel's 3-5e-3, at about
 * 7x its time (one tile in flight per CTA): the like-for-like / validation mode.  Own packed image (hi and lo of both layers + fp32 biases);
 * needs obs_dim + zone_dim <= 16.  The remaining (B, h) affine map of the forward reaches the same accuracy with
 * three launches of crl_encoder_head: (W, X), (W - bf16 W, X), (W, X - bf16 X) (encoder.py does that). */
int crl_encoder_precise_packed_bytes(const CrlEncoderShape* shape, int64_t* bytes);
int crl_encoder_pack_precise(const CrlEncoderShape* shape, const float* w1, const float* b1, const float* w2,
                             const float* b2, void* packed, void* stream);
int crl_zone_encode_precise(const CrlEncoderShape* shape, int32_t num_envs, const float* obs, const float* zone_obs,
                            const void* packed_precise, float* pooled, int32_t* status, void* stream);

/* BACKWARD of `pooled` (the B N-row part of ZoneEnvModel; training through the fused kernel): given
 * grad_pooled g = dL/dpooled float[B][h], the gradients of the first two Linears in torch layout, fp32:
 * dw1 float[h][obs_dim + zone_dim], db1 float[h], dw2 float[h][h], db2 float[h] (all overwritten, device).  The third
 * Linear and combine_net_ act on B rows and stay with the caller (torch autograd on `pooled`).  No input gradients.
 * `packed` is crl_encoder_pack's image of the weights the forward used; obs / zone_obs as for crl_zone_encode.
 * Numerics: H1 and the layer-2 pre-activation are recomputed exactly as crl_zone_encode computes them (bf16 operands,
 * fp32 accumulation, bf16 hi + lo biases); then, per row m of env e,
 *     dH2[m][i] = acc2[m][i] > 0 ? bf16_rn(fp32(g[e][i] * fp32(1/N))) : 0     (select: a masked-off NaN g gives 0)
 *     dH1[m][j] = H1[m][j] > 0 ? bf16_rn(sum_i W2[i][j] dH2[m][i]) : 0          (bf16 W2, fp32 accumulation)
 *     dW2 = sum_m dH2[m]^T H1[m],  db2 = sum_m dH2[m],  dW1 = sum_m dH1[m]^T x[m],  db1 = sum_m dH1[m]
 * with bf16 operands; padding slots contribute exact zeros.  Launch rule: the rows are cut into tiles of 64 (4 envs of 16
 * slots, or 8 of 8 when N <= 8); grid = min(tiles, SMs of the current device); CTA c sums tiles c, c + grid, ... in fp32
 * (at most 64 ceil(tiles / grid) rows per partial) into its own fp32 partial in `workspace`
 * (crl_encoder_backward_workspace_bytes; contents are scratch), and a second kernel adds the partials in CTA order in
 * fp64 and rounds once to fp32.  No float atomics: the result is bit-identical from run to run for the same B on the
 * same device.  Same shapes as crl_zone_encode; packed and workspace 16-byte aligned.  status as for crl_zone_encode. */
int crl_encoder_backward_workspace_bytes(const CrlEncoderShape* shape, int32_t num_envs, int64_t* bytes);
int crl_zone_encode_backward(const CrlEncoderShape* shape, int32_t num_envs, const float* obs, const float* zone_obs,
                             const void* packed, const float* grad_pooled, void* workspace,
                             float* dw1, float* db1, float* dw2, float* db2, int32_t* status, void* stream);

/* ---- rollout frames: the zone rows of a stored frame as a 16-byte record plus a per-episode layout ----
 * A zone row (x/3, y/3, r, g, b, 0.25 [, time left | cooldown / max_cooldown]) depends on the zone centres (and TimedTSP
 * timeouts), which change only at a reset, on the state word aux.w and on the ColourMatch cooldown bytes -- not on the
 * robot.  So a rollout can store, per env and frame, one CrlFrame instead of the N Z floats of zone_obs (360 / 420 / 168
 * bytes for PointTSP / TimedTSP / ColourMatch), and each episode's layout once, in a LAYOUT TABLE of `capacity` entries:
 *   layout_xy   float2[capacity][N]            zone centres of entry k, row-major per entry
 *   layout_tmax uint32[capacity][ceil(N/2)]    TimedTSP timeouts packed like CrlState.zone_tmax; NULL for the other tasks
 *   fill        uint32[2]                      entries handed out (<= capacity), entries requested
 * The same format serves every task.  CrlFrame.layout == CRL_FRAME_NO_LAYOUT: the capture that should have taken an entry
 * found the table full; every row built from such a record is NaN in all its features (the rows of other records are not
 * affected), and fill[1] > capacity tells the caller how many entries it would have needed. */
typedef struct CrlFrame {
  uint32_t bits;         /* aux.w verbatim: steps, visited mask / colour codes, episode parity */
  uint32_t layout;       /* entry of the layout table, or CRL_FRAME_NO_LAYOUT */
  uint32_t cooldown[2];  /* ColourMatch: CrlState.cooldown of the env (one byte per zone); 0 for the other tasks */
} CrlFrame;
#define CRL_FRAME_NO_LAYOUT 0xffffffffu

/* Record frame t of every env after a step (a kernel of its own, launched behind crl_step): frames_t[e] = {aux.w, layout,
 * cooldown}.  An env whose `result[e].done` is set -- or every env when `initial` != 0 -- takes a new table entry (one
 * atomic per warp on fill[1]) and copies its zone_xy (and zone_tmax) into it; any other env keeps the entry of its
 * previous record, which must lie at frames_t - num_envs (slot t - 1 of a [T + 1][B] array; not read when `initial`).
 * The order in which entries are handed out is not deterministic; the rows built from the records are.  `result` may be
 * NULL when `initial` != 0.  frames_t 16-byte aligned, capacity >= 1. */
int crl_frame_capture(const CrlConfig* cfg, const CrlState* st, const CrlResult* result, int32_t initial,
                      CrlFrame* frames_t, float* layout_xy, uint32_t* layout_tmax, uint32_t capacity, uint32_t* fill,
                      void* stream);
/* crl_zone_encode with the zone part of each of the M input rows built from frames[m] and the layout table (any flat or
 * gathered set of records, with their obs rows float[M][8]): bit-identical to crl_zone_encode on the rows
 * crl_frames_zone_obs materialises.  `cfg` is the env's (task, num_zones, num_steps, max_cooldown).  Needs obs_dim == 8
 * (CRL_ERR_UNSUPPORTED otherwise) and the task's zone_dim and num_zones (CRL_ERR_CONFIG otherwise). */
int crl_zone_encode_frames(const CrlEncoderShape* shape, const CrlConfig* cfg, int32_t num_rows, const float* obs,
                           const CrlFrame* frames, const float* layout_xy, const uint32_t* layout_tmax, const void* packed,
                           float* pooled, int32_t* status, void* stream);
/* crl_zone_encode_backward on the same rows: same workspace (crl_encoder_backward_workspace_bytes for num_rows), same
 * launch rule and fixed-order fp64 reduction, bit-identical to crl_zone_encode_backward on the materialised rows. */
int crl_zone_encode_backward_frames(const CrlEncoderShape* shape, const CrlConfig* cfg, int32_t num_rows, const float* obs,
                                    const CrlFrame* frames, const float* layout_xy, const uint32_t* layout_tmax,
                                    const void* packed, const float* grad_pooled, void* workspace, float* dw1, float* db1,
                                    float* dw2, float* db2, int32_t* status, void* stream);
/* The rows themselves: zone_obs float[num_rows][N][Z], bit for bit what the step wrote for those frames. */
int crl_frames_zone_obs(const CrlConfig* cfg, int32_t num_rows, const CrlFrame* frames, const float* layout_xy,
                        const uint32_t* layout_tmax, float* zone_obs, void* stream);

/* ---- env copies: snapshot, restore and branch individual envs ----
 * Copy env src_ids[i] of (src_cfg, src, src_out) onto env dst_ids[i] of (dst_cfg, dst, dst_out), i < n.  NULL ids: 0..n-1.
 * Copied bit for bit, per env: pose, aux (steps, visited mask / colour codes, return, episode parity), every zone row of
 * zone_xy (plane-major on both sides, each with its own B), seed, episode, origin, zone_tmax (TimedTSP), cooldown
 * (ColourMatch), goal when both states have that plane; and, when src_out and dst_out are both given, the obs row, the
 * zone_obs row, the result record and shaped_reward -- each output field that is non-NULL on both sides (a field, or an
 * out struct, given on one side only is CRL_ERR_NULL).  Not copied: counters (a copy is not an episode), stamp, row_list,
 * prefetch_* and next_*.  Both next_ready slots of every dst env written are cleared (when dst->next_ready is set): their
 * layouts were drawn for the old seed and episode, and the step samples inline, with the identical result, until a
 * sampler round refills them.
 * Host checks, before any launch: the configs must agree in every field but num_envs, env_offset, seed_mode, min_seed and
 * max_seed (CRL_ERR_CONFIG); NULL and alignment of the planes the task needs; n < 0 is CRL_ERR_CONFIG, n == 0 launches
 * nothing.  On the device, a pair whose src or dst id is out of range is skipped and counted in *rejected (optional,
 * device uint32, cumulative).  No host synchronisation: the call can be captured in a CUDA graph.
 * PRECONDITIONS (not checked): the dst ids are distinct; when src and dst are the same state, the src and dst id sets
 * are disjoint (copy through a second state to permute envs in place).
 * WHAT A COPY GUARANTEES: the step is a pure function of the state and the action, so a dst env that then takes the same
 * actions as its src produces the same outputs and state, bit for bit -- through auto-resets too under
 * CRL_SEED_INCREMENT and with a layout bank, since the next seed is the copied one and the timeouts, colours and layout are
 * functions of it.  Under CRL_SEED_FIXED_RANGE the next seed is drawn from the dst's global env index, and in-kernel
 * actions (actions == NULL) are keyed by it as well: a copy then matches its src until its episode ends, and branches
 * stepped with in-kernel actions diverge by construction. */
int crl_copy_envs(const CrlConfig* dst_cfg, const CrlState* dst, const CrlOut* dst_out, const int32_t* dst_ids,
                  const CrlConfig* src_cfg, const CrlState* src, const CrlOut* src_out, const int32_t* src_ids,
                  int32_t n, uint32_t* rejected, void* stream);

/* Copies the eight counters to the host (synchronises `stream`).  The first four (sum of
 * returns, episodes, successes, sum of lengths) are what ranks all-reduce. */
int crl_counters_read(const CrlState* st, double out[8], void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRL_B200_H_ */
