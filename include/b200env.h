/* b200env.h -- C-ABI of libb200env.so, the B200-native vector-env step engine.
 *
 * Drop-in boundary for Gymnasium's vectorised step()/reset() hot path.  Gymnasium (v1.4.0) is pure Python; the
 * interfaces these entry points replace are (paths relative to the reference tree):
 *   - SyncVectorEnv.reset / .step          gymnasium/vector/sync_vector_env.py:187-264, :266-337
 *   - AsyncVectorEnv.step_async/step_wait  gymnasium/vector/async_vector_env.py:440-521 (+ worker loop :773-904)
 *   - TimeLimit.step / .reset              gymnasium/wrappers/common.py:116-151
 *   - seeding.np_random                    gymnasium/utils/seeding.py:10-42
 *   - per-family dynamics, cited at each declaration below.
 * The reference-side binding is a ctypes stub inside a VectorEnv subclass registered as a spec's
 * `vector_entry_point` (gymnasium/envs/registration.py:933-963); see INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, a negative B2E_E* code for an argument error, or a positive cudaError_t;
 *     b2e_last_error() returns a thread-local message for the last non-zero return.
 *   - all array pointers are DEVICE pointers owned by the caller (torch allocates them); nothing is allocated,
 *     freed or synchronised inside a call; kernels are enqueued on `stream` (a cudaStream_t passed as void*).
 *   - shapes are given per argument; "n" is the number of envs in this shard (b2e_batch.n).
 *   - bool outputs are 1 byte (0/1), i.e. torch.bool / numpy.bool_ storage.
 */
#ifndef B200ENV_H_
#define B200ENV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2E_VERSION 1

/* error codes */
#define B2E_EINVAL (-1)  /* bad argument (null pointer, bad enum, n < 0) */
#define B2E_ENODEV (-2)  /* no CUDA device / wrong architecture */
#define B2E_ETIMEOUT (-3) /* a host-side wait (b2e_pipe_submit: consumer acknowledgement) timed out */

/* autoreset modes: gymnasium/vector/vector_env.py:34-39 */
#define B2E_AUTORESET_NEXT_STEP 0
#define B2E_AUTORESET_SAME_STEP 1
#define B2E_AUTORESET_DISABLED 2

/* rng modes */
#define B2E_RNG_NUMPY 0  /* per-env numpy Generator(PCG64(SeedSequence(seed+i))) streams, bit-exact */
#define B2E_RNG_PHILOX 1 /* stateless Philox4x32-10 keyed by (seed, global env index, call counter) */

/* action dtypes */
#define B2E_ACT_I64 0
#define B2E_ACT_I32 1
#define B2E_ACT_U8 2
#define B2E_ACT_F32 3
#define B2E_ACT_F64 4

/* Batch descriptor shared by every family (passed by pointer, host memory). */
typedef struct b2e_batch {
  int64_t n;                 /* envs in this shard */
  int64_t env_offset;        /* global index of this shard's env 0 (multi-GPU sharding; seeds are seed+offset+i) */
  int32_t max_episode_steps; /* TimeLimit; <= 0 disables truncation */
  int32_t autoreset_mode;    /* B2E_AUTORESET_* */
  int32_t rng_mode;          /* B2E_RNG_* */
  int32_t action_dtype;      /* B2E_ACT_* */
  uint64_t philox_seed;      /* B2E_RNG_PHILOX only */
  uint64_t call_counter;     /* B2E_RNG_PHILOX only: index of this reset/step call (the caller increments it) */
} b2e_batch;

int b2e_version(void);
const char* b2e_last_error(void);
/* sm_count / cc may be NULL. Returns B2E_ENODEV when no device. */
int b2e_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes);

/* ---- single host-side batch: what AsyncVectorEnv's shared-memory observations are on the reference side (one buffer all
 * workers write their slice of, gymnasium/vector/async_vector_env.py:234-245, :849-852 `write_to_shared_memory`).  Here
 * every GPU rank of a node maps ONE host buffer, page-locks it in its own CUDA context (b2e_host_register) and DMAs its
 * shard's packed step outputs into its slice over its own PCIe link (b2e_copy_to_host_async on the caller's copy stream);
 * see gymnasium_b200/distributed.py: HostBatch.  `host` is a HOST pointer (the only ones in this ABI). */
int b2e_host_register(void* host, size_t bytes);
int b2e_host_unregister(void* host);
/* One segment of a step's outputs: `height` rows of `width` bytes (height 1 = a contiguous run; struct-of-arrays outputs such as
 * Humanoid's info[13][n] land in the global [13][N_total] array as a pitched copy). */
typedef struct b2e_copy_seg {
  void* host_dst;      /* inside a b2e_host_register'ed buffer */
  const void* dev_src; /* device memory, or page-locked host memory (the sequence word's source) */
  size_t dst_pitch, src_pitch; /* bytes between rows (ignored when height == 1) */
  size_t width, height;
} b2e_copy_seg;
/* Enqueues the device->host copies of `count` segments on `stream`, in order (a trailing 8-byte segment is how a rank publishes
 * its sequence word behind the data). */
int b2e_copy_to_host_async(const b2e_copy_seg* segs, int32_t count, void* stream);

/* ---- the whole pipelined step in ONE host call: what AsyncVectorEnv.step_async (gymnasium/vector/async_vector_env.py:440-
 * 475: send the actions to the workers) plus the workers' write of their results into the shared buffer (:849-852) are on
 * the reference side.  A slot bundles everything that is fixed for one (staging buffer, output set, landing slot) triple:
 *   staging_host / actions_dev / action_bytes : page-locked staging buffer and the device buffer the step reads actions from
 *   calls / ncalls : the family's step for this output set, recorded as C-ABI calls of THIS header (function address + its
 *                    arguments; every argument of every step entry point is a pointer or an integer, i.e. one machine word)
 *   segs / nsegs   : the output segments (b2e_copy_seg) of this output set, then two 8-byte segments whose last one's
 *                    host_dst is the rank's sequence word (the landing kernel lands the first nsegs - 2 and stores the word)
 *   ev_*           : cudaEvent_t, owned by the slot (b2e_pipe_slot_init / _destroy)
 * b2e_pipe_submit(slot, host_actions, ...): memcpy into the staging buffer (skipped with B2E_PIPE_ACTIONS_PINNED: the DMA
 * reads the caller's page-locked buffer), async H2D on main_stream, the recorded step,
 * then on copy_stream (ordered after the step) the landing kernel -- after the consumer's acknowledgement word *ack_word has
 * reached need_ack (spin, timeout_s).  Never synchronises a stream; returns B2E_ETIMEOUT if the consumer stalls. */
typedef struct b2e_call {
  void* fn;
  int32_t nargs;
  int32_t _pad;
  uint64_t args[16];
} b2e_call;
typedef struct b2e_pipe_slot {
  void* staging_host;
  void* actions_dev;
  size_t action_bytes;
  const b2e_call* calls;
  b2e_copy_seg* segs;
  int32_t ncalls, nsegs;
  void *ev_h2d, *ev_step, *ev_copy;
  int32_t h2d_pending, copy_pending;
  void* land; /* landing-kernel plan, owned by the slot (b2e_pipe_slot_land_kernel); b2e_pipe_submit needs it */
} b2e_pipe_slot;
#define B2E_PIPE_ACTIONS_PINNED 1 /* host_actions is page-locked and stays untouched until the step has landed: no staging copy */
int b2e_pipe_slot_init(b2e_pipe_slot* slot);
/* The landing KERNEL: the slot's output rows are stored into the page-locked host batch by the SMs (zero-copy stores over
 * PCIe, 16 bytes per thread) in ONE launch that also publishes the sequence word (system-scope fence, last CTA stores it) --
 * no per-key copy-engine set-up, no bounce word.  Needs the host batch mapped (b2e_host_register does) and <= 8 output keys. */
int b2e_pipe_slot_land_kernel(b2e_pipe_slot* slot);
/* The same kernel without a slot (HostBatchPipeline's Python path, scripts/link_probe.py): a plan holds the device-visible
 * addresses of `count` (<= 8) segments whose host_dst lie in a b2e_host_register'ed buffer, and of the sequence word. */
int b2e_land_plan_create(const b2e_copy_seg* segs, int32_t count, int64_t* seq_host, void** plan);
int b2e_land_plan_launch(void* plan, int64_t seq_value, void* stream);
int b2e_land_plan_destroy(void* plan);
int b2e_pipe_slot_destroy(b2e_pipe_slot* slot);
/* seq_value (= step index + 1) is the sequence word the landing kernel publishes behind the step's rows. */
int b2e_pipe_submit(b2e_pipe_slot* slot, const void* host_actions, void* main_stream, void* copy_stream,
                    const int64_t* ack_word, int64_t need_ack, int64_t seq_value, int32_t flags, double timeout_s);

/* ---- RNG: gymnasium/utils/seeding.py:39-41 -> numpy SeedSequence -> PCG64 ---------------------------------------
 * rng   : uint64 [2][n][2]  = {state(lo,hi)}[n] then {inc(lo,hi)}[n]
 * seeds : uint64 [n] device, or NULL => seed_i = base_seed + env_offset + i  (SyncVectorEnv.reset seed+i, :205-208)
 * mask  : uint8 [n] device or NULL (all) -- only masked lanes are re-seeded
 */
int b2e_rng_seed(const b2e_batch* b, uint64_t base_seed, const uint64_t* seeds, const uint8_t* mask, uint64_t* rng,
                 void* stream);
/* Debug/test helper: draw k doubles per env (Generator.random()) into out[n][k], advancing the streams. */
int b2e_rng_random(const b2e_batch* b, uint64_t* rng, int32_t k, double* out, void* stream);

/* ---- CartPole-v1: gymnasium/envs/classic_control/cartpole.py:164-247 ---------------------------------------------
 * state  : float64 [4][n]     x[n], x_dot[n], theta[n], theta_dot[n] (four coalesced 8-byte streams)
 * ctrl   : int32 [n]       bits 0..30 elapsed steps (TimeLimit), bit 31 = autoreset pending (NEXT_STEP)
 * obs    : float32 [n][4]
 */
typedef struct b2e_cartpole_cfg {
  double reset_low, reset_high; /* cartpole.py:236-241 (+ options low/high, classic_control/utils.py:17-46) */
  int32_t sutton_barto_reward;  /* cartpole.py:205-220 */
} b2e_cartpole_cfg;

/* CartPoleEnv.reset for lanes with mask!=0 (NULL = all); clears elapsed/autoreset; writes obs for those lanes. */
int b2e_cartpole_reset(const b2e_batch* b, const b2e_cartpole_cfg* cfg, const uint8_t* mask, double* state,
                       int32_t* ctrl, uint64_t* rng, float* obs, void* stream);
/* One fused step + time-limit + autoreset over the batch.
 * actions: [n] of b->action_dtype in {I64,I32,U8}; reward float64 [n]; terminated/truncated uint8 [n];
 * final_obs float32 [n][4] is written for done lanes in SAME_STEP mode only (may be NULL otherwise). */
int b2e_cartpole_step(const b2e_batch* b, const b2e_cartpole_cfg* cfg, const void* actions, double* state,
                      int32_t* ctrl, uint64_t* rng, float* obs, double* reward, uint8_t* terminated,
                      uint8_t* truncated, float* final_obs, void* stream);
/* K fused steps in one launch, state kept in registers, trajectory streamed to HBM.
 * actions: [K][n] of b->action_dtype, or NULL => uniform random actions from Philox(philox_seed, env, call_counter+k),
 *          written to actions_out uint8 [K][n] when that is non-NULL.
 * obs float32 [K][n][4]; reward float32 [K][n]; terminated/truncated uint8 [K][n]. NEXT_STEP autoreset only. */
int b2e_cartpole_rollout(const b2e_batch* b, const b2e_cartpole_cfg* cfg, int32_t K, const void* actions,
                         uint8_t* actions_out, double* state, int32_t* ctrl, uint64_t* rng, float* obs, float* reward,
                         uint8_t* terminated, uint8_t* truncated, void* stream);

/* Device self-test of the CartPole fast math paths on n pseudo-random inputs: counts uint64 [3] (device, caller-zeroed)
 * receives {const-division results != IEEE division, sin/cos more than 1 ulp from libdevice, exactly 1 ulp}. */
int b2e_selftest_math(int64_t n, uint64_t seed, uint64_t* counts, void* stream);
/* Measurement aid (bench.py): enqueues a SIMT FMA loop that fills the device (8 independent chains per thread, fp64 != 0:
 * double, else float) and reports the flops it performs in *flops; the caller times it with events.  sink: >= 8 bytes. */
int b2e_fma_probe(int fp64, int64_t iters, int64_t* flops, void* sink, void* stream);

/* ---- FrozenLake-v1: gymnasium/envs/toy_text/frozen_lake.py:232-348, toy_text/utils.py:4-8 -----------------------
 * Transition table (device, immutable, built by the host from the map exactly as frozen_lake.py:256-300):
 *   table  : uint32 [nS*nA*3]  entry = next_state | done<<16 | reward_class<<17 (0..2 -> rewards[class], 3 -> 0.0) | n_out<<20
 *            n_out is 3 for a slippery row (outcomes ordered (a-1)%4, a, (a+1)%4) or 1 (terminal tile / not slippery)
 *   cum3/p3: cumulative (numpy cumsum order) and plain probabilities of the three outcomes of a slippery row;
 *            a one-outcome row has p = 1.0
 *   isd_cum: float64 [nS] device, cumulative initial-state distribution
 * pstate : int32 [n]  current state;  ctrl as for CartPole
 * obs    : int64 [n];  prob float64 [n] (info["prob"], 1.0 on reset calls)
 */
typedef struct b2e_frozenlake_cfg {
  int32_t n_states, n_actions;
  const uint32_t* table;
  const double* isd_cum;
  double cum3[3];
  double p3[3];
  double rewards[3];
} b2e_frozenlake_cfg;

int b2e_frozenlake_reset(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, const uint8_t* mask, int32_t* pstate,
                         int32_t* ctrl, uint64_t* rng, int64_t* obs, double* prob, void* stream);
int b2e_frozenlake_step(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, const void* actions, int32_t* pstate,
                        int32_t* ctrl, uint64_t* rng, int64_t* obs, double* reward, uint8_t* terminated,
                        uint8_t* truncated, double* prob, int64_t* final_obs, double* final_prob, void* stream);
/* K fused steps; actions [K][n] or NULL (Philox random, written to actions_out when non-NULL).
 * obs uint8/int64 per obs_i64 flag: obs [K][n]; reward float32 [K][n]; flags uint8 [K][n]. */
int b2e_frozenlake_rollout(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, int32_t K, const void* actions,
                           uint8_t* actions_out, int32_t* pstate, int32_t* ctrl, uint64_t* rng, int64_t* obs,
                           float* reward, uint8_t* terminated, uint8_t* truncated, void* stream);

/* ---- Taxi-v4 `fickle_passenger=True` (gymnasium/envs/toy_text/taxi.py:436-452, :466-468): fix-up kernels launched right
 * after b2e_frozenlake_reset / b2e_frozenlake_step on the same stream (they continue the env's RNG stream).
 *   fickle : uint8 [n] fickle_step flags;  u32buf : int64 [n] as for Blackjack;  prev_state : int32 [n] copy of pstate taken
 *   before the step;  pstate / ctrl / rng / obs: the tabular kernel's buffers.  numpy-parity RNG, NEXT_STEP or DISABLED. */
int b2e_taxi_fickle_reset(const b2e_batch* b, double fickle_probability, const uint8_t* mask, uint64_t* rng, uint8_t* fickle,
                          void* stream);
int b2e_taxi_fickle_step(const b2e_batch* b, double fickle_probability, const int32_t* prev_state, int32_t* pstate,
                         const int32_t* ctrl, uint64_t* rng, int64_t* u32buf, uint8_t* fickle, int64_t* obs, void* stream);

/* ---- Blackjack-v1: gymnasium/envs/toy_text/blackjack.py:10-238 ------------------------------------------------------------
 *   hand   : int32 [n]  packed (player sum/ace/count, dealer sum/ace/count, dealer's first card), see blackjack.cu
 *   u32buf : int64 [n]  PCG64's one-word 32-bit buffer (bit 32 = valid); zero it for an env whenever its stream is
 *                       (re)seeded, as numpy does for a fresh Generator; unused in Philox mode (may be NULL)
 *   ctrl / rng as for CartPole
 * obs int64 [3][n] (player sum, dealer's first card, usable ace: the three Discrete components of the reference's Tuple
 * observation, one array each); reward float64 [n] in {-1, 0, 1, 1.5}; final_obs int64 [3][n] (SAME_STEP only).
 * actions: 0 = stick, anything else = hit (the reference asserts {0, 1}). */
typedef struct b2e_blackjack_cfg {
  int32_t natural;   /* BlackjackEnv(natural=False) */
  int32_t sab;       /* BlackjackEnv(sab=False); the registered Blackjack-v1 passes sab=True */
  int32_t* hand;
  int64_t* u32buf;
  int32_t* ctrl;
  uint64_t* rng;
} b2e_blackjack_cfg;
int b2e_blackjack_reset(const b2e_batch* b, const b2e_blackjack_cfg* cfg, const uint8_t* mask, int64_t* obs, void* stream);
int b2e_blackjack_step(const b2e_batch* b, const b2e_blackjack_cfg* cfg, const void* actions, int64_t* obs, double* reward,
                       uint8_t* terminated, uint8_t* truncated, int64_t* final_obs, void* stream);

/* ---- remaining classic-control families (gymnasium/envs/classic_control/{mountain_car,continuous_mountain_car,
 * pendulum,acrobot}.py): one generic entry point pair, `family` selects the dynamics.
 *   state float64 [k][n] (k = 2, 2, 2, 4); sflag uint8 [n] (MountainCarContinuous only); ctrl / rng as for CartPole
 *   p[4]: MountainCar(-Continuous): reset low, reset high, goal_velocity; Pendulum: x_init, y_init, g;
 *         Acrobot: reset low, reset high
 *   actions: int64/int32/uint8 [n] (MountainCar, Acrobot) or float32 [n][1] (MountainCarContinuous, Pendulum)
 *   obs float32 [n][2|2|3|6]; reward float64 [n]; flags uint8 [n]
 */
#define B2E_CLASSIC_MOUNTAINCAR 0
#define B2E_CLASSIC_MOUNTAINCAR_CONTINUOUS 1
#define B2E_CLASSIC_PENDULUM 2
#define B2E_CLASSIC_ACROBOT 3
typedef struct b2e_classic_cfg {
  int32_t family;
  int32_t _pad;
  double p[4];
  double* state;
  uint8_t* sflag;
  int32_t* ctrl;
  uint64_t* rng;
} b2e_classic_cfg;

int b2e_classic_reset(const b2e_batch* b, const b2e_classic_cfg* cfg, const uint8_t* mask, float* obs, void* stream);
int b2e_classic_step(const b2e_batch* b, const b2e_classic_cfg* cfg, const void* actions, float* obs, double* reward,
                     uint8_t* terminated, uint8_t* truncated, float* final_obs, void* stream);

/* ---- LunarLander-v3: gymnasium/envs/box2d/lunar_lander.py:321-665 (+ the Box2D 2.3.x subset world.Step needs) -------
 * Discrete actions (0 nop, 1 left, 2 main, 3 right) or continuous=1 (two throttles), optional wind.  Per-env state,
 * struct-of-arrays over n envs (device):
 *   bodies  : float32 [21][n]  for b in (lander, legs[0], legs[1]): c.x, c.y, angle, v.x, v.y, w, sleepTime
 *   joints  : float32 [8][n]   for each revolute joint: impulse.x, .y, .z, motorImpulse
 *   terrain : float32 [11][n]  smooth_y of the 11 terrain chunks
 *   fat     : float32 [12][n]  broad-phase fat AABBs of the 3 polygons (lo.x, lo.y, hi.x, hi.y)
 *   contacts: uint32  [b2e_lunarlander_state_words()][n]  most-recent-first list of contact manifolds
 *   flags   : int32   [n]      awake, game_over, leg contacts, joint limit states, contact count (see lunarlander.cu)
 *   prev_shaping: float64 [n]; ctrl / rng as for CartPole
 * obs float32 [n][8]; reward float64 [n]; terminated/truncated uint8 [n]; final_obs float32 [n][8] (SAME_STEP only).
 */
typedef struct b2e_lunarlander_cfg {
  double gravity;        /* LunarLander(gravity=-10.0) */
  int32_t enable_wind;   /* lunar_lander.py:476-506: wind force / turbulence torque while no leg touches the ground */
  int32_t continuous;    /* lunar_lander.py:509-616: actions float [n][2] = (main throttle, lateral throttle) in [-1, 1] */
  double wind_power;       /* 15.0 */
  double turbulence_power; /* 1.5 */
} b2e_lunarlander_cfg;

typedef struct b2e_lunarlander_state {
  float* bodies;
  float* joints;
  float* terrain;
  float* fat;
  uint32_t* contacts;
  int32_t* flags;
  double* prev_shaping;
  int32_t* ctrl;
  uint64_t* rng;
  int32_t* wind;   /* [2][n] wind_idx, torque_idx: offsets into the wind pattern, drawn at reset (enable_wind; else NULL) */
  int64_t* u32buf; /* [n] PCG64's one-word 32-bit buffer (bit 32 = valid) that np_random.integers leaves behind
                      (enable_wind with the numpy RNG; else NULL).  Zero it whenever the streams are re-seeded. */
} b2e_lunarlander_state;

int b2e_lunarlander_state_words(void);
/* LunarLander.reset (incl. its embedded step(0), lunar_lander.py:447) for lanes with mask != 0 (NULL = all). */
int b2e_lunarlander_reset(const b2e_batch* b, const b2e_lunarlander_cfg* cfg, const b2e_lunarlander_state* st,
                          const uint8_t* mask, float* obs, void* stream);
int b2e_lunarlander_step(const b2e_batch* b, const b2e_lunarlander_cfg* cfg, const b2e_lunarlander_state* st,
                         const void* actions, float* obs, double* reward, uint8_t* terminated, uint8_t* truncated,
                         float* final_obs, void* stream);

/* ---- Humanoid-v5: gymnasium/envs/mujoco/humanoid_v5.py:436-532, mujoco_env.py:132-155, assets/humanoid.xml ---------
 * (+ the MuJoCo subset mj_step/mj_forward/mj_rnePostConstraint need for this model; see csrc/humanoid.cu)
 * Per-env state, struct-of-arrays over n envs (device, float64):
 *   qpos [24][n], qvel [23][n], qacc_warmstart [23][n], com_xy [2][n] (mass centre of the last forward evaluation);
 *   ctrl / rng as for CartPole; overflow int32 [1] (sticky: a contact/constraint buffer was exhausted)
 * actions float32 or float64 [n][17] (b->action_dtype = B2E_ACT_F32 / B2E_ACT_F64)
 * obs float64 [n][348]; reward float64 [n]; terminated/truncated uint8 [n];
 * info float64 [13][n]: x_position, y_position, tendon_length[2], tendon_velocity[2], distance_from_origin,
 *                       x_velocity, y_velocity, reward_survive, reward_forward, reward_ctrl, reward_contact
 * final_obs float64 [n][348] (SAME_STEP only).
 */
typedef struct b2e_humanoid_cfg {
  double reset_noise_scale;      /* 1e-2 */
  double forward_reward_weight;  /* 1.25 */
  double ctrl_cost_weight;       /* 0.1 */
  double contact_cost_weight;    /* 5e-7 */
  double contact_cost_max;       /* contact_cost_range[1] = 10 */
  double healthy_reward;         /* 5.0 */
  double healthy_z_min, healthy_z_max; /* (1.0, 2.0) */
  int32_t terminate_when_unhealthy;    /* 1 */
  int32_t frame_skip;                  /* 5 */
  int32_t impl;                        /* 0 = warp per env (shared memory), 1 = thread per env; results are bit-identical */
  int32_t _pad;
} b2e_humanoid_cfg;

typedef struct b2e_humanoid_state {
  double* qpos;
  double* qvel;
  double* qacc_warmstart;
  double* com_xy;
  int32_t* ctrl;
  uint64_t* rng;
  int32_t* overflow;
  int32_t* work;   /* [n] optional (may be NULL with order): constraint-solver work of every env in its last step */
  int32_t* order;  /* [n] optional scratch: env indices sorted by `work`; the warp-per-env step kernel then puts envs of
                      similar cost into the same CTA (scheduling only: results do not depend on it) */
} b2e_humanoid_state;

/* Host-side view of the compiled model constants (no GPU needed): body_mass[14], misc[8] = {meaninertia, n collision
 * pairs, total mass, ...}, invweight[14*2 + 23] = body_invweight0 then dof_invweight0. */
int b2e_humanoid_model_info(double* body_mass, double* misc, double* invweight);
int b2e_humanoid_reset(const b2e_batch* b, const b2e_humanoid_cfg* cfg, const b2e_humanoid_state* st,
                       const uint8_t* mask, double* obs, double* info, void* stream);
int b2e_humanoid_step(const b2e_batch* b, const b2e_humanoid_cfg* cfg, const b2e_humanoid_state* st,
                      const void* actions, double* obs, double* reward, uint8_t* terminated, uint8_t* truncated,
                      double* info, double* final_obs, void* stream);

/* ---- Hopper-v5 / Walker2d-v5: gymnasium/envs/mujoco/hopper_v5.py:226-343, walker2d_v5.py:257-342, mujoco_env.py:132-155,
 * assets/hopper.xml, assets/walker2d_v5.xml (+ the MuJoCo subset of humanoid.cu generalised to slide + hinge joints; see
 * csrc/mjc_planar.cuh).  nq = nv = 6 (Hopper) / 9 (Walker2d), nu = 3 / 6.
 * Per-env state, struct-of-arrays over n envs (device, float64): qpos [nq][n], qvel [nv][n], qacc_warmstart [nv][n];
 *   ctrl / rng as for CartPole; overflow int32 [1] (sticky: a contact/constraint buffer was exhausted)
 * actions float32 or float64 [n][nu]; obs float64 [n][2 nq - 1] (qpos[1:], clip(qvel, -10, 10)); reward float64 [n];
 * info float64 [6][n]: x_position, z_distance_from_origin, x_velocity, reward_forward, reward_ctrl, reward_survive
 * final_obs float64 [n][2 nq - 1] (SAME_STEP only).
 */
typedef struct b2e_mjplanar_cfg {
  double reset_noise_scale;      /* 5e-3 */
  double forward_reward_weight;  /* 1.0 */
  double ctrl_cost_weight;       /* 1e-3 */
  double healthy_reward;         /* 1.0 */
  double healthy_z_min, healthy_z_max;         /* Hopper (0.7, inf), Walker2d (0.8, 2.0) */
  double healthy_angle_min, healthy_angle_max; /* Hopper (-0.2, 0.2), Walker2d (-1, 1) */
  double healthy_state_min, healthy_state_max; /* Hopper only: (-100, 100) */
  int32_t terminate_when_unhealthy;            /* 1 */
  int32_t frame_skip;                          /* 4 */
} b2e_mjplanar_cfg;

typedef struct b2e_mjplanar_state {
  double* qpos;
  double* qvel;
  double* qacc_warmstart;
  int32_t* ctrl;
  uint64_t* rng;
  int32_t* overflow;
} b2e_mjplanar_state;

/* Host-side view of the compiled model constants (no GPU needed): body_mass[nbody], misc[8] = {meaninertia, n collision
 * pairs, total mass, ...}, invweight[nbody*2 + nv] = body_invweight0 then dof_invweight0 (nbody = 5 / 8). */
int b2e_hopper_model_info(double* body_mass, double* misc, double* invweight);
int b2e_hopper_reset(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const uint8_t* mask,
                     double* obs, double* info, void* stream);
int b2e_hopper_step(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const void* actions,
                    double* obs, double* reward, uint8_t* terminated, uint8_t* truncated, double* info, double* final_obs,
                    void* stream);
int b2e_walker2d_model_info(double* body_mass, double* misc, double* invweight);
int b2e_walker2d_reset(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const uint8_t* mask,
                       double* obs, double* info, void* stream);
int b2e_walker2d_step(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const void* actions,
                      double* obs, double* reward, uint8_t* terminated, uint8_t* truncated, double* info, double* final_obs,
                      void* stream);
/* HalfCheetah-v5: gymnasium/envs/mujoco/half_cheetah_v5.py:220-281, assets/half_cheetah.xml on the same kernels (Euler
 * integrator with implicit joint damping, joint springs, settotalmass 14, per-actuator gears).  nq = nv = 9, nu = 6; cfg uses
 * reset_noise_scale (0.1: uniform on qpos, 0.1 * standard_normal on qvel -- numpy's ziggurat over the env's PCG64 stream),
 * forward_reward_weight (1.0), ctrl_cost_weight (0.1) and frame_skip (5).  obs float64 [n][17] = qpos[1:] | qvel;
 * never terminates; info rows 0 x_position, 2 x_velocity, 3 reward_forward, 4 reward_ctrl; nbody = 8. */
int b2e_half_cheetah_model_info(double* body_mass, double* misc, double* invweight);
int b2e_half_cheetah_reset(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const uint8_t* mask,
                           double* obs, double* info, void* stream);
int b2e_half_cheetah_step(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st, const void* actions,
                          double* obs, double* reward, uint8_t* terminated, uint8_t* truncated, double* info, double* final_obs,
                          void* stream);
/* InvertedPendulum-v5: gymnasium/envs/mujoco/inverted_pendulum_v5.py:147-186, assets/inverted_pendulum.xml on the same
 * kernels.  nq = nv = 2 (slider, hinge), nu = 1 (ctrlrange +-3, gear 100), timestep 0.02; cfg uses reset_noise_scale (0.01),
 * and frame_skip (2) only.  obs float64 [n][4] = qpos | qvel; reward 1.0 while |angle| <= 0.2 and the state is
 * finite, else 0.0 and terminated; info row 5 = reward_survive (rows 0-4 zero); nbody = 3. */
int b2e_inverted_pendulum_model_info(double* body_mass, double* misc, double* invweight);
int b2e_inverted_pendulum_reset(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st,
                                const uint8_t* mask, double* obs, double* info, void* stream);
int b2e_inverted_pendulum_step(const b2e_batch* b, const b2e_mjplanar_cfg* cfg, const b2e_mjplanar_state* st,
                               const void* actions, double* obs, double* reward, uint8_t* terminated, uint8_t* truncated,
                               double* info, double* final_obs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ENV_H_ */
