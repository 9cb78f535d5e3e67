// cartpole.cu -- fused CartPole-v1 step + TimeLimit + autoreset kernels (sm_100a).
//
// Replaces, for a batch of n envs in one launch:
//   CartPoleEnv.step   gymnasium/envs/classic_control/cartpole.py:164-226 (explicit Euler :185-189)
//   CartPoleEnv.reset  cartpole.py:228-247 (np_random.uniform(low, high, size=4))
//   TimeLimit.step     gymnasium/wrappers/common.py:116-135
//   SyncVectorEnv.step gymnasium/vector/sync_vector_env.py:266-337 (NEXT_STEP / SAME_STEP / DISABLED autoreset)
//
// Arithmetic: float64 state like the reference (cartpole.py:196), every + - * / written with the round-to-nearest
// intrinsics so ptxas can never contract a*b+c into an FMA: apart from sin/cos (CUDA libdevice vs the host libm,
// <= 1-2 ulp) the op sequence is the reference's, which keeps whole trajectories inside the 1e-5 tolerance.
//
// Memory: struct-of-arrays float64 state [4][n] (four fully coalesced 8-byte streams), one packed int32 control word,
// float4 observation store, RNG state touched only by lanes that reset.  HBM-bound: 106 B/env-step with int64 actions.
// Round 2 tried two 16-byte state streams (LDG.128) and moving the rare code (autoreset draws, libdevice sincos) out of
// line; a same-box A/B of the four combinations (profiles/r2_notes.md) put this form first on the HBM-cold ring (3.98 us
// per 65536-env launch against 4.03 / 4.04 / 4.11), so it is the only one kept.
#include "common.cuh"

namespace b2e {
namespace {

struct CartPoleArgs {
  int64_t n, env_offset;
  int32_t max_steps, mode, rng_mode, sutton;
  uint64_t philox_seed, call_counter;
  double low, range;
  double* __restrict__ state;
  int32_t* __restrict__ ctrl;
  uint64_t* __restrict__ rng;
  float* __restrict__ obs;
  double* __restrict__ reward;
  uint8_t* __restrict__ term;
  uint8_t* __restrict__ trunc;
  float* __restrict__ final_obs;
  const void* __restrict__ actions;
  const uint8_t* __restrict__ mask;
};

// constants, evaluated in double exactly as CartPoleEnv.__init__ does (cartpole.py:124-136)
constexpr double kGravity = 9.8, kMassCart = 1.0, kMassPole = 0.1, kTotalMass = kMassPole + kMassCart;
constexpr double kLength = 0.5, kPoleMassLength = kMassPole * kLength, kForceMag = 10.0, kTau = 0.02;
constexpr double kThetaThreshold = 12 * 2 * 3.141592653589793 / 360, kXThreshold = 2.4;

struct State4 {
  double x, xd, th, thd;
};

// x / total_mass, correctly rounded, without the generic division sequence: q0 = x * RN(1/d), then two
// residual-correction FMAs (Markstein).  Bit-identical to __ddiv_rn(x, kTotalMass) on every input the self-test sweeps
// (b2e_selftest_math, tests/test_gpu_parity.py); ~5 FP64 issue slots instead of ~25.
__device__ __forceinline__ double div_total_mass(double x) {
  constexpr double d = kTotalMass, r = 1.0 / kTotalMass;
  double q = __dmul_rn(x, r);
  q = __fma_rn(__fma_rn(-q, d, x), r, q);
  return __fma_rn(__fma_rn(-q, d, x), r, q);
}

// libdevice's sincos (Payne-Hanek reduction and all), returning in registers
__device__ __forceinline__ double2 sincos_cold(double x) {
  double sn, cs;
  sincos(x, &sn, &cs);
  return make_double2(sn, cs);
}

// sin/cos for |x| < 0.3 (every non-terminated CartPole angle: |theta| <= 12 deg = 0.2094): the classic fdlibm kernel
// polynomials (k_sin.c / k_cos.c coefficients), no range reduction, < 1 ulp; larger arguments (custom reset bounds,
// DISABLED-mode steps past termination) take libdevice's sincos.
__device__ __forceinline__ void sincos_pole(double x, double* sn, double* cs) {
  if (fabs(x) < 0.3) {
    constexpr double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03,
                     S3 = -1.98412698298579493134e-04, S4 = 2.75573137070700676789e-06,
                     S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
    constexpr double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03,
                     C3 = 2.48015872894767294178e-05, C4 = -2.75573143513906633035e-07,
                     C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
    const double z = __dmul_rn(x, x);
    double r = __fma_rn(z, S6, S5);
    r = __fma_rn(z, r, S4);
    r = __fma_rn(z, r, S3);
    r = __fma_rn(z, r, S2);
    *sn = __fma_rn(__dmul_rn(z, x), __fma_rn(z, r, S1), x);
    double q = __fma_rn(z, C6, C5);
    q = __fma_rn(z, q, C4);
    q = __fma_rn(z, q, C3);
    q = __fma_rn(z, q, C2);
    q = __fma_rn(z, q, C1);
    q = __dmul_rn(z, q);
    *cs = __dsub_rn(1.0, __fma_rn(-z, q, __dmul_rn(0.5, z)));
  } else {
    const double2 r = sincos_cold(x);
    *sn = r.x;
    *cs = r.y;
  }
}

// cartpole.py:169-189, literal op order (each rounding the reference makes is made here, none is fused)
__device__ __forceinline__ State4 euler_step(State4 s, int action) {
  const double force = action == 1 ? kForceMag : -kForceMag;
  double sinth, costh;
  sincos_pole(s.th, &sinth, &costh);
  const double temp =
      div_total_mass(__dadd_rn(force, __dmul_rn(__dmul_rn(kPoleMassLength, __dmul_rn(s.thd, s.thd)), sinth)));
  const double denom =
      __dmul_rn(kLength, __dsub_rn(4.0 / 3.0, div_total_mass(__dmul_rn(kMassPole, __dmul_rn(costh, costh)))));
  const double thacc = __ddiv_rn(__dsub_rn(__dmul_rn(kGravity, sinth), __dmul_rn(costh, temp)), denom);
  const double xacc = __dsub_rn(temp, div_total_mass(__dmul_rn(__dmul_rn(kPoleMassLength, thacc), costh)));
  State4 o;
  o.x = __dadd_rn(s.x, __dmul_rn(kTau, s.xd));
  o.xd = __dadd_rn(s.xd, __dmul_rn(kTau, xacc));
  o.th = __dadd_rn(s.th, __dmul_rn(kTau, s.thd));
  o.thd = __dadd_rn(s.thd, __dmul_rn(kTau, thacc));
  return o;
}

__device__ __forceinline__ bool is_terminated(const State4& s) {  // cartpole.py:198-203 (strict)
  return s.x < -kXThreshold || s.x > kXThreshold || s.th < -kThetaThreshold || s.th > kThetaThreshold;
}

__device__ __forceinline__ State4 load_state(const double* __restrict__ st, int64_t n, int64_t i) {
  return State4{st[i], st[n + i], st[2 * n + i], st[3 * n + i]};
}
__device__ __forceinline__ void store_state(double* __restrict__ st, int64_t n, int64_t i, const State4& s) {
  st[i] = s.x;
  st[n + i] = s.xd;
  st[2 * n + i] = s.th;
  st[3 * n + i] = s.thd;
}
__device__ __forceinline__ float4 to_obs(const State4& s) {
  return make_float4((float)s.x, (float)s.xd, (float)s.th, (float)s.thd);
}

// CartPoleEnv.reset: 4 uniform draws in the order x, x_dot, theta, theta_dot
template <class A>
__device__ __forceinline__ State4 sample_reset(const A& a, int64_t i, uint64_t counter) {
  State4 s;
  if (a.rng_mode == B2E_RNG_NUMPY) {
    Pcg64 g = pcg64_load(a.rng, a.n, i);
    s.x = g.uniform(a.low, a.range);
    s.xd = g.uniform(a.low, a.range);
    s.th = g.uniform(a.low, a.range);
    s.thd = g.uniform(a.low, a.range);
    pcg64_store_state(a.rng, i, g);
  } else {
    const uint64_t env = (uint64_t)(a.env_offset + i);
    const uint4 r0 = philox_block(a.philox_seed, env, counter, 1u), r1 = philox_block(a.philox_seed, env, counter, 2u);
    s.x = __dadd_rn(a.low, __dmul_rn(a.range, u53_to_double(r0.x, r0.y)));
    s.xd = __dadd_rn(a.low, __dmul_rn(a.range, u53_to_double(r0.z, r0.w)));
    s.th = __dadd_rn(a.low, __dmul_rn(a.range, u53_to_double(r1.x, r1.y)));
    s.thd = __dadd_rn(a.low, __dmul_rn(a.range, u53_to_double(r1.z, r1.w)));
  }
  return s;
}

__global__ void __launch_bounds__(kBlock) cartpole_reset_kernel(const CartPoleArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  const State4 s = sample_reset(a, i, a.call_counter);
  store_state(a.state, a.n, i, s);
  a.ctrl[i] = 0;
  reinterpret_cast<float4*>(a.obs)[i] = to_obs(s);
}

// The autoreset path of the step kernel: CartPoleEnv.reset for one env -- draws, state, cleared control word,
// observation.  The PCG64 words are loaded here, by the resetting lanes only.
__device__ __forceinline__ void reset_env_cold(double* __restrict__ state, int32_t* __restrict__ ctrl, uint64_t* __restrict__ rng,
                                               float* __restrict__ obs, int64_t n, int64_t i, double low, double range,
                                               int32_t rng_mode, uint64_t philox_seed, uint64_t env, uint64_t counter) {
  State4 s;
  if (rng_mode == B2E_RNG_NUMPY) {
    Pcg64 g = pcg64_load(rng, n, i);
    s.x = g.uniform(low, range);  // cartpole.py:236-241: x, x_dot, theta, theta_dot in this order
    s.xd = g.uniform(low, range);
    s.th = g.uniform(low, range);
    s.thd = g.uniform(low, range);
    pcg64_store_state(rng, i, g);
  } else {
    const uint4 r0 = philox_block(philox_seed, env, counter, 1u), r1 = philox_block(philox_seed, env, counter, 2u);
    s.x = __dadd_rn(low, __dmul_rn(range, u53_to_double(r0.x, r0.y)));
    s.xd = __dadd_rn(low, __dmul_rn(range, u53_to_double(r0.z, r0.w)));
    s.th = __dadd_rn(low, __dmul_rn(range, u53_to_double(r1.x, r1.y)));
    s.thd = __dadd_rn(low, __dmul_rn(range, u53_to_double(r1.z, r1.w)));
  }
  store_state(state, n, i, s);
  ctrl[i] = 0;
  __stcs(reinterpret_cast<float4*>(obs) + i, to_obs(s));
}

// One thread per env.  State, control word and action are issued before the first use (one memory round trip); the
// PCG64 words are read only by the lanes that reset.  Loading them up front for every lane was measured on a B200 at
// N=65536 (profiles/r2_notes.md): 3.03 vs 3.13 us per launch while the batch is L2-resident, but 3.84 vs 3.66 us on the
// HBM-cold ring, where the +30 % DRAM reads outweigh the saved round trip.
// Launch geometry was swept on a B200 at N=65536 (graph-chained launches, us per launch, L2-resident / HBM-cold ring):
// CTA 64: 3.01 / 3.91, 128: 3.21 / 4.05, 256: 3.33 / 4.08, 448 (one CTA per SM): 3.28 / 4.01, 1024: 4.65 / 5.29; 2 or 4
// envs per thread were slower (4.10 / 6.3 us L2-resident); programmatic dependent launch made N >= 65536 slower (4.07 vs
// 3.27 us).
constexpr int kStepBlock = 64;

template <typename ActT>
__global__ void __launch_bounds__(1024) cartpole_step_kernel(const CartPoleArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  const int32_t c = a.ctrl[i];
  const State4 s0 = load_state(a.state, a.n, i);
  const int action = load_action<ActT>(a.actions, i);
  if (a.mode == B2E_AUTORESET_NEXT_STEP && ctrl_pending(c)) {
    // sync_vector_env.py:279-284: the call after a done is the reset; reward 0, flags False, action ignored
    reset_env_cold(a.state, a.ctrl, a.rng, a.obs, a.n, i, a.low, a.range, a.rng_mode, a.philox_seed,
                   (uint64_t)(a.env_offset + i), a.call_counter);
    __stcs(a.reward + i, 0.0);
    a.term[i] = 0;
    a.trunc[i] = 0;
    return;
  }
  const State4 s = euler_step(s0, action);
  const bool term = is_terminated(s);
  const int32_t elapsed = ctrl_elapsed(c) + 1;
  const bool trunc = a.max_steps > 0 && elapsed >= a.max_steps;  // wrappers/common.py:130-133
  // cartpole.py:205-220: 1.0 also on the terminating step, 0.0 on steps taken after it without a reset (only reachable with
  // autoreset DISABLED, where bit 31 of the control word stands for `steps_beyond_terminated is not None`)
  const bool beyond = a.mode == B2E_AUTORESET_DISABLED && ctrl_pending(c);
  __stcs(a.reward + i, a.sutton ? (term ? -1.0 : 0.0) : (term && beyond ? 0.0 : 1.0));
  a.term[i] = term;
  a.trunc[i] = trunc;
  int32_t cn = elapsed;
  if (term || trunc) {
    if (a.mode == B2E_AUTORESET_NEXT_STEP) {
      cn |= kPending;
    } else if (a.mode == B2E_AUTORESET_SAME_STEP) {  // sync_vector_env.py:302-319
      reinterpret_cast<float4*>(a.final_obs)[i] = to_obs(s);
      reset_env_cold(a.state, a.ctrl, a.rng, a.obs, a.n, i, a.low, a.range, a.rng_mode, a.philox_seed,
                     (uint64_t)(a.env_offset + i), a.call_counter);
      return;
    }
  }
  if (a.mode == B2E_AUTORESET_DISABLED && (term || beyond)) cn |= kPending;
  store_state(a.state, a.n, i, s);
  a.ctrl[i] = cn;
  __stcs(reinterpret_cast<float4*>(a.obs) + i, to_obs(s));
}

template <typename ActT>
cudaError_t launch_step(const CartPoleArgs& a, cudaStream_t st) {
  cartpole_step_kernel<ActT><<<grid_for(a.n, kStepBlock), kStepBlock, 0, st>>>(a);
  return cudaGetLastError();
}

struct RolloutArgs {
  CartPoleArgs a;
  int32_t K;
  uint8_t* __restrict__ actions_out;
  float* __restrict__ reward32;
};

// K fused steps: state in registers, [K][n] trajectory streamed out with coalesced stores.
template <typename ActT, bool kRandom>
__global__ void __launch_bounds__(kBlock) cartpole_rollout_kernel(const RolloutArgs r) {
  const CartPoleArgs& a = r.a;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  int32_t c = a.ctrl[i];
  State4 s = load_state(a.state, a.n, i);
  const uint64_t env = (uint64_t)(a.env_offset + i);
  uint4 bits = make_uint4(0, 0, 0, 0);
  uint64_t bits_block = ~0ull;
  for (int k = 0; k < r.K; ++k) {
    const int64_t o = (int64_t)k * a.n + i;
    const uint64_t counter = a.call_counter + (uint64_t)k;
    int action = 0;
    if (kRandom) {  // 128 one-bit actions per Philox block
      if ((counter >> 7) != bits_block) {
        bits_block = counter >> 7;
        bits = philox_block(a.philox_seed, env, bits_block, 3u);
      }
      const uint32_t j = (uint32_t)(counter & 127u);
      const uint32_t w = j < 32 ? bits.x : j < 64 ? bits.y : j < 96 ? bits.z : bits.w;
      action = (w >> (j & 31u)) & 1u;
      if (r.actions_out) r.actions_out[o] = (uint8_t)action;
    } else {
      action = load_action<ActT>(a.actions, o);
    }
    float rew;
    bool term = false, trunc = false;
    if (ctrl_pending(c)) {
      s = sample_reset(a, i, counter);
      c = 0;
      rew = 0.f;
    } else {
      s = euler_step(s, action);
      term = is_terminated(s);
      const int32_t elapsed = ctrl_elapsed(c) + 1;
      trunc = a.max_steps > 0 && elapsed >= a.max_steps;
      rew = a.sutton ? (term ? -1.f : 0.f) : 1.f;
      c = elapsed | ((term || trunc) ? kPending : 0);
    }
    __stcs(reinterpret_cast<float4*>(a.obs) + o, to_obs(s));
    __stcs(r.reward32 + o, rew);
    a.term[o] = term;
    a.trunc[o] = trunc;
  }
  store_state(a.state, a.n, i, s);
  a.ctrl[i] = c;
}

// self-test of the two fast paths against the generic device routines on pseudo-random inputs in the ranges the
// CartPole step feeds them: counts[0] = div_total_mass != __ddiv_rn, counts[1] = |sin| or |cos| off by > 1 ulp
__global__ void __launch_bounds__(kBlock) cartpole_selftest_kernel(int64_t n, uint64_t seed, unsigned long long* counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint4 r = philox_block(seed, (uint64_t)i, 0, 7u), r2 = philox_block(seed, (uint64_t)i, 1, 7u);
  // numerators: mantissa uniform, exponent uniform over 2^-40 .. 2^8, both signs
  const double mant = 1.0 + u53_to_double(r.x, r.y);
  const double x = ldexp(mant, (int)(r.z % 49u) - 40) * ((r.w & 1u) ? -1.0 : 1.0);
  if (div_total_mass(x) != __ddiv_rn(x, kTotalMass)) atomicAdd(counts + 0, 1ull);
  const double th = (u53_to_double(r2.x, r2.y) * 2.0 - 1.0) * 0.2999;
  double s0, c0, s1, c1;
  sincos_pole(th, &s0, &c0);
  sincos(th, &s1, &c1);
  const long long ds = llabs(__double_as_longlong(s0) - __double_as_longlong(s1));
  const long long dc = llabs(__double_as_longlong(c0) - __double_as_longlong(c1));
  if (ds > 1 || dc > 1) atomicAdd(counts + 1, 1ull);
  if (ds == 1 || dc == 1) atomicAdd(counts + 2, 1ull);
}

CartPoleArgs make_args(const b2e_batch* b, const b2e_cartpole_cfg* cfg) {
  CartPoleArgs a{};
  a.n = b->n;
  a.env_offset = b->env_offset;
  a.max_steps = b->max_episode_steps;
  a.mode = b->autoreset_mode;
  a.rng_mode = b->rng_mode;
  a.sutton = cfg->sutton_barto_reward;
  a.philox_seed = b->philox_seed;
  a.call_counter = b->call_counter;
  a.low = cfg->reset_low;
  a.range = cfg->reset_high - cfg->reset_low;  // Generator.uniform computes high - low once in double
  return a;
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int b2e_selftest_math(int64_t n, uint64_t seed, uint64_t* counts, void* stream) {
  if (n < 0 || !counts) {
    set_error("b2e_selftest_math: bad arguments");
    return B2E_EINVAL;
  }
  if (n == 0) return 0;
  cartpole_selftest_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(n, seed,
                                                                            (unsigned long long*)counts);
  return cuda_status(cudaGetLastError(), "b2e_selftest_math");
}

extern "C" int b2e_cartpole_reset(const b2e_batch* b, const b2e_cartpole_cfg* cfg, const uint8_t* mask, double* state,
                                  int32_t* ctrl, uint64_t* rng, float* obs, void* stream) {
  if (int e = check_batch(b, "b2e_cartpole_reset")) return e;
  if (!cfg || !state || !ctrl || !obs || (b->rng_mode == B2E_RNG_NUMPY && !rng)) {
    set_error("b2e_cartpole_reset: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  CartPoleArgs a = make_args(b, cfg);
  a.mask = mask;
  a.state = state;
  a.ctrl = ctrl;
  a.rng = rng;
  a.obs = obs;
  cartpole_reset_kernel<<<grid_for(b->n), kBlock, 0, (cudaStream_t)stream>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_cartpole_reset");
}

extern "C" int b2e_cartpole_step(const b2e_batch* b, const b2e_cartpole_cfg* cfg, const void* actions, double* state,
                                 int32_t* ctrl, uint64_t* rng, float* obs, double* reward, uint8_t* terminated,
                                 uint8_t* truncated, float* final_obs, void* stream) {
  if (int e = check_batch(b, "b2e_cartpole_step")) return e;
  if (!cfg || !actions || !state || !ctrl || !obs || !reward || !terminated || !truncated ||
      (b->rng_mode == B2E_RNG_NUMPY && !rng) || (b->autoreset_mode == B2E_AUTORESET_SAME_STEP && !final_obs)) {
    set_error("b2e_cartpole_step: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  CartPoleArgs a = make_args(b, cfg);
  a.actions = actions;
  a.state = state;
  a.ctrl = ctrl;
  a.rng = rng;
  a.obs = obs;
  a.reward = reward;
  a.term = terminated;
  a.trunc = truncated;
  a.final_obs = final_obs;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e;
  switch (b->action_dtype) {
    case B2E_ACT_I64: e = launch_step<int64_t>(a, st); break;
    case B2E_ACT_I32: e = launch_step<int32_t>(a, st); break;
    case B2E_ACT_U8: e = launch_step<uint8_t>(a, st); break;
    default: set_error("b2e_cartpole_step: action_dtype %d is not a discrete dtype", b->action_dtype); return B2E_EINVAL;
  }
  return cuda_status(e, "b2e_cartpole_step");
}

extern "C" int b2e_cartpole_rollout(const b2e_batch* b, const b2e_cartpole_cfg* cfg, int32_t K, const void* actions,
                                    uint8_t* actions_out, double* state, int32_t* ctrl, uint64_t* rng, float* obs,
                                    float* reward, uint8_t* terminated, uint8_t* truncated, void* stream) {
  if (int e = check_batch(b, "b2e_cartpole_rollout")) return e;
  if (!cfg || K < 0 || !state || !ctrl || !obs || !reward || !terminated || !truncated ||
      (b->rng_mode == B2E_RNG_NUMPY && !rng)) {
    set_error("b2e_cartpole_rollout: null pointer or K < 0");
    return B2E_EINVAL;
  }
  if (b->autoreset_mode != B2E_AUTORESET_NEXT_STEP) {
    set_error("b2e_cartpole_rollout: only NEXT_STEP autoreset is supported");
    return B2E_EINVAL;
  }
  if (b->n == 0 || K == 0) return 0;
  RolloutArgs r{};
  r.a = make_args(b, cfg);
  r.a.actions = actions;
  r.a.state = state;
  r.a.ctrl = ctrl;
  r.a.rng = rng;
  r.a.obs = obs;
  r.a.term = terminated;
  r.a.trunc = truncated;
  r.K = K;
  r.actions_out = actions_out;
  r.reward32 = reward;
  const unsigned grid = grid_for(b->n);
  cudaStream_t st = (cudaStream_t)stream;
  if (!actions) {
    cartpole_rollout_kernel<uint8_t, true><<<grid, kBlock, 0, st>>>(r);
  } else {
    switch (b->action_dtype) {
      case B2E_ACT_I64: cartpole_rollout_kernel<int64_t, false><<<grid, kBlock, 0, st>>>(r); break;
      case B2E_ACT_I32: cartpole_rollout_kernel<int32_t, false><<<grid, kBlock, 0, st>>>(r); break;
      case B2E_ACT_U8: cartpole_rollout_kernel<uint8_t, false><<<grid, kBlock, 0, st>>>(r); break;
      default: set_error("b2e_cartpole_rollout: bad action_dtype %d", b->action_dtype); return B2E_EINVAL;
    }
  }
  return cuda_status(cudaGetLastError(), "b2e_cartpole_rollout");
}
