// frozenlake.cu -- fused FrozenLake-v1 (tabular MDP) step + TimeLimit + autoreset kernels (sm_100a).
//
// Replaces, for a batch of n envs in one launch:
//   FrozenLakeEnv.step    gymnasium/envs/toy_text/frozen_lake.py:324-334
//   categorical_sample    gymnasium/envs/toy_text/utils.py:4-8  (argmax(cumsum(p) > np_random.random()))
//   FrozenLakeEnv.reset   frozen_lake.py:336-348
//   TimeLimit / SyncVectorEnv autoreset as in cartpole.cu
// The transition table P[s][a] (frozen_lake.py:256-300) is built by the host and staged into shared memory once per
// CTA (grid-stride CTAs, so the staging cost is amortised): 3 outcomes per (s,a) packed to 4 bytes each.  Integer state
// is bit-exact with the reference because the float64 draw u and the float64 cumulative sums are the reference's own.
//
// Memory: HBM-bound integer work, 1 thread/env.  Per env-step (numpy-parity RNG, int64 actions): PCG64 state 16 r + 16 w,
// inc 16 r, state 4 r/w, ctrl 4 r/w, action 8, obs 8, reward 8, flags 2, prob 8 = 98 B.
#include "common.cuh"

namespace b2e {
namespace {

constexpr int kMaxSharedEntries = 12288;  // (s,a,outcome) entries staged in shared memory (48 KB): up to 1024 states

struct LakeArgs {
  int64_t n, env_offset;
  int32_t max_steps, mode, rng_mode, n_states, n_actions, K;
  uint64_t philox_seed, call_counter;
  double rewards[3], cum3[3], p3[3];
  const uint32_t* __restrict__ table;
  const double* __restrict__ isd_cum;
  int32_t* __restrict__ pstate;
  int32_t* __restrict__ ctrl;
  uint64_t* __restrict__ rng;
  int64_t* __restrict__ obs;
  double* __restrict__ reward;
  float* __restrict__ reward32;
  uint8_t* __restrict__ term;
  uint8_t* __restrict__ trunc;
  double* __restrict__ prob_out;
  int64_t* __restrict__ final_obs;
  double* __restrict__ final_prob;
  const void* __restrict__ actions;
  uint8_t* __restrict__ actions_out;
  const uint8_t* __restrict__ mask;
};

// categorical_sample over the initial-state distribution: first index with cumsum > u, argmax-of-all-False = 0
__device__ __forceinline__ int sample_initial_state(const LakeArgs& a, double u) {
  // the cumulative sums are non-decreasing, so the first index with cum > u is an upper bound search
  int lo = 0, hi = a.n_states;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a.isd_cum + mid) > u) hi = mid; else lo = mid + 1;
  }
  return lo < a.n_states ? lo : 0;
}

// stage the packed table into (dynamic) shared memory; returns the pointer the CTA should read entries from
__device__ __forceinline__ const uint32_t* stage_table(const LakeArgs& a) {
  extern __shared__ uint32_t sh_entry[];
  const int total = a.n_states * a.n_actions * 3;
  if (total > kMaxSharedEntries) return a.table;  // huge maps: read through L1/L2 instead
  for (int j = threadIdx.x; j < total; j += blockDim.x) sh_entry[j] = __ldg(a.table + j);
  __syncthreads();
  return sh_entry;
}

struct StepOut {
  int s;
  double reward, p;
  bool done;
};

// frozen_lake.py:325-328 with toy_text/utils.py:4-8
__device__ __forceinline__ StepOut transition(const LakeArgs& a, const uint32_t* t, int s, int action, double u) {
  const int base = (s * a.n_actions + action) * 3;
  const int n_out = (int)(t[base] >> 20);
  int j = 0;  // argmax(cs > u): first True, or 0 when none is
  double p = 1.0;
  if (n_out == 3) {
    j = a.cum3[0] > u ? 0 : a.cum3[1] > u ? 1 : a.cum3[2] > u ? 2 : 0;
    p = j == 0 ? a.p3[0] : j == 1 ? a.p3[1] : a.p3[2];
  }
  const uint32_t e = t[base + j];
  StepOut o;
  o.s = (int)(e & 0xffffu);
  o.done = (e >> 16) & 1u;
  const uint32_t rc = (e >> 17) & 3u;
  o.reward = rc == 0 ? a.rewards[0] : rc == 1 ? a.rewards[1] : rc == 2 ? a.rewards[2] : 0.0;  // 3: literal 0 (:291)
  o.p = p;
  return o;
}

__device__ __forceinline__ double philox_u(const LakeArgs& a, int64_t i, uint64_t counter, uint32_t stream) {
  const uint4 r = philox_block(a.philox_seed, (uint64_t)(a.env_offset + i), counter, stream);
  return u53_to_double(r.x, r.y);
}

__global__ void __launch_bounds__(kBlock) frozenlake_reset_kernel(const LakeArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (a.mask != nullptr && a.mask[i] == 0) return;
  double u;
  if (a.rng_mode == B2E_RNG_NUMPY) {
    Pcg64 g = pcg64_load(a.rng, a.n, i);
    u = g.next_double();
    pcg64_store_state(a.rng, i, g);
  } else {
    u = philox_u(a, i, a.call_counter, 1u);
  }
  const int s = sample_initial_state(a, u);
  a.pstate[i] = s;
  a.ctrl[i] = 0;
  a.obs[i] = s;
  a.prob_out[i] = 1.0;
}

template <typename ActT>
__global__ void __launch_bounds__(kBlock) frozenlake_step_kernel(const LakeArgs a) {
  const uint32_t* t = stage_table(a);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    // all loads first (one DRAM round trip), then the arithmetic
    const int32_t c = a.ctrl[i];
    const int s_cur = a.pstate[i];
    int action = load_action<ActT>(a.actions, i);
    Pcg64 g;
    if (a.rng_mode == B2E_RNG_NUMPY) g = pcg64_load(a.rng, a.n, i);
    // exactly one draw per call on every path (step: frozen_lake.py:326, reset: :343)
    const double u = a.rng_mode == B2E_RNG_NUMPY ? g.next_double() : philox_u(a, i, a.call_counter, 1u);
    if (a.mode == B2E_AUTORESET_NEXT_STEP && ctrl_pending(c)) {
      const int s = sample_initial_state(a, u);
      if (a.rng_mode == B2E_RNG_NUMPY) pcg64_store_state(a.rng, i, g);
      a.pstate[i] = s;
      a.ctrl[i] = 0;
      __stcs(a.obs + i, (int64_t)s);
      __stcs(a.reward + i, 0.0);
      a.term[i] = 0;
      a.trunc[i] = 0;
      __stcs(a.prob_out + i, 1.0);
      continue;
    }
    action = min(max(action, 0), a.n_actions - 1);  // the reference would KeyError; clamp, never read out of bounds
    StepOut o = transition(a, t, s_cur, action, u);
    const int32_t elapsed = ctrl_elapsed(c) + 1;
    const bool trunc = a.max_steps > 0 && elapsed >= a.max_steps;
    __stcs(a.reward + i, o.reward);
    a.term[i] = o.done;
    a.trunc[i] = trunc;
    int32_t cn = elapsed;
    if (o.done || trunc) {
      if (a.mode == B2E_AUTORESET_NEXT_STEP) {
        cn |= kPending;
      } else if (a.mode == B2E_AUTORESET_SAME_STEP) {  // sync_vector_env.py:302-319
        a.final_obs[i] = o.s;
        a.final_prob[i] = o.p;
        const double u2 = a.rng_mode == B2E_RNG_NUMPY ? g.next_double() : philox_u(a, i, a.call_counter, 2u);
        o.s = sample_initial_state(a, u2);
        o.p = 1.0;
        cn = 0;
      }
    }
    if (a.rng_mode == B2E_RNG_NUMPY) pcg64_store_state(a.rng, i, g);
    a.pstate[i] = o.s;
    a.ctrl[i] = cn;
    __stcs(a.obs + i, (int64_t)o.s);
    __stcs(a.prob_out + i, o.p);
  }
}

// K fused steps, state + RNG in registers, [K][n] trajectory streamed out
template <typename ActT, bool kRandom>
__global__ void __launch_bounds__(kBlock) frozenlake_rollout_kernel(const LakeArgs a) {
  const uint32_t* t = stage_table(a);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    int32_t c = a.ctrl[i];
    int s = a.pstate[i];
    Pcg64 g;
    if (a.rng_mode == B2E_RNG_NUMPY) g = pcg64_load(a.rng, a.n, i);
    const uint64_t env = (uint64_t)(a.env_offset + i);
    for (int k = 0; k < a.K; ++k) {
      const int64_t o = (int64_t)k * a.n + i;
      const uint64_t counter = a.call_counter + (uint64_t)k;
      double u;
      uint32_t spare = 0;
      if (a.rng_mode == B2E_RNG_NUMPY) {
        u = g.next_double();
        if (kRandom) spare = philox_block(a.philox_seed, env, counter, 3u).x;
      } else {
        const uint4 r = philox_block(a.philox_seed, env, counter, 1u);
        u = u53_to_double(r.x, r.y);
        spare = r.z;
      }
      int action;
      if (kRandom) {
        action = (int)(((uint64_t)spare * (uint32_t)a.n_actions) >> 32);  // floor(u32 * nA / 2^32)
        if (a.actions_out) a.actions_out[o] = (uint8_t)action;
      } else {
        action = min(max(load_action<ActT>(a.actions, o), 0), a.n_actions - 1);
      }
      float rew = 0.f;
      bool term = false, trunc = false;
      if (ctrl_pending(c)) {
        s = sample_initial_state(a, u);
        c = 0;
      } else {
        const StepOut so = transition(a, t, s, action, u);
        s = so.s;
        term = so.done;
        rew = (float)so.reward;
        const int32_t elapsed = ctrl_elapsed(c) + 1;
        trunc = a.max_steps > 0 && elapsed >= a.max_steps;
        c = elapsed | ((term || trunc) ? kPending : 0);
      }
      __stcs(a.obs + o, (int64_t)s);
      __stcs(a.reward32 + o, rew);
      a.term[o] = term;
      a.trunc[o] = trunc;
    }
    if (a.rng_mode == B2E_RNG_NUMPY) pcg64_store_state(a.rng, i, g);
    a.pstate[i] = s;
    a.ctrl[i] = c;
  }
}

size_t table_smem_bytes(const LakeArgs& a) {
  const int total = a.n_states * a.n_actions * 3;
  return total <= kMaxSharedEntries ? (size_t)total * sizeof(uint32_t) : 0;
}

// Launch geometry: one env per thread (grid = ceil(n / 256)) by default.  A capped grid-stride launch (8 CTAs per SM,
// table staged once per CTA) was measured slower at N = 1,048,576 because 1M / 303k threads = 3.46 passes leaves the
// last pass half empty; staging 3 KB per CTA from L2 is cheap.
unsigned persistent_grid(int64_t n, size_t table_bytes) {
  // small tables (FrozenLake 8x8: 3 KB): one env per thread; big tables (Taxi: 36 KB) amortise the staging over a
  // grid-stride loop -- measured at N = 8M: Taxi 581 us plain grid (staging 140 B/env of extra L2 traffic)
  if (table_bytes <= 8192) return grid_for(n);
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  const int64_t want = (n + kBlock - 1) / kBlock;
  const int64_t cap = (int64_t)sms * 8;
  return (unsigned)(want < cap ? want : cap);
}

int fill_args(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, LakeArgs& a, const char* fn) {
  if (int e = check_batch(b, fn)) return e;
  if (!cfg || !cfg->table || !cfg->isd_cum || cfg->n_states <= 0 || cfg->n_states > 65536 || cfg->n_actions <= 0) {
    set_error("%s: bad table configuration", fn);
    return B2E_EINVAL;
  }
  a = LakeArgs{};
  a.n = b->n;
  a.env_offset = b->env_offset;
  a.max_steps = b->max_episode_steps;
  a.mode = b->autoreset_mode;
  a.rng_mode = b->rng_mode;
  a.n_states = cfg->n_states;
  a.n_actions = cfg->n_actions;
  a.philox_seed = b->philox_seed;
  a.call_counter = b->call_counter;
  for (int k = 0; k < 3; ++k) {
    a.rewards[k] = cfg->rewards[k];
    a.cum3[k] = cfg->cum3[k];
    a.p3[k] = cfg->p3[k];
  }
  a.table = cfg->table;
  a.isd_cum = cfg->isd_cum;
  return 0;
}

template <typename K>
int launch_by_dtype(int dtype, const char* fn, K&& launch) {
  switch (dtype) {
    case B2E_ACT_I64: launch((int64_t)0); return 0;
    case B2E_ACT_I32: launch((int32_t)0); return 0;
    case B2E_ACT_U8: launch((uint8_t)0); return 0;
    default: set_error("%s: action_dtype %d is not a discrete dtype", fn, dtype); return B2E_EINVAL;
  }
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int b2e_frozenlake_reset(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, const uint8_t* mask,
                                    int32_t* pstate, int32_t* ctrl, uint64_t* rng, int64_t* obs, double* prob,
                                    void* stream) {
  LakeArgs a;
  if (int e = fill_args(b, cfg, a, "b2e_frozenlake_reset")) return e;
  if (!pstate || !ctrl || !obs || !prob || (b->rng_mode == B2E_RNG_NUMPY && !rng)) {
    set_error("b2e_frozenlake_reset: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.mask = mask;
  a.pstate = pstate;
  a.ctrl = ctrl;
  a.rng = rng;
  a.obs = obs;
  a.prob_out = prob;
  frozenlake_reset_kernel<<<grid_for(b->n), kBlock, 0, (cudaStream_t)stream>>>(a);
  return cuda_status(cudaGetLastError(), "b2e_frozenlake_reset");
}

extern "C" int b2e_frozenlake_step(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, const void* actions,
                                   int32_t* pstate, int32_t* ctrl, uint64_t* rng, int64_t* obs, double* reward,
                                   uint8_t* terminated, uint8_t* truncated, double* prob, int64_t* final_obs,
                                   double* final_prob, void* stream) {
  LakeArgs a;
  if (int e = fill_args(b, cfg, a, "b2e_frozenlake_step")) return e;
  if (!actions || !pstate || !ctrl || !obs || !reward || !terminated || !truncated || !prob ||
      (b->rng_mode == B2E_RNG_NUMPY && !rng) ||
      (b->autoreset_mode == B2E_AUTORESET_SAME_STEP && (!final_obs || !final_prob))) {
    set_error("b2e_frozenlake_step: null pointer");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  a.actions = actions;
  a.pstate = pstate;
  a.ctrl = ctrl;
  a.rng = rng;
  a.obs = obs;
  a.reward = reward;
  a.term = terminated;
  a.trunc = truncated;
  a.prob_out = prob;
  a.final_obs = final_obs;
  a.final_prob = final_prob;
  const size_t smem = table_smem_bytes(a);
  const unsigned grid = persistent_grid(b->n, smem);
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = launch_by_dtype(b->action_dtype, "b2e_frozenlake_step", [&](auto tag) {
        frozenlake_step_kernel<decltype(tag)><<<grid, kBlock, smem, st>>>(a);
      }))
    return e;
  return cuda_status(cudaGetLastError(), "b2e_frozenlake_step");
}

extern "C" int b2e_frozenlake_rollout(const b2e_batch* b, const b2e_frozenlake_cfg* cfg, int32_t K,
                                      const void* actions, uint8_t* actions_out, int32_t* pstate, int32_t* ctrl,
                                      uint64_t* rng, int64_t* obs, float* reward, uint8_t* terminated,
                                      uint8_t* truncated, void* stream) {
  LakeArgs a;
  if (int e = fill_args(b, cfg, a, "b2e_frozenlake_rollout")) return e;
  if (K < 0 || !pstate || !ctrl || !obs || !reward || !terminated || !truncated ||
      (b->rng_mode == B2E_RNG_NUMPY && !rng)) {
    set_error("b2e_frozenlake_rollout: null pointer or K < 0");
    return B2E_EINVAL;
  }
  if (b->autoreset_mode != B2E_AUTORESET_NEXT_STEP) {
    set_error("b2e_frozenlake_rollout: only NEXT_STEP autoreset is supported");
    return B2E_EINVAL;
  }
  if (b->n == 0 || K == 0) return 0;
  a.K = K;
  a.actions = actions;
  a.actions_out = actions_out;
  a.pstate = pstate;
  a.ctrl = ctrl;
  a.rng = rng;
  a.obs = obs;
  a.reward32 = reward;
  a.term = terminated;
  a.trunc = truncated;
  const size_t smem = table_smem_bytes(a);
  const unsigned grid = persistent_grid(b->n, smem);
  cudaStream_t st = (cudaStream_t)stream;
  if (!actions) {
    frozenlake_rollout_kernel<uint8_t, true><<<grid, kBlock, smem, st>>>(a);
  } else if (int e = launch_by_dtype(b->action_dtype, "b2e_frozenlake_rollout", [&](auto tag) {
               frozenlake_rollout_kernel<decltype(tag), false><<<grid, kBlock, smem, st>>>(a);
             })) {
    return e;
  }
  return cuda_status(cudaGetLastError(), "b2e_frozenlake_rollout");
}
