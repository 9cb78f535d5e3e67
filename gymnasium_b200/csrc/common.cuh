// common.cuh -- shared device helpers for libb200env.so (sm_100a only).
//
//  * numpy-parity RNG: SeedSequence -> PCG64 (XSL-RR 128/64) -> Generator.random()/uniform(); the reference reaches it
//    through gymnasium/utils/seeding.py:39-41.  Bit-exact with numpy (tests/test_gpu_rng.py).
//  * Philox4x32-10 counter-based RNG for the stateless fast mode (the same generator cuRAND's
//    curandStatePhilox4_32_10_t implements; hand-written here so no per-env cuRAND state has to live in HBM).
//  * batch descriptor, control-word packing, error plumbing.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/b200env.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb200env targets sm_100a (B200) only"
#endif

namespace b2e {

// ---------------------------------------------------------------------------------------------------------------
// host-side error plumbing (api.cu owns the storage)
void set_error(const char* fmt, ...);
int check_batch(const b2e_batch* b, const char* fn);
int cuda_status(cudaError_t e, const char* fn);

constexpr int kBlock = 256;  // 8 warps; every kernel here is 1 thread/env (or grid-stride), register-light
inline unsigned grid_for(int64_t n, int block = kBlock) { return (unsigned)((n + block - 1) / block); }

// ---------------------------------------------------------------------------------------------------------------
// Scheduling helper shared by the physics families: order[] = env indices bucket-sorted by a small integer key
// (bucket 0 first).  Called by all threads of ONE CTA.  The order inside a bucket is arbitrary, which is fine: which envs
// share a warp / CTA changes how much they wait for each other, never what an env computes.
template <int NBUCKET, typename KeyFn>
__device__ __forceinline__ void group_envs_by_key(KeyFn key, int32_t* __restrict__ order, int64_t n) {
  __shared__ int hist[NBUCKET], cursor[NBUCKET];
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int k = tid; k < NBUCKET; k += nt) hist[k] = 0;
  __syncthreads();
  for (int64_t i = tid; i < n; i += nt) atomicAdd(&hist[key(i)], 1);
  __syncthreads();
  if (tid == 0) {
    int acc = 0;
    for (int k = 0; k < NBUCKET; ++k) { cursor[k] = acc; acc += hist[k]; }
  }
  __syncthreads();
  for (int64_t i = tid; i < n; i += nt) order[atomicAdd(&cursor[key(i)], 1)] = (int32_t)i;
}

// ---------------------------------------------------------------------------------------------------------------
// control word: bits 0..30 = TimeLimit elapsed steps, bit 31 = autoreset pending (NEXT_STEP)
constexpr int32_t kPending = (int32_t)0x80000000u;
__device__ __forceinline__ bool ctrl_pending(int32_t c) { return c < 0; }
__device__ __forceinline__ int32_t ctrl_elapsed(int32_t c) { return c & 0x7fffffff; }

// ---------------------------------------------------------------------------------------------------------------
// 128-bit helpers
struct u128 {
  uint64_t lo, hi;
};
__device__ __forceinline__ u128 mul128(u128 a, u128 b) {
  u128 r;
  r.lo = a.lo * b.lo;
  r.hi = __umul64hi(a.lo, b.lo) + a.lo * b.hi + a.hi * b.lo;
  return r;
}
__device__ __forceinline__ u128 add128(u128 a, u128 b) {
  u128 r;
  r.lo = a.lo + b.lo;
  r.hi = a.hi + b.hi + (r.lo < a.lo ? 1ull : 0ull);
  return r;
}

// ---------------------------------------------------------------------------------------------------------------
// numpy PCG64
struct Pcg64 {
  u128 state, inc;
  static constexpr uint64_t kMulHi = 0x2360ED051FC65DA4ull, kMulLo = 0x4385DF649FCCF645ull;

  __device__ __forceinline__ void advance() { state = add128(mul128(state, u128{kMulLo, kMulHi}), inc); }
  __device__ __forceinline__ uint64_t next_u64() {
    advance();
    uint64_t x = state.hi ^ state.lo;
    unsigned rot = (unsigned)(state.hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
  }
  // Generator.random(): 53 bits * 2^-53 (exact)
  __device__ __forceinline__ double next_double() { return (double)(next_u64() >> 11) * (1.0 / 9007199254740992.0); }
  // Generator.uniform(low, high) = low + (high - low) * u, two roundings, never contracted to an FMA
  __device__ __forceinline__ double uniform(double low, double range) {
    return __dadd_rn(low, __dmul_rn(range, next_double()));
  }
};

// SeedSequence(seed).generate_state(8) for a 64-bit seed, then PCG64 seeding (numpy/random/_pcg64.pyx, pcg64_srandom_r)
__device__ inline Pcg64 pcg64_from_seed(uint64_t seed) {
  constexpr uint32_t INIT_A = 0x43b0d7e5u, MULT_A = 0x931e8875u, INIT_B = 0x8b51f9ddu, MULT_B = 0x58f38dedu;
  constexpr uint32_t MIX_L = 0xca01f9ddu, MIX_R = 0x4973f715u;
  uint32_t hc = INIT_A;
  auto hashmix = [&](uint32_t v) {
    v ^= hc;
    hc *= MULT_A;
    v *= hc;
    v ^= v >> 16;
    return v;
  };
  auto mix = [](uint32_t x, uint32_t y) {
    uint32_t r = MIX_L * x - MIX_R * y;
    r ^= r >> 16;
    return r;
  };
  // entropy limbs, zero padded to the pool size (a one-limb and a two-limb seed with a zero high limb coincide)
  uint32_t pool[4] = {hashmix((uint32_t)seed), hashmix((uint32_t)(seed >> 32)), hashmix(0u), hashmix(0u)};
#pragma unroll
  for (int s = 0; s < 4; ++s)
#pragma unroll
    for (int d = 0; d < 4; ++d)
      if (s != d) pool[d] = mix(pool[d], hashmix(pool[s]));
  uint32_t out[8];
  uint32_t hb = INIT_B;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    uint32_t v = pool[i & 3];
    v ^= hb;
    hb *= MULT_B;
    v *= hb;
    v ^= v >> 16;
    out[i] = v;
  }
  uint64_t w0 = out[0] | ((uint64_t)out[1] << 32), w1 = out[2] | ((uint64_t)out[3] << 32);
  uint64_t w2 = out[4] | ((uint64_t)out[5] << 32), w3 = out[6] | ((uint64_t)out[7] << 32);
  u128 initstate{w1, w0}, initseq{w3, w2};
  Pcg64 g;
  g.inc.hi = (initseq.hi << 1) | (initseq.lo >> 63);
  g.inc.lo = (initseq.lo << 1) | 1ull;
  g.state = u128{0, 0};
  g.advance();
  g.state = add128(g.state, initstate);
  g.advance();
  return g;
}

// rng tensor layout: uint64 [2][n][2]: {state lo,hi}[n] then {inc lo,hi}[n]; 16-byte vector accesses, coalesced
__device__ __forceinline__ Pcg64 pcg64_load(const uint64_t* __restrict__ rng, int64_t n, int64_t i) {
  const ulonglong2 s = reinterpret_cast<const ulonglong2*>(rng)[i];
  const ulonglong2 c = __ldg(reinterpret_cast<const ulonglong2*>(rng) + n + i);
  Pcg64 g;
  g.state = u128{s.x, s.y};
  g.inc = u128{c.x, c.y};
  return g;
}
__device__ __forceinline__ void pcg64_store_state(uint64_t* __restrict__ rng, int64_t i, const Pcg64& g) {
  reinterpret_cast<ulonglong2*>(rng)[i] = make_ulonglong2(g.state.lo, g.state.hi);
}
__device__ __forceinline__ void pcg64_store_all(uint64_t* __restrict__ rng, int64_t n, int64_t i, const Pcg64& g) {
  reinterpret_cast<ulonglong2*>(rng)[i] = make_ulonglong2(g.state.lo, g.state.hi);
  reinterpret_cast<ulonglong2*>(rng)[n + i] = make_ulonglong2(g.inc.lo, g.inc.hi);
}

// ---------------------------------------------------------------------------------------------------------------
// Philox4x32-10
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// one 128-bit block for (seed, global env index, counter)
__device__ __forceinline__ uint4 philox_block(uint64_t seed, uint64_t env, uint64_t counter, uint32_t stream_id) {
  return philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)counter,
                                  (uint32_t)(counter >> 32) ^ (stream_id << 24)),
                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
__device__ __forceinline__ double u53_to_double(uint32_t a, uint32_t b) {
  uint64_t v = ((uint64_t)a << 32 | b) >> 11;
  return (double)v * (1.0 / 9007199254740992.0);
}

// action fetch for the discrete families
template <typename T>
__device__ __forceinline__ int load_action(const void* __restrict__ actions, int64_t i) {
  return (int)__ldg(reinterpret_cast<const T*>(actions) + i);
}

}  // namespace b2e
