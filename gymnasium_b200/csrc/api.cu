// api.cu -- library-wide C-ABI entry points (version, errors, device query) and the numpy-parity RNG seeding kernel.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "common.cuh"

namespace b2e {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_batch(const b2e_batch* b, const char* fn) {
  if (!b) {
    set_error("%s: batch descriptor is NULL", fn);
    return B2E_EINVAL;
  }
  if (b->n < 0 || b->env_offset < 0) {
    set_error("%s: n=%lld env_offset=%lld must be >= 0", fn, (long long)b->n, (long long)b->env_offset);
    return B2E_EINVAL;
  }
  if (b->autoreset_mode < 0 || b->autoreset_mode > 2 || b->rng_mode < 0 || b->rng_mode > 1) {
    set_error("%s: bad autoreset_mode=%d or rng_mode=%d", fn, b->autoreset_mode, b->rng_mode);
    return B2E_EINVAL;
  }
  return 0;
}

int cuda_status(cudaError_t e, const char* fn) {
  if (e == cudaSuccess) return 0;
  set_error("%s: CUDA error %d (%s)", fn, (int)e, cudaGetErrorString(e));
  return (int)e;
}

namespace {

// SyncVectorEnv.reset seeds sub-env i with seed+i (sync_vector_env.py:205-208); Env.reset(seed) builds
// Generator(PCG64(SeedSequence(seed))) (gymnasium/utils/seeding.py:39-41).
__global__ void __launch_bounds__(kBlock) rng_seed_kernel(int64_t n, int64_t env_offset, uint64_t base_seed,
                                                          const uint64_t* __restrict__ seeds,
                                                          const uint8_t* __restrict__ mask, uint64_t* __restrict__ rng) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (mask != nullptr && mask[i] == 0) return;
  const uint64_t seed = seeds ? seeds[i] : base_seed + (uint64_t)(env_offset + i);
  pcg64_store_all(rng, n, i, pcg64_from_seed(seed));
}

__global__ void __launch_bounds__(kBlock) rng_random_kernel(int64_t n, uint64_t* __restrict__ rng, int k,
                                                            double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Pcg64 g = pcg64_load(rng, n, i);
  for (int j = 0; j < k; ++j) out[i * k + j] = g.next_double();
  pcg64_store_state(rng, i, g);
}

}  // namespace
}  // namespace b2e

using namespace b2e;

extern "C" int b2e_version(void) { return B2E_VERSION; }

extern "C" const char* b2e_last_error(void) { return g_err; }

extern "C" int b2e_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || device < 0 || device >= count) {
    set_error("b2e_device_info: no CUDA device %d (count=%d, %s)", device, count, cudaGetErrorString(e));
    return B2E_ENODEV;
  }
  cudaDeviceProp p;
  if (int s = cuda_status(cudaGetDeviceProperties(&p, device), "b2e_device_info")) return s;
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (l2_bytes) *l2_bytes = (size_t)p.l2CacheSize;
  return 0;
}

// SIMT FMA throughput probe (the denominator of the FLOP roofline of the physics families): 8 independent chains per thread
template <typename T>
__global__ void __launch_bounds__(256) fma_probe_kernel(int64_t iters, T* sink) {
  T a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = (T)(threadIdx.x + k) * (T)1e-3;
  const T b = (T)0.999, c = (T)1e-6;
  for (int64_t i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = fma(a[k], b, c);
  }
  T acc = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc += a[k];
  if (acc == (T)-1) sink[0] = acc;  // never true: keeps the chains alive
}
extern "C" int b2e_fma_probe(int fp64, int64_t iters, int64_t* flops, void* sink, void* stream) {
  int dev = 0, sms = 0;
  if (!sink || iters <= 0 || cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    set_error("b2e_fma_probe: bad arguments or no device");
    return B2E_EINVAL;
  }
  const int grid = sms * 8;
  if (fp64) fma_probe_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, (double*)sink);
  else fma_probe_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(iters, (float*)sink);
  if (flops) *flops = (int64_t)grid * 256 * iters * 8 * 2;
  return cuda_status(cudaGetLastError(), "b2e_fma_probe");
}

extern "C" int b2e_rng_seed(const b2e_batch* b, uint64_t base_seed, const uint64_t* seeds, const uint8_t* mask,
                            uint64_t* rng, void* stream) {
  if (int e = check_batch(b, "b2e_rng_seed")) return e;
  if (!rng) {
    set_error("b2e_rng_seed: rng is NULL");
    return B2E_EINVAL;
  }
  if (b->n == 0) return 0;
  rng_seed_kernel<<<grid_for(b->n), kBlock, 0, (cudaStream_t)stream>>>(b->n, b->env_offset, base_seed, seeds, mask, rng);
  return cuda_status(cudaGetLastError(), "b2e_rng_seed");
}

extern "C" int b2e_rng_random(const b2e_batch* b, uint64_t* rng, int32_t k, double* out, void* stream) {
  if (int e = check_batch(b, "b2e_rng_random")) return e;
  if (!rng || !out || k < 0) {
    set_error("b2e_rng_random: null pointer or k < 0");
    return B2E_EINVAL;
  }
  if (b->n == 0 || k == 0) return 0;
  rng_random_kernel<<<grid_for(b->n), kBlock, 0, (cudaStream_t)stream>>>(b->n, rng, k, out);
  return cuda_status(cudaGetLastError(), "b2e_rng_random");
}

// ---- single host-side batch (multi-GPU): every rank DMAs its shard's packed step outputs over its own PCIe link into one
// page-locked host buffer that all ranks of the node map (gymnasium_b200/distributed.py: HostBatch)
extern "C" int b2e_host_register(void* host, size_t bytes) {
  if (!host || bytes == 0) {
    set_error("b2e_host_register: null pointer or zero size");
    return B2E_EINVAL;
  }
  return cuda_status(cudaHostRegister(host, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped), "b2e_host_register");
}

extern "C" int b2e_host_unregister(void* host) {
  if (!host) {
    set_error("b2e_host_unregister: null pointer");
    return B2E_EINVAL;
  }
  return cuda_status(cudaHostUnregister(host), "b2e_host_unregister");
}

extern "C" int b2e_copy_to_host_async(const b2e_copy_seg* segs, int32_t count, void* stream) {
  if (!segs || count < 0) {
    set_error("b2e_copy_to_host_async: null segment list or count < 0");
    return B2E_EINVAL;
  }
  for (int32_t i = 0; i < count; ++i) {
    const b2e_copy_seg& g = segs[i];
    if (!g.host_dst || !g.dev_src) {
      set_error("b2e_copy_to_host_async: segment %d has a null pointer", i);
      return B2E_EINVAL;
    }
    if (g.width == 0 || g.height == 0) continue;
    cudaError_t e = g.height == 1
                        ? cudaMemcpyAsync(g.host_dst, g.dev_src, g.width, cudaMemcpyDefault, (cudaStream_t)stream)
                        : cudaMemcpy2DAsync(g.host_dst, g.dst_pitch, g.dev_src, g.src_pitch, g.width, g.height,
                                            cudaMemcpyDefault, (cudaStream_t)stream);
    if (int st = cuda_status(e, "b2e_copy_to_host_async")) return st;
  }
  return 0;
}

// ---- landing kernel: a step's outputs written into the page-locked host batch by the SMs (zero-copy stores over PCIe) ---
// One launch replaces the copy engine's per-key copies (each costs a few microseconds of DMA set-up, which is what bounds a
// microsecond-kernel family end to end) and publishes the rank's sequence word itself: every CTA fences its stores at system
// scope, the last CTA to finish stores the word.
namespace b2e {
namespace {
constexpr int kLandMaxSegs = 8;
struct LandSeg {
  char* dst;        // device-visible address of the host rows
  const char* src;  // this output set, device memory
  size_t dst_pitch, src_pitch, width, height;
  int32_t vec;      // 1: every row starts 16-byte aligned on both sides and is a multiple of 16 bytes
};
struct LandArgs {
  LandSeg seg[kLandMaxSegs];
  int32_t count;
  int64_t* seq;       // device-visible address of the rank's sequence word in the host batch
  int64_t value;
  unsigned* counter;  // CTAs done (device memory, returns to 0)
};

__global__ void __launch_bounds__(256) land_outputs_kernel(const LandArgs a) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
  for (int s = 0; s < a.count; ++s) {
    const LandSeg& g = a.seg[s];
    if (g.vec) {
      const size_t per_row = g.width / 16, n = per_row * g.height;
      if (g.height == 1) {
        const int4* src = reinterpret_cast<const int4*>(g.src);
        int4* dst = reinterpret_cast<int4*>(g.dst);
        for (size_t c = tid; c < n; c += stride) dst[c] = src[c];
      } else {
        for (size_t c = tid; c < n; c += stride) {
          const size_t r = c / per_row, k = c - r * per_row;
          reinterpret_cast<int4*>(g.dst + r * g.dst_pitch)[k] = reinterpret_cast<const int4*>(g.src + r * g.src_pitch)[k];
        }
      }
    } else {
      const size_t n = g.width * g.height;
      for (size_t c = tid; c < n; c += stride) {
        const size_t r = c / g.width, k = c - r * g.width;
        g.dst[r * g.dst_pitch + k] = g.src[r * g.src_pitch + k];
      }
    }
  }
  __syncthreads();  // the CTA's stores are ordered before thread 0's fence (cumulative at system scope)
  if (threadIdx.x == 0) {
    __threadfence_system();
    const unsigned prev = atomicAdd(a.counter, 1u);
    if (prev == gridDim.x - 1) {  // every other CTA's rows are visible to the host: publish
      *a.counter = 0;
      __threadfence_system();
      *reinterpret_cast<volatile int64_t*>(a.seq) = a.value;
    }
  }
}

struct LandPlan {
  LandArgs args;
  int grid;
};
}  // namespace
}  // namespace b2e
using namespace b2e;

// ---- pipelined end-to-end step in ONE host call (gymnasium_b200/distributed.py: HostBatchPipeline) ----------------------
extern "C" int b2e_pipe_slot_init(b2e_pipe_slot* s) {
  if (!s) {
    set_error("b2e_pipe_slot_init: slot is NULL");
    return B2E_EINVAL;
  }
  cudaEvent_t ev[3];
  for (int i = 0; i < 3; ++i)
    if (int st = cuda_status(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming), "b2e_pipe_slot_init")) return st;
  s->ev_h2d = ev[0];
  s->ev_step = ev[1];
  s->ev_copy = ev[2];
  s->h2d_pending = s->copy_pending = 0;
  s->land = nullptr;
  return 0;
}

// A landing plan: the device-visible addresses of `count` output segments + the rank's sequence word, and the CTA counter.
extern "C" int b2e_land_plan_create(const b2e_copy_seg* segs, int32_t count, int64_t* seq_host, void** plan_out) {
  if (!segs || count < 0 || !seq_host || !plan_out) {
    set_error("b2e_land_plan_create: null pointer or count < 0");
    return B2E_EINVAL;
  }
  if (count > kLandMaxSegs) {
    set_error("b2e_land_plan_create: %d output keys, at most %d", count, kLandMaxSegs);
    return B2E_EINVAL;
  }
  LandPlan* p = new LandPlan();
  memset(p, 0, sizeof(*p));
  size_t chunks = 0;
  for (int i = 0; i < count; ++i) {
    const b2e_copy_seg& g = segs[i];
    LandSeg& d = p->args.seg[i];
    void* dev = nullptr;
    if (int st = cuda_status(cudaHostGetDevicePointer(&dev, g.host_dst, 0), "b2e_land_plan_create (host batch not mapped)")) {
      delete p;
      return st;
    }
    d.dst = (char*)dev;
    d.src = (const char*)g.dev_src;
    d.width = g.width;
    d.height = g.height ? g.height : 1;
    d.dst_pitch = d.height > 1 ? g.dst_pitch : g.width;
    d.src_pitch = d.height > 1 ? g.src_pitch : g.width;
    const uintptr_t bits = (uintptr_t)d.dst | (uintptr_t)d.src | d.width | (d.height > 1 ? (d.dst_pitch | d.src_pitch) : 0);
    d.vec = (bits & 15) == 0;
    chunks += (d.vec ? d.width / 16 : d.width) * d.height;
  }
  p->args.count = count;
  void* seq_dev = nullptr;
  if (int st = cuda_status(cudaHostGetDevicePointer(&seq_dev, seq_host, 0), "b2e_land_plan_create (sequence word)")) {
    delete p;
    return st;
  }
  p->args.seq = (int64_t*)seq_dev;
  if (int st = cuda_status(cudaMalloc(&p->args.counter, sizeof(unsigned)), "b2e_land_plan_create (counter)")) {
    delete p;
    return st;
  }
  cudaMemset(p->args.counter, 0, sizeof(unsigned));
  int dev_id = 0, sms = 148;
  cudaGetDevice(&dev_id);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_id);
  // few CTAs: measured on B200 (scripts/link_probe.py, 1.7 MB): 37 CTAs 40.9 us, 148 CTAs 41.9, 296+ CTAs 45.8 (copy engine: 33.3)
  const size_t cap = (size_t)(sms / 4 > 0 ? sms / 4 : 1);
  const size_t want = (chunks + 255) / 256;
  p->grid = (int)(want < 1 ? 1 : (want > cap ? cap : want));
  *plan_out = p;
  return cuda_status(cudaDeviceSynchronize(), "b2e_land_plan_create");
}

extern "C" int b2e_land_plan_launch(void* plan, int64_t seq_value, void* stream) {
  if (!plan) {
    set_error("b2e_land_plan_launch: plan is NULL");
    return B2E_EINVAL;
  }
  LandPlan* p = (LandPlan*)plan;
  p->args.value = seq_value;
  land_outputs_kernel<<<p->grid, 256, 0, (cudaStream_t)stream>>>(p->args);
  return cuda_status(cudaGetLastError(), "b2e_land_plan_launch");
}

extern "C" int b2e_land_plan_destroy(void* plan) {
  if (!plan) return 0;
  LandPlan* p = (LandPlan*)plan;
  if (p->args.counter) cudaFree(p->args.counter);
  delete p;
  return 0;
}

extern "C" int b2e_pipe_slot_land_kernel(b2e_pipe_slot* s) {
  if (!s || !s->segs || s->nsegs < 2) {
    set_error("b2e_pipe_slot_land_kernel: slot or segments missing");
    return B2E_EINVAL;
  }
  if (s->land) return 0;
  // the last two segments publish the sequence word the copy-engine way; the kernel stores it itself
  return b2e_land_plan_create(s->segs, s->nsegs - 2, (int64_t*)s->segs[s->nsegs - 1].host_dst, &s->land);
}

extern "C" int b2e_pipe_slot_destroy(b2e_pipe_slot* s) {
  if (!s) return 0;
  void** ev[3] = {&s->ev_h2d, &s->ev_step, &s->ev_copy};
  for (int i = 0; i < 3; ++i)
    if (*ev[i]) {
      cudaEventDestroy((cudaEvent_t)*ev[i]);
      *ev[i] = nullptr;
    }
  if (s->land) {
    b2e_land_plan_destroy(s->land);
    s->land = nullptr;
  }
  return 0;
}

typedef int (*b2e_anyfn)(uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t,
                         uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t);

extern "C" int b2e_pipe_submit(b2e_pipe_slot* s, const void* host_actions, void* main_stream, void* copy_stream,
                               const int64_t* ack_word, int64_t need_ack, int64_t seq_value, int32_t flags, double timeout_s) {
  if (!s || !host_actions || !s->actions_dev || !s->calls) {
    set_error("b2e_pipe_submit: null pointer in the slot or its arguments");
    return B2E_EINVAL;
  }
  const bool pinned = (flags & B2E_PIPE_ACTIONS_PINNED) != 0;
  if (!s->land || (!pinned && !s->staging_host)) {
    set_error("b2e_pipe_submit: no landing kernel (b2e_pipe_slot_land_kernel), or no staging buffer for pageable actions");
    return B2E_EINVAL;
  }
  cudaStream_t ms = (cudaStream_t)main_stream, cs = (cudaStream_t)copy_stream;
  const void* h2d_src = host_actions;
  if (!pinned) {
    // (1) stage this step's actions: the DMA that last read the staging buffer must be done
    if (s->h2d_pending)
      if (int st = cuda_status(cudaEventSynchronize((cudaEvent_t)s->ev_h2d), "b2e_pipe_submit (staging)")) return st;
    memcpy(s->staging_host, host_actions, s->action_bytes);
    h2d_src = s->staging_host;
  }
  // (2) the kernel re-uses the output set whose last landing copies must have drained
  if (s->copy_pending)
    if (int st = cuda_status(cudaStreamWaitEvent(ms, (cudaEvent_t)s->ev_copy, 0), "b2e_pipe_submit (output set)")) return st;
  if (int st = cuda_status(cudaMemcpyAsync(s->actions_dev, h2d_src, s->action_bytes, cudaMemcpyHostToDevice, ms),
                           "b2e_pipe_submit (H2D)"))
    return st;
  if (!pinned) {
    cudaEventRecord((cudaEvent_t)s->ev_h2d, ms);
    s->h2d_pending = 1;
  }
  // (3) the family's fused step: the recorded C-ABI call(s), every argument a pointer or an integer
  for (int32_t c = 0; c < s->ncalls; ++c) {
    const b2e_call& k = s->calls[c];
    if (!k.fn || k.nargs < 0 || k.nargs > 16) {
      set_error("b2e_pipe_submit: bad recorded call %d", c);
      return B2E_EINVAL;
    }
    const uint64_t* a = k.args;
    const int st = ((b2e_anyfn)k.fn)(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], a[9], a[10], a[11], a[12], a[13],
                                     a[14], a[15]);
    if (st) return st;  // the callee has set the error text
  }
  cudaEventRecord((cudaEvent_t)s->ev_step, ms);
  cudaStreamWaitEvent(cs, (cudaEvent_t)s->ev_step, 0);
  // (4) the consumer must have released the slot this step lands in
  if (ack_word) {
    const volatile int64_t* ack = ack_word;
    if (*ack < need_ack) {
      struct timespec t0, t1;
      clock_gettime(CLOCK_MONOTONIC, &t0);
      unsigned spins = 0;
      while (*ack < need_ack) {
        if ((++spins & 0x3ffu) == 0) {
          clock_gettime(CLOCK_MONOTONIC, &t1);
          if ((double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec) > timeout_s) {
            set_error("b2e_pipe_submit: timed out waiting for the consumer to release step %lld", (long long)(need_ack - 1));
            return B2E_ETIMEOUT;
          }
          struct timespec nap = {0, 2000};
          nanosleep(&nap, nullptr);  // several ranks may share a core
        }
      }
    }
  }
  // (5) the SMs store the outputs into the host batch, then the sequence word
  if (int st = b2e_land_plan_launch(s->land, seq_value, copy_stream)) return st;
  cudaEventRecord((cudaEvent_t)s->ev_copy, cs);
  s->copy_pending = 1;
  return cuda_status(cudaGetLastError(), "b2e_pipe_submit (landing kernel)");
}
