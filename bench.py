#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused step+autoreset hot path on B200 (contract in the task statement).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA engine
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU vectorisers on the host cores

A "step" is ONE vectorised step() over ONE batch of --num-envs (65536) CartPole-v1 envs = one launch of
cartpole_step_kernel.  Workload = BASELINE.json configs[1]: "CartPole-v1 65536 envs on 1 B200, fused step+auto-reset
kernel", random actions, NEXT_STEP autoreset, TimeLimit 500, numpy-parity PCG64 streams (seed + i).

Timed region (value): inputs resident in HBM.  To keep every launch HBM-cold the bench rotates over a RING of independent
65536-env batches whose total footprint is > 2x the L2 (so a batch's state has been evicted before it is stepped again),
launched as CUDA graphs, timed with CUDA events on the launch stream, max over ranks.
e2e: the public API (`gymnasium_b200.make_vec(...).step(host_actions)` -> host numpy arrays) with the pinned
host->device action copy and the device->host result copy inside every step.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env steps/sec at N=65536 random-action, 1/2/4/8 B200 vs CPU AsyncVectorEnv"
UNIT = "env-steps/s"
# algorithmic HBM bytes per env-step of cartpole_step_kernel (DESIGN.md section 4): read state 4xf64 + ctrl i32 +
# action i64, write state + ctrl + obs 4xf32 + reward f64 + terminated u8 + truncated u8
CARTPOLE_STEP_BYTES = (32 + 4 + 8) + (32 + 4 + 16 + 8 + 1 + 1)
FROZENLAKE_STEP_BYTES = (16 + 16 + 4 + 4 + 8) + (16 + 4 + 4 + 8 + 8 + 1 + 1 + 8)  # rng state+inc, s, ctrl, act | outs
ROLLOUT_STEP_BYTES = 16 + 4 + 1 + 1  # obs f32x4 + reward f32 + flags per env-step streamed by the fused-K kernel


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_ncu_traffic(kernel_key):
    """dram bytes per launch from the committed ncu capture (profiles/ncu_summary.json), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel_key, {}).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock + clock-event reasons through NVML in a background thread while the timed regions run."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index, period=0.02):
        self.samples, self.windows, self.period, self._stop = [], [], period, threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _one(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        try:
            reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        self.samples.append((time.perf_counter(), mhz, reasons))

    def _run(self):
        while not self._stop.is_set():
            try:
                self._one()
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self.t.start()
        return self

    def window(self):
        s = self

        class W:
            def __enter__(self_w):
                self_w.t0 = time.perf_counter()

            def __exit__(self_w, *a):
                s.windows.append((self_w.t0, time.perf_counter()))
                if s.ok:
                    try:
                        s._one()
                    except Exception:
                        pass

        return W()

    def stop(self):
        self._stop.set()
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        self.t.join(timeout=1)
        inside = [(m, r) for (t, m, r) in self.samples if any(a - 0.005 <= t <= b + 0.005 for a, b in self.windows)]
        if not inside:
            inside = [(m, r) for (_, m, r) in self.samples]
        bits = 0
        for _, r in inside:
            bits |= r
        return {"sm_mhz": statistics.median([m for m, _ in inside]) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in self.REASONS.items() if bits & k), "samples": len(inside)}


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path on this host's cores."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(os.path.join(ref, "gymnasium")) and ref not in sys.path:
        sys.path.insert(0, ref)
    import numpy as np

    cores = effective_cores()
    budget = float(args.ref_budget)
    args.num_envs = args.num_envs or ENV_FACTS[args.env]["default_n"]
    line = {"impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "gpu_launches": 0}
    try:
        import gymnasium as gym
        from gymnasium.utils.performance import benchmark_vector_step

        have_ref = True
    except Exception as e:  # noqa: BLE001
        have_ref, why = False, repr(e)

    alternatives = {}
    if have_ref and args.env in ("LunarLander-v3", "Humanoid-v5", "Hopper-v5"):
        have_ref, why = False, "Box2D / mujoco wheels are not installable here (no runnable reference for this env)"
    if have_ref:
        import warnings

        warnings.filterwarnings("ignore")

        def time_async(C, seconds):
            """AsyncVectorEnv with C worker processes for ~`seconds`: (steps/s calls x C, steps/s without reset calls, calls)."""
            envs = gym.make_vec(args.env, num_envs=C, vectorization_mode="async", **env_kwargs(args.env))
            envs.action_space.seed(0)
            envs.reset(seed=0)
            for _ in range(max(args.warmup, 3)):
                envs.step(envs.action_space.sample())
            done_prev = np.zeros(C, dtype=bool)
            counted = calls = 0
            t0 = time.perf_counter()
            while True:
                for _ in range(20):
                    _, _, te, tr, _ = envs.step(envs.action_space.sample())
                    counted += C - int(done_prev.sum())  # gymnasium/utils/performance.py:88-90
                    done_prev = te | tr
                calls += 20
                dt = time.perf_counter() - t0
                if dt >= seconds:
                    break
            envs.close()
            return calls * C / dt, counted / dt, calls, dt

        # BASELINE.md section 4: C in {cores, 2 cores, 4 cores} worker processes, keep the best and say which
        tried = {}
        best = None
        for mult in (1, 2, 4):
            C = max(2, min(cores * mult, 512))
            try:
                r = time_async(C, budget / 3.0)
            except Exception as ex:  # noqa: BLE001
                tried[f"num_envs={C}"] = f"failed: {ex!r}"
                continue
            tried[f"num_envs={C}"] = r[0]
            if best is None or r[0] > best[1][0]:
                best = (C, r)
        C, (value, value_excl, calls, dt) = best
        args.steps = calls
        total = calls * C
        sample = (f"AsyncVectorEnv({args.env}), one worker process per sub-env (65536 processes is not runnable): best of "
                  f"num_envs in {{C, 2C, 4C}} for C = {cores} effective host cores -> num_envs={C}, {calls} vector calls in "
                  f"{dt:.1f} s, host action sampling included (host budget: {host_cpu_budget()})")
        kind = "reference"
        alternatives["async_by_num_envs"] = tried
        line["value_excluding_reset_calls"] = value_excl
        if not args.no_extras:
            for mode, n, kw in [("sync", 4, {}), ("vector_entry_point", args.num_envs, {})]:
                if mode == "vector_entry_point" and not args.env.startswith("CartPole"):
                    continue
                try:
                    e = gym.make_vec(args.env, num_envs=n, vectorization_mode=mode, **env_kwargs(args.env))
                    alternatives[f"{mode}_n{n}"] = benchmark_vector_step(e, target_duration=3, seed=0)
                    e.close()
                except Exception as ex:  # noqa: BLE001
                    alternatives[f"{mode}_n{n}"] = f"failed: {ex!r}"
        else:
            try:
                e = gym.make_vec(args.env, num_envs=4, vectorization_mode="sync", **env_kwargs(args.env))
                alternatives["sync_n4"] = benchmark_vector_step(e, target_duration=2, seed=0)
                e.close()
            except Exception as ex:  # noqa: BLE001
                alternatives["sync_n4"] = f"failed: {ex!r}"
    else:
        # oracle port (numpy restatement), one core
        from oracle.cartpole import OracleCartPole
        from oracle.frozenlake import OracleFrozenLake

        if args.env == "LunarLander-v3":
            from oracle.lunar_lander import OracleLunarLander

            n, env = 1024, OracleLunarLander(1024)
        elif args.env == "Humanoid-v5":
            from oracle.humanoid import OracleHumanoid

            n, env = 64, OracleHumanoid(64)
        elif args.env == "Hopper-v5":
            from oracle.hopper import OracleHopper

            n, env = 256, OracleHopper(256)
        elif args.env.startswith("CartPole"):
            n = args.num_envs or 65536
            env = OracleCartPole(n)
        else:
            n, env = 4096, OracleFrozenLake(4096, map_name="8x8")
        if args.env in ("LunarLander-v3", "Humanoid-v5", "Hopper-v5"):
            # the C restatement releases the GIL inside its ctypes call: one env batch per host thread, all host cores
            import threading

            T = max(1, min(cores, 256))
            cls = type(env)
            n = {"LunarLander-v3": 2048, "Humanoid-v5": 128, "Hopper-v5": 1024}[args.env]  # long calls: the GIL-held wrapper code stays < 1 %
            pool = host_action_pool(np, args.env, 8, n, 0)
            envs = [cls(n) for _ in range(T)]
            for t, e in enumerate(envs):
                e.reset(seed=1000 * t)
            t0 = time.perf_counter()
            for k in range(3):
                envs[0].step_inplace(np.ascontiguousarray(pool[k % 8]))
            t_call = (time.perf_counter() - t0) / 3
            steps = max(2, min(args.steps * 50, int(budget / t_call)))  # every thread steps its own batch `steps` times
            gate = threading.Barrier(T + 1)

            pool = [np.ascontiguousarray(a) for a in pool]

            def work(e):
                gate.wait()
                for k in range(steps):
                    e.step_inplace(pool[k % 8])  # no allocations / copies under the GIL; the C call releases it
                gate.wait()

            threads = [threading.Thread(target=work, args=(e,)) for e in envs]
            for th in threads:
                th.start()
            gate.wait()
            t0 = time.perf_counter()
            gate.wait()
            dt = time.perf_counter() - t0
            for th in threads:
                th.join()
            total, value = steps * n * T, steps * n * T / dt
            sample = (f"oracle port (C restatement), {T} host threads x {n} envs, {steps} vector steps each ({why}); "
                      f"one thread alone: {n / t_call:.4g} env-steps/s, all threads: {value / (n / t_call):.1f}x that "
                      f"(host budget: {host_cpu_budget()})")
            args.steps = steps
            kind, cores = "port", T
            if args.env == "Humanoid-v5":  # inputs of the FLOP model (SURVEY 8d): constraint rows and PGS sweeps per mj_forward
                e0 = envs[0]
                cnt = np.zeros((0, 3))
                for k in range(40):
                    e0.step(pool[k % 8])
                    cnt = np.concatenate([cnt, np.stack([e0.debug(i)[3] for i in range(n)]).astype(float)])
                solver_stats = {"mean_ncon": float(cnt[:, 0].mean()), "mean_nefc": float(cnt[:, 1].mean()),
                                "mean_pgs_sweeps": float(cnt[:, 2].mean()), "sample": f"{len(cnt)} env-steps (last mj_forward of each)"}
        else:
            pool = host_action_pool(np, args.env, 8, n, 0)
            env.reset(seed=0)
            t0 = time.perf_counter()
            for k in range(max(args.warmup, 3)):
                env.step(pool[k % 8])
            t_call = (time.perf_counter() - t0) / max(args.warmup, 3)
            steps = max(1, min(args.steps, int(budget / t_call)))
            t0 = time.perf_counter()
            for k in range(steps):
                env.step(pool[k % 8])
            dt = time.perf_counter() - t0
            total, value = steps * n, steps * n / dt
            sample = f"oracle port (1 core), N={n}, {steps} vector steps ({why})"
            args.steps = steps
            kind, cores = "port", 1
    if "solver_stats" in locals():
        line["solver_stats"] = solver_stats
    line.update({
        "value": value, "ms_per_step": dt / args.steps * 1e3,
        "config": {"workload": f"{args.env} reference CPU vectoriser, bounded sample: {sample}"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": sample, "alternatives": alternatives},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })
    print(json.dumps(line))
    return 0


def env_kwargs(env_id):
    return {"map_name": "8x8"} if env_id.startswith("FrozenLake") else {}


# per-family bench facts: algorithmic HBM bytes per env-step, dominant kernel, arithmetic type, default batch per GPU
ENV_FACTS = {
    "CartPole-v1": dict(step_bytes=CARTPOLE_STEP_BYTES, kernel="cartpole_step_kernel<int64>", dtype="f64", nact=2,
                        out_bytes=16 + 8 + 1 + 1, act_bytes=8, default_n=65536),
    "FrozenLake-v1": dict(step_bytes=FROZENLAKE_STEP_BYTES, kernel="frozenlake_step_kernel<int64>", dtype="int32+f64",
                          nact=4, out_bytes=8 + 8 + 8 + 1 + 1, act_bytes=8, default_n=1 << 20),
    # state r/w (21+8+12 floats, flags, prev_shaping, ctrl, rng words) + action + outputs; contact slots excluded
    "LunarLander-v3": dict(step_bytes=2 * (41 * 4 + 4 + 8 + 4) + 32 + 8 + 32 + 8 + 2, kernel="lunarlander_step_kernel<int64>",
                           dtype="f32+f64", nact=4, out_bytes=32 + 8 + 1 + 1, act_bytes=8, default_n=16384),
    # qpos/qvel/warmstart/com r+w (72 doubles x 2) + action 17 f32 + obs 348 f64 + reward + info 13 f64 + flags
    "Humanoid-v5": dict(step_bytes=2 * 72 * 8 + 68 + 348 * 8 + 8 + 13 * 8 + 2 + 8, kernel="humanoid_step_warp_kernel<float, 10>", launches_per_step=2,
                        dtype="f64", nact=0, out_bytes=348 * 8 + 8 + 13 * 8 + 2, act_bytes=68, default_n=8192),
    # SURVEY 8f rank 4: qpos/qvel/warmstart r+w (18 doubles x 2) + action 3 f32 + obs 11 f64 + reward + info 6 f64 + flags + ctrl
    "Hopper-v5": dict(step_bytes=2 * 18 * 8 + 12 + 11 * 8 + 8 + 6 * 8 + 2 + 8, kernel="hopper_step_kernel<float>", dtype="f64",
                      nact=0, act_dim=3, act_range=1.0, out_bytes=11 * 8 + 8 + 6 * 8 + 2, act_bytes=12, default_n=16384),
}


def device_actions(torch, env_id, shape_prefix, n, dev, gen=None):
    f = ENV_FACTS[env_id]
    if f["nact"]:
        return torch.randint(0, f["nact"], (*shape_prefix, n), device=dev, dtype=torch.int64, generator=gen)
    k, r = f.get("act_dim", 17), f.get("act_range", 0.4)
    return (torch.rand((*shape_prefix, n, k), device=dev, generator=gen) * (2 * r) - r).float()


FLOP_BOUND = ("Humanoid-v5", "LunarLander-v3", "Hopper-v5")  # families whose bound is SIMT arithmetic latency/throughput, not HBM


def measure_fma_peak(torch, dev, fp64):
    """SIMT FMA peak of this GPU in TFLOP/s (b2e_fma_probe, CUDA events, best of 3)."""
    import ctypes as C

    from gymnasium_b200 import _lib

    lib = _lib.load()
    sink = torch.zeros(4, dtype=torch.float64, device=dev)
    flops = C.c_int64(0)
    st = torch.cuda.current_stream(dev)
    best = 0.0
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        _lib.check(lib.b2e_fma_probe(int(fp64), 1 << 14, C.byref(flops), sink.data_ptr(), st.cuda_stream), "b2e_fma_probe")
        e1.record(st)
        torch.cuda.synchronize(dev)
        if it:
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def flop_roofline(env_id, steps_per_s_per_gpu, peak_tflops, cpu_baseline):
    """Algorithmic FLOPs per env-step (SURVEY.md 8d model) x measured steps/s against the measured SIMT FMA peak."""
    if env_id == "Humanoid-v5":
        st = (cpu_baseline or {}).get("solver_stats") or {}
        nefc = st.get("mean_nefc", HUMANOID_NOMINAL_STATS["mean_nefc"])
        sweeps = st.get("mean_pgs_sweeps", HUMANOID_NOMINAL_STATS["mean_pgs_sweeps"])
        nv = 23
        f_fwd = 30e3 + 10e3 + nefc * (2 * nv * nv + 2 * nefc * nv) + sweeps * 2 * nefc * nefc
        flops = 20 * f_fwd + 2e3
        model = (f"20 x (30k smooth + 10k collision + nefc(2 nv^2 + 2 nefc nv) + sweeps 2 nefc^2) + 2k, nv=23, "
                 f"nefc={nefc:.2f}, sweeps={sweeps:.2f} ({'measured on the oracle sample of this run' if st else 'oracle sample of ' + HUMANOID_NOMINAL_STATS['source']})")
        dtype = "f64"
    elif env_id == "Hopper-v5":
        nv, nefc, sweeps = 6, 5.0, 20.0
        f_fwd = 4e3 + 1e3 + nefc * (2 * nv * nv + 2 * nefc * nv) + sweeps * 2 * nefc * nefc
        flops = 16 * f_fwd  # frame_skip 4 x RK4
        model, dtype = ("16 x (4k smooth + 1k collision + nefc(2 nv^2 + 2 nefc nv) + sweeps 2 nefc^2), nv=6, nominal nefc=5, "
                        "sweeps=20 (SURVEY 8d formula scaled to the 6-dof model)"), "f64"
    else:
        flops, model, dtype = 47.5e3, "nominal 45-50 kflop per Box2D step (180 velocity + 60 position iterations)", "f32"
    achieved = flops * steps_per_s_per_gpu / 1e12
    return {"bound": "simt-" + dtype, "flops_per_env_step": flops, "model": model, "achieved": achieved,
            "peak": peak_tflops, "unit": "TFLOP/s", "frac": achieved / peak_tflops if peak_tflops else None,
            "peak_source": "b2e_fma_probe measured in this run (8 FMA chains/thread, 8 CTAs x 256 threads per SM)",
            "note": "serial dependency chains per env (tree recursions, factorisation pivots, Gauss-Seidel sweeps): the "
                    "kernel is bound by dependent-issue latency at 8 warps/SM, see profiles/ for the stall breakdown"}


def effective_cores():
    """CPUs this process may really use: min(scheduler affinity, cgroup CPU quota) -- os.cpu_count() counts the machine."""
    b = host_cpu_budget()
    c = b.get("sched_affinity") or b.get("os_cpu_count") or 1
    q = b.get("cgroup_cpu_max")
    if q:
        c = min(c, max(1, int(math.ceil(q))))
    return max(1, int(c))


def host_cpu_budget():
    """What the container may actually use: os.cpu_count() counts the machine's CPUs, the cgroup quota can be smaller."""
    out = {"os_cpu_count": os.cpu_count()}
    try:
        out["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        out["cgroup_cpu_max"] = None if quota == "max" else round(int(quota) / int(period), 2)
    except Exception:  # noqa: BLE001
        pass
    return out


def host_action_pool(np, env_id, count, n, seed):
    f = ENV_FACTS[env_id]
    rs = np.random.default_rng(seed)
    if f["nact"]:
        return rs.integers(0, f["nact"], size=(count, n)).astype(np.int64)
    k, r = f.get("act_dim", 17), f.get("act_range", 0.4)
    return rs.uniform(-r, r, size=(count, n, k)).astype(np.float32)


# ----------------------------------------------------------------------------------------------------------------------
BURN_IN = {"LunarLander-v3": 120, "Humanoid-v5": 60, "Hopper-v5": 40}  # untimed steps per batch that bring a physics family to its steady mix
PIPE_DEPTH = 3  # output sets / host slots in flight (see pipe_depth())


def pipe_depth(env_id):
    """Deeper for the families whose step is much shorter than the host's per-step work: the ranks then run ahead of the
    consumer by several steps and per-step jitter (scheduling, the consumer's own submit) averages out instead of stalling all ranks."""
    return 8 if env_id in ("CartPole-v1", "FrozenLake-v1") else PIPE_DEPTH
# constraint rows / PGS sweeps per mj_forward of the random-action steady state (oracle sample, profiles/r1_bench_humanoid.json);
# used for the FLOP model when the run has no fresh oracle sample (N > 1)
HUMANOID_NOMINAL_STATS = {"mean_nefc": 2.71, "mean_pgs_sweeps": 12.29, "source": "profiles/r1_bench_humanoid.json"}


class Ctx:
    pass


def bind_near_gpu(index):
    """Runs this rank on the CPUs of its GPU's NUMA node (what `numactl --cpunodebind` under torchrun does): the rank's
    launches, its slice of the host-side batch (first touch) and the DMA target are then local to the GPU's root complex."""
    try:
        import pynvml

        import torch

        pynvml.nvmlInit()
        try:  # CUDA_VISIBLE_DEVICES may renumber the devices: find the NVML device by its PCI address
            p = torch.cuda.get_device_properties(index)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{p.pci_domain_id:08X}:{p.pci_bus_id:02X}:{p.pci_device_id:02X}.0".encode())
        except Exception:  # noqa: BLE001
            h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no GPU-local CPUs in this process' affinity mask"
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} CPUs of GPU {index}'s NUMA node (nvmlDeviceGetCpuAffinity)"
    except Exception as e:  # noqa: BLE001 -- placement is an optimisation, never a requirement
        return f"not bound ({type(e).__name__}: {e})"


def make_ctx(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from gymnasium_b200 import _lib
    from gymnasium_b200.distributed import env_rank_world

    cx = Ctx()
    cx.np, cx.torch, cx.dist = np, torch, dist
    cx.rank, cx.local_rank, cx.world = env_rank_world()
    if cx.world != args.gpus and cx.world > 1:
        args.gpus = cx.world
    torch.cuda.set_device(cx.local_rank)
    cx.dev = torch.device("cuda", cx.local_rank)
    cx.host_affinity = bind_near_gpu(cx.local_rank) if not args.no_bind else "not bound (--no-bind)"
    if cx.world > 1:
        dist.init_process_group("nccl", device_id=cx.dev)
    cx.info = _lib.device_info(cx.local_rank)
    cx.hbm_peak, cx.peak_src = load_peaks()
    cx.sampler = ClockSampler(cx.local_rank).start() if cx.rank == 0 else None
    return cx


def sync_all(cx):
    cx.torch.cuda.synchronize()
    if cx.world > 1:
        cx.dist.barrier()
        cx.torch.cuda.synchronize()


def max_over_ranks(cx, x):
    if cx.world == 1:
        return x
    t = cx.torch.tensor([x], dtype=cx.torch.float64, device=cx.dev)
    cx.dist.all_reduce(t, op=cx.dist.ReduceOp.MAX)
    return float(t.item())


class _NullWindow:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def clock_window(cx):
    return cx.sampler.window() if cx.sampler else _NullWindow()


def measure_device(cx, args, env_id, n, K, W, ring_arg=0):
    """`value`: inputs resident in HBM.  A ring of independent n-env batches (footprint > 2 x L2 for the HBM-bound families)
    is stepped round-robin, one fused launch per bench step, and the steps are ordered so that every timed launch finds
    its batch evicted from L2.  After the set-up, exactly K step launches are timed: one CUDA graph holds the W warm-up
    launches, a CUDA event, the K launches and a second event (max over ranks).  `outputs` is what the last timed step
    returned to its caller (device tensors the graph replay writes)."""
    import gymnasium_b200

    torch, dev, rank = cx.torch, cx.dev, cx.rank
    facts = ENV_FACTS[env_id]
    kw = env_kwargs(env_id)
    foot = n * (facts["step_bytes"] + 32)  # + the PCG64 words each batch also owns
    ring = ring_arg or max(2, math.ceil(2.0 * cx.info["l2_bytes"] / foot))
    if env_id in FLOP_BOUND and not ring_arg:
        ring = min(ring, 4)  # latency/FLOP-bound families: L2 residency is irrelevant, keep set-up short
    T = 8  # distinct action vectors per batch
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    envs, acts = [], []
    for j in range(ring):
        e = gymnasium_b200.make_vec(env_id, num_envs=n, device=dev, copy=False, env_offset=(rank * ring + j) * n, **kw)
        e.reset(seed=0)
        envs.append(e)
        acts.append(device_actions(torch, env_id, (T,), n, dev, gen))
    torch.cuda.synchronize()

    def launch(i):  # one bench step = one fused step launch on the next batch of the ring
        j = i % ring
        return envs[j].step(acts[j][(i // ring) % T])

    burn = BURN_IN.get(env_id, 0)
    setup = ring * (1 + burn)
    for i in range(setup):  # every code path once + the steady-state mix of a physics family (set-up, untimed)
        launch(i)
    # ONE graph: the W warm-up launches (ending on the last batch of the ring), an event, the K timed launches from the
    # first batch, an event.  The events are nodes of the graph, so no launch boundary or host gap falls in the window.
    a, b = (torch.cuda.Event(enable_timing=True, external=True) for _ in range(2))
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(setup - W, setup):
            launch(i)
        a.record()
        for i in range(setup, setup + K):
            outputs = launch(i)
        b.record()
    g.replay()  # uploads the graph (set-up, untimed)
    # `pad` set-up launches continue the round-robin up to the batch before the warm-up's first, so that every timed
    # launch finds its batch the least recently stepped one
    pad = -(W + K) % ring
    for i in range(setup + K, setup + K + pad):
        launch(i)
    sync_all(cx)
    with clock_window(cx):
        sync_all(cx)
        g.replay()
        sync_all(cx)
    elapsed = max_over_ranks(cx, a.elapsed_time(b) * 1e-3)
    del g
    reset_frac = float(torch.stack([(e._ctrl < 0).float().mean() for e in envs]).mean().item())
    cold = ring * foot > 2 * cx.info["l2_bytes"]
    return {
        "value": cx.world * K * n / elapsed, "elapsed_s": elapsed, "timed_steps": K, "graph_launches": W + K,
        "ms_per_step": elapsed / K * 1e3, "ring": ring, "foot": foot, "reset_frac": reset_frac, "envs": envs,
        "acts": acts, "outputs": outputs,
        "l2_policy": (f"inputs larger than L2: ring of {ring} independent {n}-env batches ({ring * foot / 1e6:.0f} MB > 2 x "
                      f"{cx.info['l2_bytes'] / 1e6:.0f} MB L2) stepped round-robin; the timed launches step the batches "
                      f"in least-recently-stepped order, so no timed launch is L2-warm"
                      if cold else
                      f"ring of {ring} independent {n}-env batches ({ring * foot / 1e6:.0f} MB); this family is latency/FLOP-"
                      f"bound, not HBM-bound, so L2 residency does not affect the timing"),
    }


DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs at most


def dump_outputs(directory, outputs):
    """Writes what one step() returned -- obs, reward, terminated, truncated and the info arrays ("info.<key>", nested keys
    joined by ".") -- as <directory>/<name>.npy in float32 (flags, small integers) or float64 (other integers).  Above
    DUMP_LIMIT bytes in all, every array keeps the same fixed, seeded sample of env rows, listed in env_index.npy."""
    import numpy as np
    import torch

    obs, reward, terminated, truncated, info = outputs
    arrays = {"obs": obs, "reward": reward, "terminated": terminated, "truncated": truncated}

    def add_info(d, prefix):
        for k, v in d.items():
            if isinstance(v, dict):
                add_info(v, f"{prefix}{k}.")
            elif isinstance(v, torch.Tensor):
                arrays[prefix + k] = v

    add_info(info, "info.")
    host = {}
    for k, v in arrays.items():
        a = v.detach().cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64)
        host[k] = a
    n = len(host["reward"])
    row_bytes = sum(a.nbytes for a in host.values()) / n
    if row_bytes * n > DUMP_LIMIT:
        m = int((DUMP_LIMIT - 1024 * len(host)) // (row_bytes + 8))  # 1 KB per file for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, m, replace=False))
        host = {k: a[idx] for k, a in host.items()}
        host["env_index"] = idx.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def measure_e2e(cx, args, env_id, n, mode, tag):
    """End to end through the public API with HOST buffers: every step copies that step's actions from pinned host memory to
    the device, runs the fused launch and lands the step's outputs in the single host-side batch
    (gymnasium_b200.distributed.HostBatchPipeline).  mode 'dma': every rank writes its rows over its own PCIe link;
    'nccl': one NCCL gather to rank 0 + rank 0's D2H.  Both overlap step k's copies with step k+1's kernel.  Wall clock
    around K_e steps + the drain of the last one, barrier on both sides, max over ranks."""
    import gymnasium_b200
    from gymnasium_b200.distributed import HostBatchPipeline

    torch, np, dev, rank, world = cx.torch, cx.np, cx.dev, cx.rank, cx.world
    facts = ENV_FACTS[env_id]
    kw = env_kwargs(env_id)
    depth = pipe_depth(env_id)
    env = gymnasium_b200.make_vec(env_id, num_envs=n, device=dev, copy=False, out_buffers=depth, env_offset=rank * n, **kw)
    env.reset(seed=0)
    burn = BURN_IN.get(env_id, 0)
    if burn:  # same steady-state mix as the device-resident batches (untimed set-up)
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        dev_pool = device_actions(torch, env_id, (4,), n, dev, gen)
        for k in range(burn):
            env.step(dev_pool[k % 4])
        torch.cuda.synchronize()
    pipe = HostBatchPipeline(env, world, rank, tag=tag, depth=depth, mode=mode)
    pool = host_action_pool(np, env_id, 16, n, rank)
    # this step's inputs live in page-locked host memory (16 distinct action batches, cycled): the pipeline DMAs from them;
    # `--pageable-actions` measures the variant that takes pageable numpy arrays (one extra host copy into a staging buffer)
    host_actions = list(pool) if args.pageable_actions else pipe.pinned_actions(16, dtype=pool.dtype)
    for dst, src in zip(host_actions, pool):
        dst[...] = src
    check = {}

    lag = max(1, depth // 2)  # the consumer takes step k - lag after submitting step k: it rarely has to wait for the slowest rank
    done = [0]                # steps consumed so far (consumer rank)

    def run(count):
        last = -1
        for _ in range(count):
            t = pipe.submit(host_actions[pipe.k % 16])
            if pipe.is_consumer and t >= lag:
                pipe.consume(t - lag)
                done[0] = t - lag + 1
            last = t
        if pipe.is_consumer:
            while done[0] <= last:  # drain: every submitted step is consumed inside the timed region
                check["batch"] = pipe.consume(done[0])
                done[0] += 1
        pipe.drain()

    warm = max(5, min(args.warmup, 50))
    run(warm)  # first calls: lazy initialisation (pinned staging buffers, copy segments, NCCL channels)
    sync_all(cx)
    t0 = time.perf_counter()
    run(warm)
    sync_all(cx)
    t_est = max_over_ranks(cx, (time.perf_counter() - t0) / warm)
    Ke = int(min(args.e2e_steps, max(20, math.ceil(0.3 / t_est))))
    Ke = int(max_over_ranks(cx, float(Ke)))
    with clock_window(cx):
        sync_all(cx)
        t0 = time.perf_counter()
        run(Ke)
        sync_all(cx)
        elapsed = max_over_ranks(cx, time.perf_counter() - t0)
    ok = None
    if pipe.is_consumer:  # the landed batch is the real thing: right shapes, finite observations from every rank
        bt = check["batch"]
        ok = bool(bt["obs"].shape[0] == n * world and np.isfinite(np.asarray(bt["obs"], dtype=np.float64)).all())
    landing = pipe.landing if pipe._fast else "copies (python path)"
    pipe.close()
    del env
    return {"value": world * Ke * n / elapsed, "unit": UNIT, "h2d_bytes_per_step": n * facts["act_bytes"],
            "d2h_bytes_per_step": n * facts["out_bytes"], "steps": Ke, "ms_per_step": elapsed / Ke * 1e3,
            "host_batch_ok": ok, "pipeline_depth": depth,
            "actions": "pageable numpy (staged)" if args.pageable_actions else "page-locked numpy (pipe.pinned_actions)",
            "landing": {"kernel": "landing kernel: SM stores into the mapped host batch, one launch per step",
                        "graph": "copy engine, one CUDA graph per step",
                        "copies": "copy engine, one cudaMemcpyAsync per output key"}.get(landing, landing),
            "path": ("gymnasium_b200.distributed.HostBatchPipeline(make_vec(...)).submit(host numpy actions) / .consume(): pinned "
                     "H2D of the actions + fused step launch + " +
                     ("D2H of every rank's rows over its own PCIe link into ONE page-locked host batch shared by all ranks"
                      if mode == "dma" else
                      "ONE NCCL gather of all shards' packed outputs to rank 0 (NVLink) + rank 0's D2H of the gathered batch") +
                     "; the copies of step k overlap the kernel of step k+1")}


def measure_e2e_sync(cx, args, env_id, n):
    """The blocking call: env.step(host numpy actions) -> host numpy arrays (H2D + launch + one D2H + stream sync per call)."""
    import gymnasium_b200

    torch, np, dev = cx.torch, cx.np, cx.dev
    env = gymnasium_b200.make_vec(env_id, num_envs=n, device=dev, copy=False, output="numpy", **env_kwargs(env_id))
    env.reset(seed=0)
    burn = BURN_IN.get(env_id, 0)
    if burn:
        gen = torch.Generator(device=dev).manual_seed(7)
        dev_pool = device_actions(torch, env_id, (4,), n, dev, gen)
        env.output = "torch"
        for k in range(burn):
            env.step(dev_pool[k % 4])
        env.output = "numpy"
        torch.cuda.synchronize()
    host_actions = host_action_pool(np, env_id, 16, n, 0)
    for k in range(5):
        env.step(host_actions[k % 16])
    t0 = time.perf_counter()
    for k in range(5):
        env.step(host_actions[k % 16])
    t_est = (time.perf_counter() - t0) / 5
    Ke = int(min(args.e2e_steps, max(20, math.ceil(0.3 / t_est))))
    with clock_window(cx):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(Ke):
            env.step(host_actions[k % 16])
        torch.cuda.synchronize()
        elapsed = time.perf_counter() - t0
    return {"value": Ke * n / elapsed, "unit": UNIT, "steps": Ke, "ms_per_step": elapsed / Ke * 1e3,
            "path": "gymnasium_b200.make_vec(..., output='numpy').step(host numpy actions) -> host numpy arrays (blocking)"}


def family_block(cx, args, env_id, n, K, W, with_sync_e2e, fma_cache, cpu_baseline=None):
    """Everything measured for one family at this world size: device-timed value, roofline, pipelined e2e (+ NCCL variant)."""
    facts = ENV_FACTS[env_id]
    res = measure_device(cx, args, env_id, n, K, W, args.ring if env_id == args.env else 0)
    envs, acts, outputs = res.pop("envs"), res.pop("acts"), res.pop("outputs")
    per_gpu = res["value"] / cx.world
    kernel_s = res["elapsed_s"] / res["timed_steps"]
    if env_id in FLOP_BOUND:
        fp64 = env_id in ("Humanoid-v5", "Hopper-v5")
        if fp64 not in fma_cache:
            fma_cache[fp64] = measure_fma_peak(cx.torch, cx.dev, fp64=fp64)
        roof = flop_roofline(env_id, per_gpu, fma_cache[fp64], cpu_baseline)
        roof["kernel"] = facts["kernel"]
        roof["avg_launch_us"] = kernel_s * 1e6
        roof["traffic"] = load_ncu_traffic(facts["kernel"])
        hbm = facts["step_bytes"] * n / kernel_s / 1e9
        roof["hbm"] = {"achieved_GBs": hbm, "frac_of_hbm_peak": hbm / cx.hbm_peak,
                       "algorithmic_bytes_per_env_step": facts["step_bytes"]}
    else:
        achieved = facts["step_bytes"] * n / kernel_s / 1e9
        roof = {"kernel": facts["kernel"], "bound": "hbm", "achieved": achieved, "peak": cx.hbm_peak, "unit": "GB/s",
                "frac": achieved / cx.hbm_peak, "peak_source": cx.peak_src,
                "algorithmic_bytes_per_env_step": facts["step_bytes"], "avg_launch_us": kernel_s * 1e6,
                "traffic": load_ncu_traffic(facts["kernel"])}
    block = {k: res[k] for k in ("value", "ms_per_step", "timed_steps", "graph_launches", "l2_policy")}
    block["timed_region_ms"] = res["elapsed_s"] * 1e3
    block["value_excluding_reset_calls"] = res["value"] * (1 - res["reset_frac"])
    block["reset_call_fraction"] = res["reset_frac"]
    block["roofline"] = roof
    block["gpu_launches"] = res["timed_steps"] * facts.get("launches_per_step", 1)
    return block, envs, acts, outputs


def run_b200(args):
    import gymnasium_b200

    cx = make_ctx(args)
    torch, rank, world, dev = cx.torch, cx.rank, cx.world, cx.dev
    facts = ENV_FACTS[args.env]
    n = args.num_envs or facts["default_n"]
    args.num_envs = n
    K, W = args.steps, args.warmup
    fma_cache = {}

    # CPU baselines first (rank 0, N = 1 only): the Humanoid oracle sample also feeds the FLOP model
    cpu_baseline = None
    cpu_other = {}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_subprocess(args, args.env, n, 12)

    block, envs, acts, outputs = family_block(cx, args, args.env, n, K, W, True, fma_cache, cpu_baseline)
    if args.dump_outputs and rank == 0:  # before anything else steps these batches
        dump_outputs(args.dump_outputs, outputs)
    del outputs
    extras = {}
    if not args.no_extras and rank == 0 and world == 1:  # supporting numbers belong to the 1-GPU line
        try:
            extras = run_extras(args, cx, gymnasium_b200, envs[0], acts[0], fma_cache)
        except Exception as e:  # noqa: BLE001 -- supporting numbers must never cost the headline line
            extras = {"extras_error": f"{type(e).__name__}: {e}"}
    del envs, acts
    torch.cuda.empty_cache()

    e2e = measure_e2e(cx, args, args.env, n, "dma", "main")
    if world > 1:
        e2e["nccl_gather_variant"] = measure_e2e(cx, args, args.env, n, "nccl", "main")
    else:
        e2e["blocking_step_variant"] = measure_e2e_sync(cx, args, args.env, n)

    # BASELINE configs[4] / north_star: Humanoid-v5, 8192 envs per GPU, at EVERY world size (SCALE carries the curve)
    humanoid = None
    if args.env.startswith("CartPole") and not args.no_humanoid:
        hn = ENV_FACTS["Humanoid-v5"]["default_n"]
        hcpu = None
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            hcpu = cpu_baseline_subprocess(args, "Humanoid-v5", hn, 10)
        humanoid, henvs, hacts, _ = family_block(cx, args, "Humanoid-v5", hn, K, W, False, fma_cache, hcpu)
        del henvs, hacts
        torch.cuda.empty_cache()
        humanoid["e2e"] = measure_e2e(cx, args, "Humanoid-v5", hn, "dma", "hum")
        if world > 1:
            humanoid["e2e"]["nccl_gather_variant"] = measure_e2e(cx, args, "Humanoid-v5", hn, "nccl", "hum")
        humanoid["cpu_baseline"] = hcpu
        humanoid["config"] = {"workload": f"Humanoid-v5 {hn} envs per GPU (BASELINE configs[4]), random actions U[-0.4,0.4]^17, "
                                          f"NEXT_STEP autoreset, TimeLimit 1000, steady state after {BURN_IN['Humanoid-v5']} burn-in steps",
                              "num_envs_per_gpu": hn, "dtype": "f64"}
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.no_extras and args.env.startswith("CartPole"):
        cpu_other["FrozenLake-v1"] = cpu_baseline_subprocess(args, "FrozenLake-v1", 1 << 20, 8)
        cpu_other["LunarLander-v3"] = cpu_baseline_subprocess(args, "LunarLander-v3", 16384, 8)
        if "frozenlake_8x8_1M" in extras:
            extras["frozenlake_8x8_1M"]["cpu_baseline"] = cpu_other["FrozenLake-v1"]
        if "lunarlander_16384" in extras:
            extras["lunarlander_16384"]["cpu_baseline"] = cpu_other["LunarLander-v3"]
        if "hopper_16384" in extras:
            extras["hopper_16384"]["cpu_baseline"] = cpu_baseline_subprocess(args, "Hopper-v5", 16384, 6)

    clocks = cx.sampler.stop() if cx.sampler else None
    if rank == 0:
        line = {
            "metric": METRIC, "value": block["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": block["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": facts["dtype"], "data": "synthetic",
            "config": {
                "workload": f"{args.env} {n} envs per GPU, fused step+auto-reset kernel, random actions, NEXT_STEP "
                            f"autoreset, TimeLimit, numpy-parity PCG64 streams",
                "num_envs_per_gpu": n, "parallelism": f"env-shards x{world} (no data-path collective)",
                "l2_policy": block["l2_policy"],
                "launch": (f"one CUDA graph of {block['graph_launches']} step launches: {W} warm-up launches, then the "
                           f"{block['timed_steps']} timed ones (--steps) between two CUDA event nodes of the graph, "
                           f"{block['timed_region_ms']:.3f} ms region"),
                "counting": "calls x N (reset calls included); see value_excluding_reset_calls",
                "steady_state": (f"{BURN_IN[args.env]} untimed burn-in steps per batch before warm-up" if args.env in BURN_IN else None),
            },
            "timing": {k: block[k] for k in ("timed_steps", "graph_launches", "timed_region_ms")},
            "value_excluding_reset_calls": block["value_excluding_reset_calls"],
            "reset_call_fraction": block["reset_call_fraction"],
            "gpu_launches": block["gpu_launches"],
            "roofline": block["roofline"],
            "e2e": e2e,
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "device": torch.cuda.get_device_name(dev),
            "host_affinity": cx.host_affinity,
        }
        if humanoid is not None:
            line["humanoid_8192_per_gpu"] = humanoid
        line.update(extras)
        print(json.dumps(line))
    if world > 1:
        cx.dist.destroy_process_group()
    return 0


def run_extras(args, cx, gymnasium_b200, env0, acts0, fma_cache):
    """Supporting measurements (rank 0, N = 1): the same kernel at a DRAM-sized batch, the fused-K rollout kernel, the
    L2-resident single-batch rate, the launch floor, FrozenLake and LunarLander at their BASELINE sizes."""
    torch, dev, sampler, hbm_peak = cx.torch, cx.dev, cx.sampler, cx.hbm_peak
    out = {}
    is_cartpole = args.env.startswith("CartPole")
    facts = ENV_FACTS[args.env]
    nact = facts["nact"]
    kw = env_kwargs(args.env)
    if not nact or args.env == "LunarLander-v3":
        return out  # the supporting numbers below are for the HBM-bound discrete families

    def timed(fn, iters, warm=3, min_s=0.05):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total, count = 0.0, 0
        with clock_window(cx):
            while total < min_s and count < 200 * iters:
                a.record()
                for _ in range(iters):
                    fn()
                b.record()
                torch.cuda.synchronize()
                total += a.elapsed_time(b) * 1e-3
                count += iters
        return total / count

    step_bytes = CARTPOLE_STEP_BYTES if is_cartpole else FROZENLAKE_STEP_BYTES
    # (0) launch floor of this part: a graph-replayed chain of the cheapest possible kernel (32-env step launches)
    tiny = gymnasium_b200.make_vec(args.env, num_envs=32, device=dev, copy=False, **kw)
    tiny.reset(seed=0)
    ta = torch.zeros(32, dtype=torch.int64, device=dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(512):
            tiny.step(ta)
    t = timed(g.replay, 10) / 512
    out["launch_floor"] = {"us_per_graph_node": t * 1e6,
                           "note": "the same step kernel over 32 envs, 512 launches per CUDA graph: what one graph node costs "
                                   "on this part with no data to move; N=65536 moves 6.9 MB = 1.06 us at the HBM peak on top"}
    del g, tiny
    # (1) L2-resident: one batch stepped back to back (what a single training loop sees)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for t_ in range(256):
            env0.step(acts0[t_ % acts0.shape[0]])
    t = timed(g.replay, 10) / 256
    out["l2_resident"] = {"steps_per_s": args.num_envs / t, "us_per_launch": t * 1e6,
                          "note": f"single {args.num_envs}-env batch, state stays in L2 (not HBM-cold)"}
    del g
    # (2) same step kernel, DRAM-sized batch: kernel quality away from the launch-latency floor
    big = 1 << 24
    e = gymnasium_b200.make_vec(args.env, num_envs=big, device=dev, copy=False, **kw)
    e.reset(seed=0)
    a = torch.randint(0, nact, (big,), device=dev, dtype=torch.int64)
    t = timed(lambda: e.step(a), 20)
    bw = step_bytes * big / t / 1e9
    out["roofline_large_batch"] = {"kernel": "same step kernel, N=16,777,216 (1.7 GB footprint)", "achieved": bw,
                                   "peak": hbm_peak, "unit": "GB/s", "frac": bw / hbm_peak,
                                   "steps_per_s": big / t, "us_per_launch": t * 1e6}
    del e, a
    torch.cuda.empty_cache()
    # (3) fused K-step rollout kernel with on-device Philox actions, trajectory streamed to HBM
    Kf = 64
    e = gymnasium_b200.make_vec(args.env, num_envs=args.num_envs, device=dev, **kw)
    e.reset(seed=0)
    t = timed(lambda: e.rollout(Kf), 30)
    rb = (ROLLOUT_STEP_BYTES if is_cartpole else 8 + 4 + 1 + 1)
    out["rollout_fused"] = {"K": Kf, "steps_per_s": args.num_envs * Kf / t, "us_per_env_batch_step": t / Kf * 1e6,
                            "hbm_write_GBs": rb * args.num_envs * Kf / t / 1e9,
                            "frac_of_hbm_peak": rb * args.num_envs * Kf / t / 1e9 / hbm_peak,
                            "bytes_per_env_step": rb, "gpu_launches": 1,
                            "note": f"{Kf} steps per launch, state in registers, [K,N] trajectory written once"}
    del e
    if is_cartpole:
        # (4) BASELINE configs[2]: FrozenLake-v1 8x8, 1,048,576 envs
        nfl = 1 << 20
        ringf = 4  # 4 x 103 MB > 2 x L2
        fls = []
        for j in range(ringf):
            f = gymnasium_b200.make_vec("FrozenLake-v1", num_envs=nfl, map_name="8x8", device=dev, copy=False,
                                        env_offset=j * nfl)
            f.reset(seed=0)
            fls.append((f, torch.randint(0, 4, (nfl,), device=dev, dtype=torch.int64)))
        k = [0]

        def fstep():
            f, a = fls[k[0] % ringf]
            f.step(a)
            k[0] += 1

        t = timed(fstep, 40, warm=8)
        bw = FROZENLAKE_STEP_BYTES * nfl / t / 1e9
        out["frozenlake_8x8_1M"] = {"steps_per_s": nfl / t, "us_per_launch": t * 1e6,
                                    "roofline": {"kernel": "frozenlake_step_kernel<int64>", "bound": "hbm", "achieved": bw,
                                                 "peak": hbm_peak, "unit": "GB/s", "frac": bw / hbm_peak,
                                                 "algorithmic_bytes_per_env_step": FROZENLAKE_STEP_BYTES},
                                    "l2_policy": f"ring of {ringf} batches of 1,048,576 envs (inputs larger than L2)"}
        del fls
        torch.cuda.empty_cache()
        # (5) BASELINE configs[3]: LunarLander-v3, 16384 envs (latency-bound rigid-body solve: FLOP roofline, not HBM)
        nl = 16384
        ll = gymnasium_b200.make_vec("LunarLander-v3", num_envs=nl, device=dev, copy=False)
        ll.reset(seed=0)
        la = torch.randint(0, 4, (8, nl), device=dev, dtype=torch.int64)
        k = [0]

        def lstep():
            ll.step(la[k[0] % 8])
            k[0] += 1

        t = timed(lstep, 100, warm=BURN_IN["LunarLander-v3"])
        if False not in fma_cache:
            fma_cache[False] = measure_fma_peak(torch, dev, fp64=False)
        out["lunarlander_16384"] = {"steps_per_s": nl / t, "us_per_launch": t * 1e6,
                                    "roofline": flop_roofline("LunarLander-v3", nl / t, fma_cache[False], None),
                                    "note": "one fused step+autoreset launch per call, random actions, steady state after 120 "
                                            "burn-in steps; bit-exact vs oracle/lunar_lander.c (Box2D parity unpinned)"}
        # (6) SURVEY 8f rank 4: Hopper-v5 (the Humanoid solver on another MuJoCo robot), 16384 envs
        nh = 16384
        hp = gymnasium_b200.make_vec("Hopper-v5", num_envs=nh, device=dev, copy=False)
        hp.reset(seed=0)
        ha = (torch.rand((8, nh, 3), device=dev) * 2 - 1).float()
        k = [0]

        def hstep():
            hp.step(ha[k[0] % 8])
            k[0] += 1

        t = timed(hstep, 20, warm=BURN_IN["Hopper-v5"])
        if True not in fma_cache:
            fma_cache[True] = measure_fma_peak(torch, dev, fp64=True)
        out["hopper_16384"] = {"steps_per_s": nh / t, "us_per_launch": t * 1e6,
                               "roofline": flop_roofline("Hopper-v5", nh / t, fma_cache[True], None),
                               "note": "Hopper-v5, one thread per env, random actions U[-1,1]^3, steady state after 40 burn-in "
                                       "steps; bit-exact vs oracle/hopper.c (MuJoCo parity unpinned)"}
        del hp
        # (7) InvertedPendulum-v5 and Walker2d-v5 on the same planar kernels
        for env_id, nn, nu, hi in (("InvertedPendulum-v5", 65536, 1, 3.0), ("Walker2d-v5", 16384, 6, 1.0),
                                   ("LunarLanderContinuous-v3", 16384, 2, 1.0)):
            kwp = {"enable_wind": True} if env_id.startswith("LunarLander") else {}
            pe = gymnasium_b200.make_vec(env_id, num_envs=nn, device=dev, copy=False, **kwp)
            pe.reset(seed=0)
            pa = ((torch.rand((8, nn, nu), device=dev) * 2 - 1) * hi).float()
            kk = [0]

            def pstep():
                pe.step(pa[kk[0] % 8])
                kk[0] += 1

            t = timed(pstep, 20, warm=40)
            out[env_id.split("-")[0].lower() + f"_{nn}"] = {
                "steps_per_s": nn / t, "us_per_launch": t * 1e6,
                "note": f"{env_id}{' with enable_wind=True' if kwp else ''}, one thread per env, random actions, steady state "
                        "after 40 burn-in steps; bit-exact vs its C oracle (engine parity unpinned; InvertedPendulum pinned to "
                        "the cart-pole equations of motion)"}
            del pe
        for big in (131072, 1048576):
            ll = gymnasium_b200.make_vec("LunarLander-v3", num_envs=big, device=dev, copy=False)
            ll.reset(seed=0)
            la2 = torch.randint(0, 4, (big,), device=dev, dtype=torch.int64)
            t = timed(lambda: ll.step(la2), 10, warm=60)
            out[f"lunarlander_{big}"] = {"steps_per_s": big / t, "us_per_launch": t * 1e6}
        del ll
    return out


def cpu_baseline_subprocess(args, env_id, num_envs, budget_s):
    """Times the reference arm in a fresh process (AsyncVectorEnv forks workers; keep that away from the CUDA context)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "20", "--warmup", "3",
           "--env", env_id, "--num-envs", str(num_envs), "--ref-budget", str(budget_s)]
    if env_id != args.env:
        cmd.append("--no-extras")
    try:
        env = dict(os.environ)
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
            env.pop(k, None)
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
        for ln in reversed(p.stdout.strip().splitlines()):
            if ln.startswith("{"):
                d = json.loads(ln)
                if "solver_stats" in d:
                    d["cpu_baseline"]["solver_stats"] = d["solver_stats"]
                return d["cpu_baseline"]
        return {"error": (p.stderr or p.stdout)[-400:]}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--env", default="CartPole-v1", choices=sorted(ENV_FACTS))
    ap.add_argument("--num-envs", type=int, default=0, help="envs per GPU (0 = the BASELINE size of --env)")
    ap.add_argument("--ring", type=int, default=0, help="batches in the L2-defeating ring (0 = auto: > 2 x L2)")
    ap.add_argument("--e2e-steps", type=int, default=2000)
    ap.add_argument("--ref-budget", type=float, default=20.0, help="seconds of CPU work for the reference arm")
    ap.add_argument("--pageable-actions", action="store_true",
                    help="e2e: pass pageable numpy action batches (staged through one host copy) instead of page-locked ones")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-humanoid", action="store_true", help="skip the Humanoid-v5 8192-envs/GPU block of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of --env returned as DIR/<name>.npy (float32/float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        try:  # the CPU arm gets every core the container has, whatever the parent (a NUMA-bound bench rank) ran on
            os.sched_setaffinity(0, range(os.cpu_count()))
        except OSError:
            pass
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
