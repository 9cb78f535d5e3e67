"""ctypes binding of libb200env.so (the C-ABI declared in include/b200env.h).

There is NO CPU fallback: if the shared library is missing, fails to load, or there is no CUDA device, the engine
raises.  Build the library with ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C gymnasium_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B2E_LIB_PATH: load another build of the same library (e.g. one installed elsewhere, or a build to compare against)
LIB_PATH = os.environ.get("B2E_LIB_PATH") or os.path.join(_HERE, "libb200env.so")

# enums (include/b200env.h)
AUTORESET_NEXT_STEP, AUTORESET_SAME_STEP, AUTORESET_DISABLED = 0, 1, 2
RNG_NUMPY, RNG_PHILOX = 0, 1
ACT_I64, ACT_I32, ACT_U8, ACT_F32, ACT_F64 = 0, 1, 2, 3, 4

c_void_p, c_i32, c_i64, c_u64, c_double = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double


class Batch(C.Structure):
    """``b2e_batch``."""

    _fields_ = [
        ("n", c_i64),
        ("env_offset", c_i64),
        ("max_episode_steps", c_i32),
        ("autoreset_mode", c_i32),
        ("rng_mode", c_i32),
        ("action_dtype", c_i32),
        ("philox_seed", c_u64),
        ("call_counter", c_u64),
    ]


class CartPoleCfg(C.Structure):
    """``b2e_cartpole_cfg``."""

    _fields_ = [("reset_low", c_double), ("reset_high", c_double), ("sutton_barto_reward", c_i32)]


class FrozenLakeCfg(C.Structure):
    """``b2e_frozenlake_cfg``."""

    _fields_ = [
        ("n_states", c_i32),
        ("n_actions", c_i32),
        ("table", c_void_p),
        ("isd_cum", c_void_p),
        ("cum3", c_double * 3),
        ("p3", c_double * 3),
        ("rewards", c_double * 3),
    ]


class ClassicCfg(C.Structure):
    """``b2e_classic_cfg``."""

    _fields_ = [("family", c_i32), ("_pad", c_i32), ("p", c_double * 4), ("state", c_void_p), ("sflag", c_void_p),
                ("ctrl", c_void_p), ("rng", c_void_p)]


class BlackjackCfg(C.Structure):
    """``b2e_blackjack_cfg``."""

    _fields_ = [("natural", c_i32), ("sab", c_i32), ("hand", c_void_p), ("u32buf", c_void_p), ("ctrl", c_void_p),
                ("rng", c_void_p)]


class LunarLanderCfg(C.Structure):
    """``b2e_lunarlander_cfg``."""

    _fields_ = [("gravity", c_double), ("enable_wind", c_i32), ("continuous", c_i32), ("wind_power", c_double),
                ("turbulence_power", c_double)]


class LunarLanderState(C.Structure):
    """``b2e_lunarlander_state`` (device pointers)."""

    _fields_ = [(k, c_void_p) for k in ("bodies", "joints", "terrain", "fat", "contacts", "flags", "prev_shaping",
                                        "ctrl", "rng", "wind", "u32buf")]


class HumanoidCfg(C.Structure):
    """``b2e_humanoid_cfg``."""

    _fields_ = [(k, c_double) for k in ("reset_noise_scale", "forward_reward_weight", "ctrl_cost_weight",
                                        "contact_cost_weight", "contact_cost_max", "healthy_reward", "healthy_z_min",
                                        "healthy_z_max")] + [("terminate_when_unhealthy", c_i32), ("frame_skip", c_i32),
                                                             ("impl", c_i32), ("_pad", c_i32)]


class HumanoidState(C.Structure):
    """``b2e_humanoid_state`` (device pointers)."""

    _fields_ = [(k, c_void_p) for k in ("qpos", "qvel", "qacc_warmstart", "com_xy", "ctrl", "rng", "overflow", "work",
                                           "order")]


class MjPlanarCfg(C.Structure):
    """``b2e_mjplanar_cfg`` (Hopper-v5, Walker2d-v5)."""

    _fields_ = [(k, c_double) for k in ("reset_noise_scale", "forward_reward_weight", "ctrl_cost_weight", "healthy_reward",
                                        "healthy_z_min", "healthy_z_max", "healthy_angle_min", "healthy_angle_max",
                                        "healthy_state_min", "healthy_state_max")] + [
        ("terminate_when_unhealthy", c_i32), ("frame_skip", c_i32)]


class MjPlanarState(C.Structure):
    """``b2e_mjplanar_state`` (device pointers)."""

    _fields_ = [(k, c_void_p) for k in ("qpos", "qvel", "qacc_warmstart", "ctrl", "rng", "overflow")]


class CopySeg(C.Structure):
    """``b2e_copy_seg``."""

    _fields_ = [("host_dst", c_void_p), ("dev_src", c_void_p), ("dst_pitch", C.c_size_t), ("src_pitch", C.c_size_t),
                ("width", C.c_size_t), ("height", C.c_size_t)]


class Call(C.Structure):
    """``b2e_call``."""

    _fields_ = [("fn", c_void_p), ("nargs", c_i32), ("_pad", c_i32), ("args", c_u64 * 16)]


class PipeSlot(C.Structure):
    """``b2e_pipe_slot``."""

    _fields_ = [("staging_host", c_void_p), ("actions_dev", c_void_p), ("action_bytes", C.c_size_t),
                ("calls", C.POINTER(Call)), ("segs", C.POINTER(CopySeg)), ("ncalls", c_i32), ("nsegs", c_i32),
                ("ev_h2d", c_void_p), ("ev_step", c_void_p), ("ev_copy", c_void_p), ("h2d_pending", c_i32),
                ("copy_pending", c_i32), ("land", c_void_p)]


P = c_void_p
_BP = C.POINTER(Batch)

# symbol -> (restype, argtypes); every symbol include/b200env.h declares must be listed here (tests check both ways)
SIGNATURES = {
    "b2e_version": (C.c_int, []),
    "b2e_last_error": (C.c_char_p, []),
    "b2e_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_size_t)]),
    "b2e_host_register": (C.c_int, [P, C.c_size_t]),
    "b2e_host_unregister": (C.c_int, [P]),
    "b2e_copy_to_host_async": (C.c_int, [P, c_i32, P]),
    "b2e_pipe_slot_init": (C.c_int, [C.POINTER(PipeSlot)]),
    "b2e_pipe_slot_destroy": (C.c_int, [C.POINTER(PipeSlot)]),
    "b2e_pipe_slot_land_kernel": (C.c_int, [C.POINTER(PipeSlot)]),
    "b2e_land_plan_create": (C.c_int, [P, c_i32, P, C.POINTER(c_void_p)]),
    "b2e_land_plan_launch": (C.c_int, [P, c_i64, P]),
    "b2e_land_plan_destroy": (C.c_int, [P]),
    "b2e_pipe_submit": (C.c_int, [C.POINTER(PipeSlot), P, P, P, P, c_i64, c_i64, c_i32, c_double]),
    "b2e_rng_seed": (C.c_int, [_BP, c_u64, P, P, P, P]),
    "b2e_rng_random": (C.c_int, [_BP, P, c_i32, P, P]),
    "b2e_cartpole_reset": (C.c_int, [_BP, C.POINTER(CartPoleCfg), P, P, P, P, P, P]),
    "b2e_cartpole_step": (C.c_int, [_BP, C.POINTER(CartPoleCfg), P, P, P, P, P, P, P, P, P, P]),
    "b2e_cartpole_rollout": (C.c_int, [_BP, C.POINTER(CartPoleCfg), c_i32, P, P, P, P, P, P, P, P, P, P]),
    "b2e_selftest_math": (C.c_int, [c_i64, c_u64, P, P]),
    "b2e_fma_probe": (C.c_int, [C.c_int, c_i64, C.POINTER(c_i64), P, P]),
    "b2e_classic_reset": (C.c_int, [_BP, C.POINTER(ClassicCfg), P, P, P]),
    "b2e_classic_step": (C.c_int, [_BP, C.POINTER(ClassicCfg), P, P, P, P, P, P, P]),
    "b2e_lunarlander_state_words": (C.c_int, []),
    "b2e_taxi_fickle_reset": (C.c_int, [_BP, c_double, P, P, P, P]),
    "b2e_taxi_fickle_step": (C.c_int, [_BP, c_double, P, P, P, P, P, P, P, P]),
    "b2e_blackjack_reset": (C.c_int, [_BP, C.POINTER(BlackjackCfg), P, P, P]),
    "b2e_blackjack_step": (C.c_int, [_BP, C.POINTER(BlackjackCfg), P, P, P, P, P, P, P]),
    "b2e_lunarlander_reset": (C.c_int, [_BP, C.POINTER(LunarLanderCfg), C.POINTER(LunarLanderState), P, P, P]),
    "b2e_lunarlander_step": (C.c_int, [_BP, C.POINTER(LunarLanderCfg), C.POINTER(LunarLanderState), P, P, P, P, P, P,
                                       P]),
    "b2e_humanoid_model_info": (C.c_int, [P, P, P]),
    "b2e_humanoid_reset": (C.c_int, [_BP, C.POINTER(HumanoidCfg), C.POINTER(HumanoidState), P, P, P, P]),
    "b2e_humanoid_step": (C.c_int, [_BP, C.POINTER(HumanoidCfg), C.POINTER(HumanoidState), P, P, P, P, P, P, P, P]),
    "b2e_hopper_model_info": (C.c_int, [P, P, P]),
    "b2e_hopper_reset": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P]),
    "b2e_hopper_step": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P, P, P, P, P]),
    "b2e_walker2d_model_info": (C.c_int, [P, P, P]),
    "b2e_walker2d_reset": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P]),
    "b2e_walker2d_step": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P, P, P, P, P]),
    "b2e_half_cheetah_model_info": (C.c_int, [P, P, P]),
    "b2e_half_cheetah_reset": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P]),
    "b2e_half_cheetah_step": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P, P, P, P, P]),
    "b2e_inverted_pendulum_model_info": (C.c_int, [P, P, P]),
    "b2e_inverted_pendulum_reset": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P]),
    "b2e_inverted_pendulum_step": (C.c_int, [_BP, C.POINTER(MjPlanarCfg), C.POINTER(MjPlanarState), P, P, P, P, P, P, P, P]),
    "b2e_frozenlake_reset": (C.c_int, [_BP, C.POINTER(FrozenLakeCfg), P, P, P, P, P, P, P]),
    "b2e_frozenlake_step": (C.c_int, [_BP, C.POINTER(FrozenLakeCfg), P, P, P, P, P, P, P, P, P, P, P, P]),
    "b2e_frozenlake_rollout": (C.c_int, [_BP, C.POINTER(FrozenLakeCfg), c_i32, P, P, P, P, P, P, P, P, P, P]),
}


class B200EnvError(RuntimeError):
    """A libb200env call returned non-zero."""


_lib = None


def load() -> C.CDLL:
    """Load libb200env.so once; raises if it is not built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is not built. Run `make -C gymnasium_b200/csrc` (needs nvcc, targets sm_100a). "
            "gymnasium_b200 has no CPU fallback."
        )
    import torch  # noqa: F401  -- loads the CUDA runtime (libcudart.so.12) this library links against dynamically

    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.b2e_version() != 1:
        raise ImportError(f"libb200env.so ABI version {lib.b2e_version()} != 1; rebuild it")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().b2e_last_error().decode(errors="replace")
        raise B200EnvError(f"{what} failed with status {status}: {msg}")


def device_info(device: int = 0) -> dict:
    lib = load()
    sm, maj, mnr, l2 = C.c_int(), C.c_int(), C.c_int(), C.c_size_t()
    check(lib.b2e_device_info(device, C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(l2)), "b2e_device_info")
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "l2_bytes": l2.value}
