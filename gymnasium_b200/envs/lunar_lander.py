"""LunarLander-v3 on the B200 engine.

Mirrors ``LunarLander`` (gymnasium/envs/box2d/lunar_lander.py:79-665) behind the vector API with SyncVectorEnv's
conventions; the rigid-body solve that the reference delegates to the Box2D wheel runs in
``gymnasium_b200/csrc/lunarlander.cu``.  Discrete actions (``LunarLander-v3``) or ``continuous=True``
(``LunarLanderContinuous-v3``), optional wind / turbulence (``enable_wind``).  Numeric parity with the real Box2D wheel is unpinned (it cannot be installed here); see DESIGN.md.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from .. import _lib
from .._api import AutoresetMode, Box, Discrete
from ..vector_env import B200VectorEnv, ptr


class LunarLanderVectorEnv(B200VectorEnv):
    """N LunarLander-v3 envs.  Observation ``(N, 8) float32``; action ``(N,) int64`` in {0..3}, or with ``continuous=True``
    ``(N, 2) float32`` in [-1, 1] (main throttle, lateral throttle; clipped like the reference); reward float64."""

    metadata = {"render_modes": [], "render_fps": 50, "autoreset_mode": AutoresetMode.NEXT_STEP}

    def __init__(self, num_envs: int = 1, max_episode_steps: int | None = 1000, continuous: bool = False,
                 gravity: float = -10.0, enable_wind: bool = False, wind_power: float = 15.0,
                 turbulence_power: float = 1.5, render_mode: str | None = None, **engine_kwargs):
        assert -12.0 < gravity and gravity < 0.0, f"gravity (current value: {gravity}) must be between -12 and 0"  # :233
        if 0.0 > wind_power or wind_power > 20.0:  # :236-246: recommended ranges only
            import warnings

            warnings.warn(f"wind_power value is recommended to be between 0.0 and 20.0, (current value: {wind_power})")
        if 0.0 > turbulence_power or turbulence_power > 2.0:
            import warnings

            warnings.warn(f"turbulence_power value is recommended to be between 0.0 and 2.0, (current value: {turbulence_power})")
        self.continuous, self.enable_wind = bool(continuous), bool(enable_wind)
        self.wind_power, self.turbulence_power = float(wind_power), float(turbulence_power)
        self.discrete_actions = not self.continuous
        low = np.array([-2.5, -2.5, -10.0, -10.0, -2 * math.pi, -10.0, -0.0, -0.0]).astype(np.float32)  # :258-293
        high = np.array([2.5, 2.5, 10.0, 10.0, 2 * math.pi, 10.0, 1.0, 1.0]).astype(np.float32)
        # :298-305: Box(-1, +1, (2,), float32) = (main engine throttle, left-right throttle) / Discrete(4)
        act_space = Box(-1, +1, (2,), dtype=np.float32) if self.continuous else Discrete(4)
        super().__init__(num_envs, Box(low, high), act_space, max_episode_steps=max_episode_steps,
                         render_mode=render_mode, **engine_kwargs)
        self.gravity = float(gravity)
        n, dev = self.num_envs, self.device
        self._cfg = _lib.LunarLanderCfg(gravity=self.gravity, enable_wind=int(self.enable_wind), continuous=int(self.continuous),
                                        wind_power=self.wind_power, turbulence_power=self.turbulence_power)
        words = self._lib.b2e_lunarlander_state_words()
        self._s = {
            "bodies": torch.zeros((21, n), dtype=torch.float32, device=dev),
            "joints": torch.zeros((8, n), dtype=torch.float32, device=dev),
            "terrain": torch.zeros((11, n), dtype=torch.float32, device=dev),
            "fat": torch.zeros((12, n), dtype=torch.float32, device=dev),
            "contacts": torch.zeros((words, n), dtype=torch.int32, device=dev),
            "flags": torch.zeros(n, dtype=torch.int32, device=dev),
            "prev_shaping": torch.zeros(n, dtype=torch.float64, device=dev),
        }
        if self.enable_wind:  # wind pattern offsets + the 32-bit word np_random.integers leaves in PCG64's buffer
            self._s["wind"] = torch.zeros((2, n), dtype=torch.int32, device=dev)
            self._s["u32buf"] = torch.zeros(n, dtype=torch.int64, device=dev)
        self._state = _lib.LunarLanderState(ctrl=self._ctrl.data_ptr(), rng=ptr(self._rng),
                                            **{k: v.data_ptr() for k, v in self._s.items()})

    def _on_streams_seeded(self, lanes):
        """A freshly seeded numpy Generator starts with an empty 32-bit buffer."""
        if self.enable_wind:
            if lanes is None:
                self._s["u32buf"].zero_()
            else:
                self._s["u32buf"].masked_fill_(lanes, 0)

    def _prepare_actions(self, actions):
        if not self.continuous:
            return super()._prepare_actions(actions)
        n = self.num_envs
        if isinstance(actions, torch.Tensor):
            t = actions
            if tuple(t.shape) != (n, 2):
                raise ValueError(f"expected actions of shape ({n}, 2), got {tuple(t.shape)}")
            if t.dtype not in (torch.float32, torch.float64):
                t = t.to(torch.float32)
            return t.to(self.device).contiguous()
        a = np.asarray(actions)
        if a.ndim == 0:
            raise TypeError(f"actions must have a leading dimension of num_envs={n}, got a scalar")
        if a.shape != (n, 2):
            raise ValueError(f"expected actions of shape ({n}, 2), got {a.shape}")
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        return super()._prepare_actions(np.ascontiguousarray(a))

    def wind_state(self) -> torch.Tensor:
        """int32 ``(N, 2)``: (wind_idx, torque_idx) per env (``enable_wind=True``)."""
        return self._s["wind"].t().contiguous()

    def _alloc_outputs(self):
        n = self.num_envs
        layout = {"obs": ((n, 8), torch.float32), "reward": ((n,), torch.float64),
                  "terminated": ((n,), torch.bool), "truncated": ((n,), torch.bool)}
        if self.autoreset_mode == AutoresetMode.SAME_STEP:
            layout["final_obs"] = ((n, 8), torch.float32)
        out = self._alloc_packed(layout)
        if "final_obs" in out:
            out["final_obs"].zero_()
        return out

    def _reset_kernel(self, mask, options, out):
        if mask is not None and self.copy and self._has_reset:
            out["obs"].copy_(self._last_obs)
        _lib.check(
            self._lib.b2e_lunarlander_reset(C.byref(self._batch), C.byref(self._cfg), C.byref(self._state),
                                            ptr(None if mask is None else mask.view(torch.uint8)), ptr(out["obs"]),
                                            self._stream),
            "b2e_lunarlander_reset",
        )
        self._last_obs = out["obs"]

    def _step_kernel(self, actions, out):
        _lib.check(
            self._lib.b2e_lunarlander_step(C.byref(self._batch), C.byref(self._cfg), C.byref(self._state), ptr(actions),
                                           ptr(out["obs"]), ptr(out["reward"]), ptr(out["terminated"]),
                                           ptr(out["truncated"]), ptr(out.get("final_obs")), self._stream),
            "b2e_lunarlander_step",
        )
        self._last_obs = out["obs"]

    def _step_info(self, out):
        if self.autoreset_mode == AutoresetMode.SAME_STEP:
            done = out["terminated"] | out["truncated"]
            return {"final_obs": out["final_obs"], "_final_obs": done, "final_info": {}, "_final_info": done}
        return {}

    # introspection used by the parity tests ------------------------------------------------------------------------
    def body_state(self) -> torch.Tensor:
        """float32 ``(N, 3, 7)``: per body (lander, legs[0], legs[1]) c.x, c.y, angle, v.x, v.y, w, sleepTime."""
        return self._s["bodies"].view(3, 7, self.num_envs).permute(2, 0, 1).contiguous()

    def contact_overflow(self) -> bool:
        """True if any env ever ran out of contact slots (never expected for this scene)."""
        return bool(((self._s["flags"] >> 12) & 1).any())
