"""Humanoid-v5 on the B200 engine.

Mirrors ``HumanoidEnv`` v5 (gymnasium/envs/mujoco/humanoid_v5.py:24-541) and the ``MujocoEnv`` plumbing it uses
(gymnasium/envs/mujoco/mujoco_env.py:35-229) behind the vector API with SyncVectorEnv's conventions; the multibody
dynamics the reference delegates to the MuJoCo wheel run in ``gymnasium_b200/csrc/humanoid.cu``.
Numeric parity with the real MuJoCo wheel is unpinned (it cannot be installed here); see DESIGN.md.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from .._api import AutoresetMode, Box
from ..vector_env import B200VectorEnv, ptr

INFO_KEYS = ("x_position", "y_position", "tendon_length", "tendon_velocity", "distance_from_origin", "x_velocity",
             "y_velocity", "reward_survive", "reward_forward", "reward_ctrl", "reward_contact")
_IMPLS = {"warp": 0, "thread": 1}  # b2e_humanoid_cfg.impl: kernel mapping (same results bit for bit)
OBS_SIZE = 22 + 23 + 130 + 78 + 17 + 78  # humanoid_v5.py:376-393


class HumanoidVectorEnv(B200VectorEnv):
    """N Humanoid-v5 envs.  Observation ``(N, 348) float64``, action ``(N, 17) float32`` in [-0.4, 0.4], reward float64,
    info = the 11 keys of ``HumanoidEnv.step`` as ``(N,)`` / ``(N, 2)`` arrays with their ``_key`` masks."""

    metadata = {"render_modes": [], "render_fps": 67, "autoreset_mode": AutoresetMode.NEXT_STEP}
    discrete_actions = False
    soa_output_keys = ("info",)  # outputs laid out [c][n] rather than [n][...] (distributed.HostBatch lands them pitched)

    def __init__(self, num_envs: int = 1, max_episode_steps: int | None = 1000, xml_file: str = "humanoid.xml",
                 frame_skip: int = 5, forward_reward_weight: float = 1.25, ctrl_cost_weight: float = 0.1,
                 contact_cost_weight: float = 5e-7, contact_cost_range=(-np.inf, 10.0), healthy_reward: float = 5.0,
                 terminate_when_unhealthy: bool = True, healthy_z_range=(1.0, 2.0), reset_noise_scale: float = 1e-2,
                 exclude_current_positions_from_observation: bool = True, include_cinert_in_observation: bool = True,
                 include_cvel_in_observation: bool = True, include_qfrc_actuator_in_observation: bool = True,
                 include_cfrc_ext_in_observation: bool = True, render_mode: str | None = None,
                 impl: str = "warp", **engine_kwargs):
        if impl not in _IMPLS:
            raise ValueError(f"impl must be one of {sorted(_IMPLS)}, got {impl!r}")
        if xml_file != "humanoid.xml":
            raise NotImplementedError("gymnasium_b200 compiles the stock humanoid.xml only")
        # observation layout (humanoid_v5.py:376-393, :436-470): the kernel always writes the full 348 columns
        # qpos[2:] (22) | qvel (23) | cinert[1:] (130) | cvel[1:] (78) | qfrc_actuator[6:] (17) | cfrc_ext[1:] (78); the
        # non-default flags select columns of it (and prepend qpos[0:2], which the info block carries) on the way out
        keep = [(0, 45, True), (45, 175, include_cinert_in_observation), (175, 253, include_cvel_in_observation),
                (253, 270, include_qfrc_actuator_in_observation), (270, 348, include_cfrc_ext_in_observation)]
        cols = np.concatenate([np.arange(a, b) for a, b, on in keep if on])
        self._prepend_xy = not exclude_current_positions_from_observation
        self._obs_cols = None if len(cols) == OBS_SIZE else cols
        obs_size = len(cols) + (2 if self._prepend_xy else 0)
        self.observation_structure = {  # humanoid_v5.py:399-407
            "skipped_qpos": 2 * bool(exclude_current_positions_from_observation),
            "qpos": 24 - 2 * bool(exclude_current_positions_from_observation), "qvel": 23,
            "cinert": 130 * bool(include_cinert_in_observation), "cvel": 78 * bool(include_cvel_in_observation),
            "qfrc_actuator": 17 * bool(include_qfrc_actuator_in_observation),
            "cfrc_ext": 78 * bool(include_cfrc_ext_in_observation), "ten_length": 0, "ten_velocity": 0}
        if contact_cost_range[0] > 0 or not np.isneginf(contact_cost_range[0]) and contact_cost_range[0] != 0:
            raise NotImplementedError("contact_cost_range lower bounds other than -inf/0 are not implemented")
        obs_space = Box(low=-np.inf, high=np.inf, shape=(obs_size,), dtype=np.float64)  # humanoid_v5.py:395-397
        act_space = Box(low=-0.4, high=0.4, shape=(17,), dtype=np.float32)             # ctrlrange, mujoco_env.py:105-110
        super().__init__(num_envs, obs_space, act_space, max_episode_steps=max_episode_steps, render_mode=render_mode,
                         **engine_kwargs)
        n, dev = self.num_envs, self.device
        self.frame_skip = int(frame_skip)
        self.dt = 0.003 * self.frame_skip  # mujoco_env.py:189-191
        self._cfg = _lib.HumanoidCfg(
            reset_noise_scale=float(reset_noise_scale), forward_reward_weight=float(forward_reward_weight),
            ctrl_cost_weight=float(ctrl_cost_weight), contact_cost_weight=float(contact_cost_weight),
            contact_cost_max=float(contact_cost_range[1]), healthy_reward=float(healthy_reward),
            healthy_z_min=float(healthy_z_range[0]), healthy_z_max=float(healthy_z_range[1]),
            terminate_when_unhealthy=int(bool(terminate_when_unhealthy)), frame_skip=self.frame_skip, impl=_IMPLS[impl])
        self._s = {
            "qpos": torch.zeros((24, n), dtype=torch.float64, device=dev),
            "qvel": torch.zeros((23, n), dtype=torch.float64, device=dev),
            "qacc_warmstart": torch.zeros((23, n), dtype=torch.float64, device=dev),
            "com_xy": torch.zeros((2, n), dtype=torch.float64, device=dev),
            "overflow": torch.zeros(1, dtype=torch.int32, device=dev),
            "work": torch.zeros(n, dtype=torch.int32, device=dev),    # solver work of the last step (scheduling hint)
            "order": torch.zeros(n, dtype=torch.int32, device=dev),   # scratch: envs grouped by that work
        }
        self._last_done = None  # terminated | truncated of the previous step() (NEXT_STEP: those lanes are on their reset call)
        self._info_sid, self._info_prev = -1, None
        self._state = _lib.HumanoidState(ctrl=self._ctrl.data_ptr(), rng=ptr(self._rng),
                                         **{k: v.data_ptr() for k, v in self._s.items()})

    def _alloc_outputs(self):
        n = self.num_envs
        layout = {"obs": ((n, OBS_SIZE), torch.float64), "reward": ((n,), torch.float64), "info": ((13, n), torch.float64),
                  "terminated": ((n,), torch.bool), "truncated": ((n,), torch.bool)}
        if self.autoreset_mode == AutoresetMode.SAME_STEP:
            layout["final_obs"] = ((n, OBS_SIZE), torch.float64)
        out = self._alloc_packed(layout)
        if "final_obs" in out:
            out["final_obs"].zero_()
        return out

    def _prepare_actions(self, actions):
        n = self.num_envs
        if isinstance(actions, torch.Tensor):
            t = actions
            if t.dim() != 2 or tuple(t.shape) != (n, 17):
                raise ValueError(f"Action dimension mismatch. Expected {(n, 17)}, found {tuple(t.shape)}")  # mujoco_env.py:198-201
            if t.dtype not in (torch.float32, torch.float64):
                t = t.to(torch.float32)
            return t.to(self.device).contiguous()
        a = np.asarray(actions)
        if a.ndim == 0:
            raise TypeError(f"actions must have a leading dimension of num_envs={n}, got a scalar")
        if a.shape != (n, 17):
            raise ValueError(f"Action dimension mismatch. Expected {(n, 17)}, found {a.shape}")
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        return super()._prepare_actions(np.ascontiguousarray(a))

    def _reset_kernel(self, mask, options, out):
        if mask is not None:
            if self.copy and self._has_reset:
                out["obs"].copy_(self._last_obs)
            out["info"].zero_()
        _lib.check(
            self._lib.b2e_humanoid_reset(C.byref(self._batch), C.byref(self._cfg), C.byref(self._state),
                                         ptr(None if mask is None else mask.view(torch.uint8)), ptr(out["obs"]),
                                         ptr(out["info"]), self._stream),
            "b2e_humanoid_reset",
        )
        self._last_obs = out["obs"]

    def _step_kernel(self, actions, out):
        _lib.check(
            self._lib.b2e_humanoid_step(C.byref(self._batch), C.byref(self._cfg), C.byref(self._state), ptr(actions),
                                        ptr(out["obs"]), ptr(out["reward"]), ptr(out["terminated"]),
                                        ptr(out["truncated"]), ptr(out["info"]), ptr(out.get("final_obs")), self._stream),
            "b2e_humanoid_step",
        )
        self._last_obs = out["obs"]

    def _info_dict(self, out, mask, keys):
        raw = out["info"]
        host = isinstance(raw, np.ndarray)
        n = self.num_envs
        if mask is None:
            mask = np.ones(n, dtype=np.bool_) if host else torch.ones(n, dtype=torch.bool, device=self.device)
        rows = {"x_position": raw[0], "y_position": raw[1], "tendon_length": raw[2:4].T, "tendon_velocity": raw[4:6].T,
                "distance_from_origin": raw[6], "x_velocity": raw[7], "y_velocity": raw[8], "reward_survive": raw[9],
                "reward_forward": raw[10], "reward_ctrl": raw[11], "reward_contact": raw[12]}
        info = {}
        for k in keys:
            info[k] = rows[k]
            info["_" + k] = mask
        return info

    def _reset_info(self, out, mask):
        # HumanoidEnv._get_reset_info (humanoid_v5.py:534-541): the five state keys
        if mask is None:
            self._last_done = None
        elif self._last_done is not None:  # lanes reset by hand are no longer waiting for their autoreset call
            self._last_done = self._same_kind(self._last_done, mask) & ~mask
        self._info_sid = -1
        return self._info_dict(out, mask, INFO_KEYS[:5])

    def _same_kind(self, x, like):
        """x as a numpy array / torch tensor, whichever `like` is (the output kind may be switched between calls)."""
        if isinstance(x, np.ndarray) == isinstance(like, np.ndarray):
            return x
        return x.cpu().numpy() if isinstance(x, torch.Tensor) else torch.as_tensor(x, device=self.device)

    def _step_info(self, out):
        """Info of a step call.  In NEXT_STEP mode a lane whose previous step ended its episode is on its reset call
        (sync_vector_env.py:279-284) and reports only the five keys of ``_get_reset_info``; in SAME_STEP mode a lane that
        ends its episode has its step info replaced by the reset info (:302-319).  The masks of the six step-only keys
        (velocities, reward terms) are therefore False on those lanes, as ``SyncVectorEnv._add_info`` leaves them."""
        done = out["terminated"] | out["truncated"]
        sid = int(self._batch.call_counter)
        if sid != self._info_sid:  # step_wait() asks again for the same step (host arrays): keep that step's predecessor
            self._info_sid, self._info_prev = sid, self._last_done
        info = self._info_dict(out, None, INFO_KEYS[:5])
        step_mask = None
        if self.autoreset_mode == AutoresetMode.NEXT_STEP and self._info_prev is not None:
            step_mask = ~self._same_kind(self._info_prev, done)
        elif self.autoreset_mode == AutoresetMode.SAME_STEP:
            step_mask = ~done
        info.update(self._info_dict(out, step_mask, INFO_KEYS[5:]))
        self._last_done = done.copy() if isinstance(done, np.ndarray) else done
        if self.autoreset_mode == AutoresetMode.SAME_STEP:
            info.update({"final_obs": out["final_obs"], "_final_obs": done})
        return info

    # ---- non-default observation layouts: column selection on the way out ----------------------------------------------
    def _shape_obs(self, obs, info_block):
        if self._obs_cols is None and not self._prepend_xy:
            return obs
        host = isinstance(obs, np.ndarray)
        if self._obs_cols is not None:
            if host:
                obs = obs[:, self._obs_cols]
            else:
                if not hasattr(self, "_obs_cols_dev"):
                    self._obs_cols_dev = torch.as_tensor(self._obs_cols, device=self.device)
                obs = obs.index_select(1, self._obs_cols_dev)
        if self._prepend_xy:
            xy = info_block[0:2].T
            obs = np.concatenate([xy, obs], axis=1) if host else torch.cat([xy, obs], dim=1)
        return obs

    def _custom_layout(self) -> bool:
        return self._obs_cols is not None or self._prepend_xy

    def _host_obs(self, host):
        return self._shape_obs(host["obs"], host["info"])

    def reset(self, *, seed=None, options=None):
        obs, info = super().reset(seed=seed, options=options)
        if self._custom_layout():
            raw = self._pinned_np_info() if isinstance(obs, np.ndarray) else self._out["info"]
            obs = self._shape_obs(obs, raw)
        return obs, info

    def step(self, actions):
        obs, reward, terminated, truncated, info = super().step(actions)
        if self._custom_layout():
            if self.autoreset_mode == AutoresetMode.SAME_STEP and self._prepend_xy:
                raise NotImplementedError("exclude_current_positions_from_observation=False is not available in SAME_STEP mode")
            raw = self._pinned_np_info() if isinstance(obs, np.ndarray) else self._out["info"]
            obs = self._shape_obs(obs, raw)
            if "final_obs" in info:
                info["final_obs"] = self._shape_obs(info["final_obs"], raw)
        return obs, reward, terminated, truncated, info

    def _pinned_np_info(self):
        """The info block [13][n] of the last host copy (output='numpy')."""
        for k, shape, dt, off, nbytes in self._wire_layout:
            if k == "info":
                return self._pinned_np[off:off + nbytes].view(np.float64).reshape(shape)
        raise KeyError("info")

    # introspection -------------------------------------------------------------------------------------------------
    def qpos(self) -> torch.Tensor:
        return self._s["qpos"].t().contiguous()

    def qvel(self) -> torch.Tensor:
        return self._s["qvel"].t().contiguous()

    def buffer_overflow(self) -> bool:
        """True if any env ever exhausted the per-env contact (12) or constraint-row (24) buffers."""
        return bool(self._s["overflow"].item())
