"""Generate golden fixtures from the LIVE reference (Gymnasium v1.4.0).

Run in the build container only (the GPU box has no /root/reference):

    PYTHONPATH=/root/reference python tests/golden/make_golden.py

Every fixture is produced by the reference's own ``gymnasium.make_vec(..., vectorization_mode="sync")``
(``gymnasium/envs/registration.py:833``, ``gymnasium/vector/sync_vector_env.py``) stepping the reference's
``CartPoleEnv`` / ``FrozenLakeEnv``; nothing from this repo is involved.  Action tapes are drawn from a
numpy Generator seeded per fixture and stored next to the outputs.
"""
import os
import sys

import numpy as np

import gymnasium as gym
from gymnasium.vector import AutoresetMode

HERE = os.path.dirname(os.path.abspath(__file__))


def rollout(envs, seed, actions, options=None, state_attr=None):
    obs0, info0 = envs.reset(seed=seed, options=options)
    T = actions.shape[0]
    obs = np.zeros((T + 1,) + obs0.shape, dtype=obs0.dtype)
    obs[0] = obs0
    rew = np.zeros((T, envs.num_envs), np.float64)
    term = np.zeros((T, envs.num_envs), bool)
    trunc = np.zeros((T, envs.num_envs), bool)
    extras = {}
    states = []
    if state_attr:
        states.append(np.stack([np.asarray(s, dtype=np.float64) for s in envs.get_attr(state_attr)]))
    disabled = envs.metadata.get("autoreset_mode") == AutoresetMode.DISABLED
    for t in range(T):
        o, r, te, tr, info = envs.step(actions[t])
        obs[t + 1], rew[t], term[t], trunc[t] = o, r, te, tr
        if disabled and (te | tr).any():  # the caller resets finished sub-envs itself (test_autoreset_mode.py:105-260)
            o2, _ = envs.reset(options={"reset_mask": te | tr})
            extras.setdefault("reset_obs", np.zeros((T,) + o2.shape, dtype=np.float64))
            extras["reset_obs"][t] = o2
        for k, v in info.items():
            if k in ("final_obs", "_final_obs", "final_info", "_final_info"):
                continue
            extras.setdefault(k, np.zeros((T,) + v.shape, dtype=np.float64 if not k.startswith("_") else bool))
            extras[k][t] = v
        if state_attr:
            states.append(np.stack([np.asarray(s, dtype=np.float64) for s in envs.get_attr(state_attr)]))
    out = dict(obs=obs, reward=rew, terminated=term, truncated=trunc, actions=actions, seed=np.uint64(seed))
    for k, v in extras.items():
        out["info_" + k] = v
    if state_attr:
        out["state"] = np.stack(states)
    return out


def cartpole(name, n, T, seed, max_episode_steps=None, policy="random", options=None, mode=AutoresetMode.NEXT_STEP,
             **kw):
    mk = dict(max_episode_steps=max_episode_steps) if max_episode_steps else {}
    envs = gym.make_vec("CartPole-v1", num_envs=n, vectorization_mode="sync",
                        vector_kwargs={"autoreset_mode": mode}, **mk, **kw)
    rng = np.random.default_rng(1000 + seed)
    actions = rng.integers(0, 2, size=(T, n)).astype(np.int64)
    if policy == "balance":
        # closed-loop tape: second half of the lanes follow theta+theta_dot sign so they reach the time limit
        e2 = gym.make_vec("CartPole-v1", num_envs=n, vectorization_mode="sync",
                          vector_kwargs={"autoreset_mode": mode}, **mk, **kw)
        o, _ = e2.reset(seed=seed, options=options)
        for t in range(T):
            a = actions[t]
            a[n // 2:] = (o[n // 2:, 2] + 0.5 * o[n // 2:, 3] > 0).astype(np.int64)
            o, _, te_, tr_, _ = e2.step(a)
            if mode == AutoresetMode.DISABLED and (te_ | tr_).any():
                o, _ = e2.reset(options={"reset_mask": te_ | tr_})
        e2.close()
    out = rollout(envs, seed, actions, options=options, state_attr="state")
    out["max_episode_steps"] = np.int64(max_episode_steps or 500)
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")}, "term", out["terminated"].sum(), "trunc",
          out["truncated"].sum())


def frozenlake(name, n, T, seed, mode=AutoresetMode.NEXT_STEP, **kw):
    envs = gym.make_vec("FrozenLake-v1", num_envs=n, vectorization_mode="sync",
                        vector_kwargs={"autoreset_mode": mode}, **kw)
    rng = np.random.default_rng(2000 + seed)
    actions = rng.integers(0, 4, size=(T, n)).astype(np.int64)
    out = rollout(envs, seed, actions)
    out["max_episode_steps"] = np.int64(envs.envs[0].spec.max_episode_steps if "max_episode_steps" not in kw else kw["max_episode_steps"])
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")}, "term", out["terminated"].sum(), "trunc",
          out["truncated"].sum(), "reward", out["reward"].sum())


def classic(name, env_id, n, T, seed, options=None, act_scale=None, nA=None, state_attr="state", policy=None, **kw):
    envs = gym.make_vec(env_id, num_envs=n, vectorization_mode="sync", **kw)
    rng = np.random.default_rng(4000 + seed)
    if nA:
        actions = rng.integers(0, nA, size=(T, n)).astype(np.int64)
    else:  # a few out-of-bound torques/forces exercise the clip paths
        actions = (rng.uniform(-1.15, 1.15, size=(T, n, 1)) * act_scale).astype(np.float32)
    if policy is not None:  # closed-loop tape on the second half of the lanes so that episodes actually terminate
        e2 = gym.make_vec(env_id, num_envs=n, vectorization_mode="sync", **kw)
        o, _ = e2.reset(seed=seed, options=options)
        for t in range(T):
            a = actions[t]
            a[n // 2:] = policy(o[n // 2:]).astype(a.dtype).reshape(a[n // 2:].shape)
            o, *_ = e2.step(a)
        e2.close()
    out = rollout(envs, seed, actions, options=options, state_attr=state_attr)
    out["max_episode_steps"] = np.int64(kw.get("max_episode_steps", envs.envs[0].spec.max_episode_steps))
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")}, "term", out["terminated"].sum(), "trunc",
          out["truncated"].sum(), "reward %.3f" % out["reward"].sum())


def tabular(name, env_id, n, T, seed, nA, policy="random", **kw):
    envs = gym.make_vec(env_id, num_envs=n, vectorization_mode="sync", **kw)
    rng = np.random.default_rng(3000 + seed)
    actions = rng.integers(0, nA, size=(T, n)).astype(np.int64)
    if policy == "pickup":  # Taxi: pick the passenger up / drop him whenever the action mask allows it, so that rides happen
        _, info = envs.reset(seed=seed)
        for t in range(T):
            m = info["action_mask"]
            actions[t] = np.where(m[:, 4] == 1, 4, np.where((m[:, 5] == 1) & (rng.random(n) < 0.3), 5, actions[t]))
            _, _, _, _, info = envs.step(actions[t])
    out = rollout(envs, seed, actions)
    mes = envs.envs[0].spec.max_episode_steps
    out["max_episode_steps"] = np.int64(kw.get("max_episode_steps", mes if mes is not None else 0))
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items() if hasattr(v, "shape")}, "term", out["terminated"].sum(), "trunc",
          out["truncated"].sum(), "reward", out["reward"].sum())


def blackjack(name, n, T, seed, mode=AutoresetMode.NEXT_STEP, **kw):
    """Blackjack-v1: the observation is a Tuple of three Discrete spaces, batched by SyncVectorEnv into a tuple of three
    (n,) int64 arrays (vector/utils/space_utils.py:120-131); stored here stacked as (T+1, n, 3)."""
    envs = gym.make_vec("Blackjack-v1", num_envs=n, vectorization_mode="sync", vector_kwargs={"autoreset_mode": mode}, **kw)
    rng = np.random.default_rng(5000 + seed)
    actions = rng.integers(0, 2, size=(T, n)).astype(np.int64)
    o, _ = envs.reset(seed=seed)
    assert isinstance(o, tuple) and len(o) == 3 and o[0].dtype == np.int64
    obs = np.zeros((T + 1, n, 3), np.int64)
    obs[0] = np.stack(o, axis=1)
    rew, term, trunc = np.zeros((T, n)), np.zeros((T, n), bool), np.zeros((T, n), bool)
    final = np.full((T, n, 3), -1, np.int64)
    for t in range(T):
        o, r, te, tr, info = envs.step(actions[t])
        obs[t + 1], rew[t], term[t], trunc[t] = np.stack(o, axis=1), r, te, tr
        if "final_obs" in info:
            for i in np.flatnonzero(info["_final_obs"]):
                final[t, i] = np.asarray(info["final_obs"][i])
    out = dict(seed=np.uint64(seed), actions=actions, obs=obs, reward=rew, terminated=term, truncated=trunc, final_obs=final,
               natural=np.int64(kw.get("natural", False)), sab=np.int64(kw.get("sab", True)), mode=np.str_(mode.value),
               max_episode_steps=np.int64(0))
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.shape}, "term", term.sum(), "reward",
          rew.sum(), "rewards seen", sorted(set(rew.ravel().tolist())))


def cartpole_beyond(name, n, T, seed):
    """Single reference CartPoleEnvs (TimeLimit far away) stepped PAST termination without a reset: reward 1.0 on the
    terminating step, 0.0 afterwards (cartpole.py:205-220).  SyncVectorEnv refuses to do this (sync_vector_env.py asserts in
    DISABLED mode), so the tape comes from `gym.make` envs seeded seed+i like its sub-envs would be."""
    import warnings

    warnings.filterwarnings("ignore")
    envs = [gym.make("CartPole-v1", max_episode_steps=10 * T) for _ in range(n)]
    obs0 = np.stack([e.reset(seed=seed + i)[0] for i, e in enumerate(envs)])
    rs = np.random.default_rng(seed)
    actions = (rs.random((T, n)) < 0.85).astype(np.int64)  # mostly push right: falls after ~10 steps
    obs = np.zeros((T + 1, n, 4), np.float32)
    obs[0] = obs0
    rew, term = np.zeros((T, n), np.float64), np.zeros((T, n), bool)
    for t in range(T):
        for i, e in enumerate(envs):
            o, r, te, _tr, _ = e.step(int(actions[t, i]))
            obs[t + 1, i], rew[t, i], term[t, i] = o, r, te
    np.savez_compressed(os.path.join(HERE, name), obs=obs, rew=rew, term=term, actions=actions, seed=np.int64(seed))
    print(name, "term", term.sum(), "zero rewards", int((rew == 0).sum()))


def dropin(name, env_id, n, T, seed, nA, spaces=False, **kw):
    """The stock sync vectoriser's outputs and output dtypes on a seeded action tape, with its spaces if asked
    (tests/test_gpu_dropin.py)."""
    envs = gym.make_vec(env_id, num_envs=n, vectorization_mode="sync", **kw)
    actions = np.random.default_rng(6000 + seed).integers(0, nA, size=(T, n)).astype(np.int64)
    o, _ = envs.reset(seed=seed)
    obs = [o]
    rew, term, trunc = [], [], []
    for t in range(T):
        o, r, te, tr, _ = envs.step(actions[t])
        obs.append(o); rew.append(r); term.append(te); trunc.append(tr)
    out = dict(seed=np.int64(seed), actions=actions, obs=np.stack(obs), reward=np.stack(rew), terminated=np.stack(term),
               truncated=np.stack(trunc), step_dtypes=np.array([str(r.dtype), str(te.dtype), str(tr.dtype)]))
    for tag, sp in (("obs_space", envs.observation_space), ("single_obs_space", envs.single_observation_space),
                    ("action_space", envs.action_space)) if spaces else ():
        if isinstance(sp, gym.spaces.Box):
            out.update({tag + "_low": sp.low, tag + "_high": sp.high})
        else:
            out.update({tag + "_nvec": sp.nvec, tag + "_start": sp.start})
        out[tag + "_dtype"] = np.array(str(sp.dtype))
    envs.close()
    np.savez_compressed(os.path.join(HERE, name), **out)
    print(name, {k: v.shape for k, v in out.items()}, "term", out["terminated"].sum(), "reward", out["reward"].sum())


if __name__ == "__main__":
    assert "reference" in gym.__file__ or "_ref" in gym.__file__, gym.__file__
    print("reference:", gym.__version__, gym.__file__, "numpy", np.__version__)
    if len(sys.argv) > 1 and sys.argv[1] == "dropin":  # regenerate only the drop-in fixtures
        dropin("dropin_cartpole_n5_s123_T150.npz", "CartPole-v1", 5, 150, 123, 2, spaces=True)
        dropin("dropin_frozenlake8x8_n6_s5_T200.npz", "FrozenLake-v1", 6, 200, 5, 4, map_name="8x8")
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "cartpole_beyond":
        cartpole_beyond("beyond_cartpole_n4_s5.npz", 4, 40, 5)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "blackjack":  # regenerate only the Blackjack fixtures
        blackjack("blackjack_sab_n32_s11.npz", 32, 400, 11)
        blackjack("blackjack_natural_n32_s12.npz", 32, 400, 12, natural=True, sab=False)
        blackjack("blackjack_plain_n17_s13.npz", 17, 300, 13, natural=False, sab=False)
        blackjack("blackjack_samestep_n16_s14.npz", 16, 300, 14, mode=AutoresetMode.SAME_STEP)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "taxi_rainy":  # regenerate only the rainy-Taxi fixture
        tabular("taxi_rainy_n16_s6_T400.npz", "Taxi-v4", 16, 400, 6, 6, is_rainy=True)
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "taxi_fickle":  # regenerate only the fickle-passenger fixtures
        tabular("taxi_fickle_n24_s7_T600.npz", "Taxi-v4", 24, 600, 7, 6, policy="pickup", fickle_passenger=True)
        tabular("taxi_fickle_rainy_n24_s8_T600.npz", "Taxi-v4", 24, 600, 8, 6, policy="pickup", fickle_passenger=True,
                is_rainy=True)
        sys.exit(0)
    cartpole("cartpole_n8_s42_T300.npz", 8, 300, 42)
    cartpole("cartpole_n16_s7_T400_limit60_balance.npz", 16, 400, 7, max_episode_steps=60, policy="balance")
    cartpole("cartpole_n4_s123_bounds.npz", 4, 60, 123, options={"low": -0.1, "high": 0.1})
    cartpole("cartpole_n4_s5_sutton.npz", 4, 120, 5, sutton_barto_reward=True)
    cartpole("cartpole_n6_s11_samestep.npz", 6, 200, 11, max_episode_steps=40, policy="balance", mode=AutoresetMode.SAME_STEP)
    cartpole("cartpole_n3_s2p40.npz", 3, 50, 2**40 + 12345)
    frozenlake("frozenlake8x8_n16_s0_T400.npz", 16, 400, 0, map_name="8x8")
    frozenlake("frozenlake4x4_n8_s3_T300.npz", 8, 300, 3)
    frozenlake("frozenlake8x8_n8_s9_noslip.npz", 8, 150, 9, map_name="8x8", is_slippery=False)
    frozenlake("frozenlake8x8_n8_s21_limit25.npz", 8, 200, 21, map_name="8x8", max_episode_steps=25)
    frozenlake("frozenlake8x8_n6_s4_samestep.npz", 6, 300, 4, map_name="8x8", mode=AutoresetMode.SAME_STEP)
    # round-1 additions: DISABLED mode with caller-driven partial resets, odd batch sizes, custom map / probabilities /
    # reward schedule, a two-start-tile map (non-trivial initial-state distribution), near-2^64 seeds
    cartpole("cartpole_n5_s9_disabled.npz", 5, 160, 9, max_episode_steps=30, policy="balance", mode=AutoresetMode.DISABLED)
    cartpole("cartpole_n1_s77.npz", 1, 120, 77)
    cartpole("cartpole_n33_s3_limit20.npz", 33, 90, 3, max_episode_steps=20)
    cartpole("cartpole_n2_s2p64m9.npz", 2, 40, 2**64 - 9)
    frozenlake("frozenlake8x8_n7_s6_disabled.npz", 7, 260, 6, map_name="8x8", mode=AutoresetMode.DISABLED)
    tabular("cliffwalking_n8_s1_T400.npz", "CliffWalking-v1", 8, 400, 1, 4)
    tabular("cliffwalking_n8_s2_limit50.npz", "CliffWalking-v1", 8, 300, 2, 4, max_episode_steps=50)
    tabular("cliffwalkingslippery_n8_s3_T400.npz", "CliffWalkingSlippery-v1", 8, 400, 3, 4)
    tabular("taxi_n12_s4_T500.npz", "Taxi-v4", 12, 500, 4, 6)
    tabular("taxi_n6_s5_limit30.npz", "Taxi-v4", 6, 200, 5, 6, max_episode_steps=30)
    classic("mountaincar_n8_s1_T500.npz", "MountainCar-v0", 8, 500, 1, nA=3, policy=lambda o: np.where(o[:, 1] > 0, 2, 0))
    classic("mountaincar_n4_s2_bounds.npz", "MountainCar-v0", 4, 120, 2, nA=3, options={"low": -0.7, "high": -0.3},
            max_episode_steps=40)
    classic("mountaincarcontinuous_n8_s3_T400.npz", "MountainCarContinuous-v0", 8, 400, 3, act_scale=1.0,
            max_episode_steps=150, policy=lambda o: np.where(o[:, 1] > 0, 1.0, -1.0))
    classic("pendulum_n8_s4_T450.npz", "Pendulum-v1", 8, 450, 4, act_scale=2.0)
    classic("pendulum_n4_s5_init.npz", "Pendulum-v1", 4, 90, 5, act_scale=2.0, options={"x_init": 1.0, "y_init": 0.5},
            max_episode_steps=30)
    classic("acrobot_n8_s6_T600.npz", "Acrobot-v1", 8, 600, 6, nA=3, policy=lambda o: np.where(o[:, 5] > 0, 2, 0))
    classic("acrobot_n4_s7_limit50.npz", "Acrobot-v1", 4, 200, 7, nA=3, max_episode_steps=50)
    frozenlake("frozenlakecustom_n9_s8_p80.npz", 9, 220, 8, desc=["SFFHF", "FHFFF", "FFSFH", "HFFFG"], map_name=None,
               success_rate=0.8, reward_schedule=(10, -5, -1), max_episode_steps=40)
