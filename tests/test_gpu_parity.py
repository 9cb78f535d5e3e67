"""GPU parity tests (pytest -m gpu): the CUDA path, called through the C-ABI / B200VectorEnv, against
(1) golden fixtures from the live reference, (2) the numpy oracle on seeded inputs, (3) size-independent properties at
BASELINE.json's full sizes.  Tolerances: integer/bool/RNG bit-exact; CartPole float32 observations rtol=atol=1e-5
(the reference's own `data_equivalence`, gymnasium/utils/env_checker.py:34-75)."""
import ctypes as C

import numpy as np
import pytest

from conftest import (check_reset_obs, fixture_kwargs, fixture_options, golden, golden_files, have_cuda,
                      replay_fixture)

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_cuda(), reason="needs a CUDA device")]

RTOL = ATOL = 1e-5


def make(env_id, n, **kw):
    import gymnasium_b200

    kw.setdefault("output", "numpy")
    return gymnasium_b200.make_vec(env_id, num_envs=n, **kw)


def replay(env, seed, actions, options=None):
    obs, info = env.reset(seed=seed, options=options)
    out = dict(obs=[obs], reward=[], terminated=[], truncated=[], info=[info])
    for a in actions:
        o, r, te, tr, info = env.step(a)
        out["obs"].append(o); out["reward"].append(r); out["terminated"].append(te); out["truncated"].append(tr)
        out["info"].append(info)
    return {k: (np.stack(v) if k != "info" else v) for k, v in out.items()}


# ---------------------------------------------------------------------------------------------------------------------
# RNG
@pytest.mark.parametrize("base", [0, 42, 2**32 - 2, 2**40 + 12345, 2**63 + 11])
def test_rng_streams_bit_exact_with_numpy(base):
    import torch
    from gymnasium_b200 import _lib

    lib = _lib.load()
    n, k = 257, 9
    b = _lib.Batch(n=n, env_offset=3)
    rng = torch.zeros((2, n, 2), dtype=torch.int64, device="cuda")
    out = torch.zeros((n, k), dtype=torch.float64, device="cuda")
    _lib.check(lib.b2e_rng_seed(C.byref(b), base, None, None, rng.data_ptr(), None))
    state = rng.cpu().numpy().view(np.uint64)
    _lib.check(lib.b2e_rng_random(C.byref(b), rng.data_ptr(), k, out.data_ptr(), None))
    got = out.cpu().numpy()
    for i in [0, 1, 2, 100, 256]:
        g = np.random.Generator(np.random.PCG64(np.random.SeedSequence(base + 3 + i)))
        st = g.bit_generator.state["state"]
        assert int(state[0, i, 0]) | (int(state[0, i, 1]) << 64) == st["state"]
        assert int(state[1, i, 0]) | (int(state[1, i, 1]) << 64) == st["inc"]
        np.testing.assert_array_equal(got[i], g.random(k))
    # explicit seed list + mask
    seeds = np.array([7, 2**64 - 1, 5, 2**33], dtype=np.uint64)
    b = _lib.Batch(n=4)
    rng = torch.zeros((2, 4, 2), dtype=torch.int64, device="cuda")
    mask = torch.tensor([1, 1, 0, 1], dtype=torch.uint8, device="cuda")
    sd = torch.from_numpy(seeds.view(np.int64)).cuda()
    _lib.check(lib.b2e_rng_seed(C.byref(b), 0, sd.data_ptr(), mask.data_ptr(), rng.data_ptr(), None))
    out = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    st_before = rng.clone()
    _lib.check(lib.b2e_rng_random(C.byref(b), rng.data_ptr(), 3, out.data_ptr(), None))
    for i in [0, 1, 3]:
        g = np.random.Generator(np.random.PCG64(np.random.SeedSequence(int(seeds[i]))))
        np.testing.assert_array_equal(out[i].cpu().numpy(), g.random(3))
    assert (st_before[:, 2] == 0).all()  # masked-out lane untouched by seeding


def test_fast_math_paths_match_ieee_division_and_libdevice():
    """div_total_mass (reciprocal + 2 residual FMAs) must equal IEEE division bit for bit; the short sin/cos kernels must
    stay within 1 ulp of libdevice on the whole non-terminated angle range (2^28 samples each)."""
    import torch
    from gymnasium_b200 import _lib

    lib = _lib.load()
    counts = torch.zeros(3, dtype=torch.int64, device="cuda")
    n = 1 << 28
    for seed in (1, 2):
        _lib.check(lib.b2e_selftest_math(n, seed, counts.data_ptr(), None))
    c = counts.cpu().tolist()
    assert c[0] == 0, f"{c[0]} constant-division results differ from __ddiv_rn"
    assert c[1] == 0, f"{c[1]} sin/cos results are more than 1 ulp from libdevice"
    assert c[2] < 0.25 * 2 * n, c  # 1-ulp disagreements with libdevice are the minority


# ---------------------------------------------------------------------------------------------------------------------
# CartPole
@pytest.mark.parametrize("name", golden_files("cartpole"))
def test_cartpole_matches_reference_golden(name):
    g = golden(name)
    n = g["actions"].shape[1]
    env = make("CartPole-v1", n, max_episode_steps=int(g["max_episode_steps"]), **fixture_kwargs(name))
    out = replay_fixture(env, g, fixture_options(name), disabled="disabled" in name)
    check_reset_obs(out, g)  # reset draws are exact fp64 RNG math
    np.testing.assert_array_equal(out["obs"][0], g["obs"][0])  # reset draws: exact fp64 RNG math
    np.testing.assert_array_equal(out["terminated"], g["terminated"])
    np.testing.assert_array_equal(out["truncated"], g["truncated"])
    np.testing.assert_array_equal(out["reward"], g["reward"])
    assert out["reward"].dtype == np.float64 and out["obs"].dtype == np.float32
    np.testing.assert_allclose(out["obs"], g["obs"], rtol=RTOL, atol=ATOL)
    # in practice far tighter than the contract: sin/cos are the only non-identical ops
    assert np.max(np.abs(out["obs"].astype(np.float64) - g["obs"])) < 1e-6


def test_cartpole_state_fp64_vs_reference():
    g = golden("cartpole_n8_s42_T300.npz")
    env = make("CartPole-v1", 8)
    env.reset(seed=42)
    np.testing.assert_array_equal(env.state.cpu().numpy(), g["state"][0])
    worst = 0.0
    for t, a in enumerate(g["actions"]):
        env.step(a)
        worst = max(worst, np.max(np.abs(env.state.cpu().numpy() - g["state"][t + 1])))
    assert worst < 1e-11, worst


@pytest.mark.parametrize("rng_dtype", [np.int64, np.int32, np.uint8])
def test_cartpole_vs_oracle_4096(rng_dtype):
    from oracle.cartpole import OracleCartPole

    n, T, seed = 4096, 260, 1234
    acts = np.random.default_rng(5).integers(0, 2, size=(T, n)).astype(rng_dtype)
    env = make("CartPole-v1", n, max_episode_steps=100)
    ora = OracleCartPole(n, max_episode_steps=100)
    o1, _ = env.reset(seed=seed)
    o2, _ = ora.reset(seed=seed)
    np.testing.assert_array_equal(o1, o2)
    n_done = n_trunc = 0
    for t in range(T):
        a1 = env.step(acts[t])
        a2 = ora.step(acts[t].astype(np.int64))
        np.testing.assert_allclose(a1[0], a2[0], rtol=RTOL, atol=ATOL)
        for k in (1, 2, 3):
            np.testing.assert_array_equal(a1[k], a2[k])
        n_done += a2[2].sum(); n_trunc += a2[3].sum()
    assert n_done > n and n_trunc > 0  # every lane reset at least once on average; the time limit was exercised


def test_cartpole_rollout_equals_step_loop_full_size():
    """Property at BASELINE size (N=65536): K fused steps == K step() calls, bit for bit (same device arithmetic)."""
    import torch

    n, K = 65536, 64
    acts = torch.randint(0, 2, (K, n), dtype=torch.int64, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    a = make("CartPole-v1", n, output="torch")
    b = make("CartPole-v1", n, output="torch")
    a.reset(seed=99); b.reset(seed=99)
    traj = a.rollout(K, actions=acts)
    for k in range(K):
        o, r, te, tr, _ = b.step(acts[k])
        assert torch.equal(o, traj["obs"][k]) and torch.equal(te, traj["terminated"][k])
        assert torch.equal(tr, traj["truncated"][k]) and torch.equal(r.float(), traj["reward"][k])
    assert torch.equal(a.state, b.state) and torch.equal(a._ctrl, b._ctrl) and torch.equal(a._rng, b._rng)
    done = traj["terminated"] | traj["truncated"]
    assert 0.03 < done.float().mean().item() < 0.06  # ~1/22.8 of random-action steps end an episode (SURVEY 8d)
    # rows after a done are resets: reward 0 and |obs| <= 0.05
    after = done[:-1]
    assert (traj["reward"][1:][after] == 0).all() and (traj["obs"][1:][after].abs() <= 0.05).all()


def test_cartpole_sharding_is_invariant():
    """Shards with env_offset reproduce the matching slice of one big batch (seeds are global: seed + offset + i)."""
    n, T = 1024, 40
    acts = np.random.default_rng(3).integers(0, 2, size=(T, n))
    whole = make("CartPole-v1", n)
    parts = [make("CartPole-v1", n // 4, env_offset=r * (n // 4)) for r in range(4)]
    ow, _ = whole.reset(seed=17)
    op = np.concatenate([p.reset(seed=17)[0] for p in parts])
    np.testing.assert_array_equal(ow, op)
    for t in range(T):
        w = whole.step(acts[t])
        ps = [p.step(acts[t, r * (n // 4):(r + 1) * (n // 4)]) for r, p in enumerate(parts)]
        for k in range(4):
            np.testing.assert_array_equal(w[k], np.concatenate([x[k] for x in ps]))


def test_cartpole_random_rollout_philox_statistics():
    import torch

    n, K = 65536, 200
    env = make("CartPole-v1", n, output="torch", rng="philox")
    env.reset(seed=5)
    traj = env.rollout(K, return_actions=True)
    assert abs(traj["actions"].float().mean().item() - 0.5) < 0.002
    done = (traj["terminated"] | traj["truncated"])
    ep_len = (K * n) / max(done.sum().item(), 1)
    assert 20.0 < ep_len < 26.0, ep_len  # mean random-policy episode ~22.8 steps + 1 reset call
    env2 = make("CartPole-v1", n, output="torch", rng="philox")
    env2.reset(seed=5)
    t2 = env2.rollout(K, return_actions=True)
    assert all(torch.equal(traj[k], t2[k]) for k in traj)  # deterministic


# ---------------------------------------------------------------------------------------------------------------------
# FrozenLake
@pytest.mark.parametrize("name", golden_files("frozenlake"))
def test_frozenlake_matches_reference_golden_bit_exact(name):
    g = golden(name)
    n = g["actions"].shape[1]
    env = make("FrozenLake-v1", n, max_episode_steps=int(g["max_episode_steps"]), **fixture_kwargs(name))
    out = replay_fixture(env, g, disabled="disabled" in name)
    check_reset_obs(out, g)
    assert out["obs"].dtype == np.int64
    np.testing.assert_array_equal(out["obs"], g["obs"])
    np.testing.assert_array_equal(out["reward"], g["reward"])
    np.testing.assert_array_equal(out["terminated"], g["terminated"])
    np.testing.assert_array_equal(out["truncated"], g["truncated"])
    for t, info in enumerate(out["info"][1:]):
        ref = g["info_prob"][t]
        assert ((ref == info["prob"]) | (ref == np.floor(info["prob"]))).all()  # SURVEY App. C #6
        np.testing.assert_array_equal(info["_prob"], g["info__prob"][t])


def test_frozenlake_vs_oracle_2048():
    from oracle.frozenlake import OracleFrozenLake

    n, T, seed = 2048, 230, 77
    acts = np.random.default_rng(8).integers(0, 4, size=(T, n))
    env = make("FrozenLake-v1", n, map_name="8x8", max_episode_steps=100)
    ora = OracleFrozenLake(n, map_name="8x8", max_episode_steps=100)
    np.testing.assert_array_equal(env.reset(seed=seed)[0], ora.reset(seed=seed)[0])
    for t in range(T):
        a1, a2 = env.step(acts[t]), ora.step(acts[t])
        for k in range(4):
            np.testing.assert_array_equal(a1[k], a2[k])
        np.testing.assert_array_equal(a1[4]["prob"], a2[4]["prob"])


def test_frozenlake_rollout_equals_step_loop_full_size():
    """Property at BASELINE size (N=1,048,576, 8x8): fused rollout == step loop bit-exact; states stay on the map."""
    import torch

    n, K = 1 << 20, 24
    acts = torch.randint(0, 4, (K, n), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    a = make("FrozenLake-v1", n, map_name="8x8", output="torch", copy=False)
    b = make("FrozenLake-v1", n, map_name="8x8", output="torch", copy=False)
    a.reset(seed=3); b.reset(seed=3)
    traj = a.rollout(K, actions=acts)
    for k in range(K):
        o, r, te, tr, info = b.step(acts[k])
        assert torch.equal(o, traj["obs"][k]) and torch.equal(te, traj["terminated"][k])
        assert torch.equal(tr, traj["truncated"][k]) and torch.equal(r.float(), traj["reward"][k])
    assert torch.equal(a._pstate, b._pstate) and torch.equal(a._rng, b._rng) and torch.equal(a._ctrl, b._ctrl)
    assert int(traj["obs"].min()) >= 0 and int(traj["obs"].max()) < 64
    holes = torch.tensor([19, 29, 35, 41, 42, 46, 49, 52, 54, 59], device="cuda")
    term_obs = traj["obs"][traj["terminated"]]
    assert torch.isin(term_obs, torch.cat([holes, torch.tensor([63], device="cuda")])).all()
    assert (traj["reward"][traj["terminated"] & (traj["obs"] == 63)] == 1).all()


def test_frozenlake_numpy_stream_consumption():
    """One draw per call on every path: after T calls env i's PCG64 state equals numpy's after T+1 draws."""
    n, T = 64, 37
    env = make("FrozenLake-v1", n, map_name="8x8")
    env.reset(seed=1000)
    for t in range(T):
        env.step(np.full(n, t % 4))
    st = env.rng_state()
    for i in [0, 5, 63]:
        g = np.random.Generator(np.random.PCG64(np.random.SeedSequence(1000 + i)))
        g.random(T + 1)
        assert int(st[0, i, 0]) | (int(st[0, i, 1]) << 64) == g.bit_generator.state["state"]["state"]


# ---------------------------------------------------------------------------------------------------------------------
# API behaviour shared with SyncVectorEnv
def test_api_errors_and_reset_mask():
    import torch
    from gymnasium_b200 import errors

    env = make("CartPole-v1", 3)
    with pytest.raises(errors.ResetNeeded):
        env.step([0, 1, 0])
    env.reset(seed=0)
    with pytest.raises(ValueError):
        env.step([0, 1])
    with pytest.raises(TypeError):
        env.step(1)
    with pytest.raises(TypeError):
        env.reset(options={"reset_mask": [True, False, False]})
    with pytest.raises(ValueError):
        env.reset(options={"reset_mask": np.array([True, False])})
    with pytest.raises(TypeError):
        env.reset(options={"reset_mask": np.array([1, 0, 0])})
    with pytest.raises(ValueError):
        env.reset(options={"reset_mask": np.zeros(3, dtype=bool)})
    with pytest.raises(ValueError):
        env.reset(seed=[1, 2])
    assert env.np_random_seed == (0, 1, 2)
    assert env.metadata["autoreset_mode"].value == "NextStep"
    assert env.observation_space.shape == (3, 4) and env.action_space.shape == (3,)
    # partial reset (DISABLED mode workflow, tests/vector/test_autoreset_mode.py:105-260)
    from oracle.cartpole import OracleCartPole

    env = make("CartPole-v1", 4, autoreset_mode="Disabled", max_episode_steps=15)
    ora = OracleCartPole(4, max_episode_steps=15, autoreset_mode="Disabled")
    np.testing.assert_array_equal(env.reset(seed=11)[0], ora.reset(seed=11)[0])
    rs = np.random.default_rng(0)
    for t in range(80):
        a = rs.integers(0, 2, 4)
        x, y = env.step(a), ora.step(a)
        np.testing.assert_allclose(x[0], y[0], rtol=RTOL, atol=ATOL)
        for k in (1, 2, 3):
            np.testing.assert_array_equal(x[k], y[k])
        done = y[2] | y[3]
        if done.any():
            o1, _ = env.reset(options={"reset_mask": done.copy()})
            o2, _ = ora.reset(options={"reset_mask": done.copy()})
            np.testing.assert_allclose(o1, o2, rtol=RTOL, atol=ATOL)
    env.close()
    assert env.closed


@pytest.mark.gpu
def test_cartpole_reward_on_steps_beyond_termination_matches_reference():
    """Autoreset DISABLED, lanes stepped past termination without a reset (the reference's vector layer asserts instead; the
    env itself keeps stepping): reward 1.0 on the terminating step, 0.0 afterwards (cartpole.py:205-220) -- fixture recorded
    from single reference envs."""
    g = golden("beyond_cartpole_n4_s5.npz")
    n = g["actions"].shape[1]
    env = make("CartPole-v1", n, autoreset_mode="Disabled", max_episode_steps=10_000)
    np.testing.assert_allclose(env.reset(seed=int(g["seed"]))[0], g["obs"][0], rtol=RTOL, atol=ATOL)
    for t, a in enumerate(g["actions"]):
        obs, rew, term, trunc, _ = env.step(a)
        np.testing.assert_array_equal(rew, g["rew"][t], err_msg=f"step {t}")
        np.testing.assert_array_equal(term, g["term"][t])
        np.testing.assert_allclose(obs, g["obs"][t + 1], rtol=1e-4, atol=1e-4)
        assert not trunc.any()
    # a masked reset clears the flag: the next termination pays 1.0 again
    env.reset(options={"reset_mask": np.ones(n, dtype=bool)})
    for _ in range(40):
        obs, rew, term, trunc, _ = env.step(np.ones(n, dtype=np.int64))
        if term.any():
            break
    assert term.any() and (rew[term] == 1.0).all()


def test_validate_actions_mode_raises_like_the_reference():
    env = make("CartPole-v1", 4, validate_actions=True)
    env.reset(seed=0)
    env.step(np.array([0, 1, 1, 0]))
    with pytest.raises(AssertionError, match="invalid"):  # cartpole.py:165-167, tests/envs/test_action_dim_check.py:59-86
        env.step(np.array([0, 1, 2, 0]))
    lenient = make("CartPole-v1", 4)
    lenient.reset(seed=0)
    lenient.step(np.array([0, 1, 7, -3]))  # default: clamped in-kernel, no host sync


def test_torch_outputs_and_devices():
    import torch

    env = make("CartPole-v1", 8, output="torch")
    obs, info = env.reset(seed=1)
    assert obs.is_cuda and obs.dtype == torch.float32 and info == {}
    o, r, te, tr, info = env.step(torch.ones(8, dtype=torch.int64, device="cuda"))
    assert o.is_cuda and r.dtype == torch.float64 and te.dtype == torch.bool and tr.dtype == torch.bool
    o2, *_ = env.step(np.zeros(8, dtype=np.int64))
    assert o2.data_ptr() != o.data_ptr()  # copy=True hands out fresh tensors, like SyncVectorEnv(copy=True)
    fl = make("FrozenLake-v1", 8, map_name="8x8", output="torch")
    obs, info = fl.reset(seed=1)
    assert obs.dtype == torch.int64 and info["prob"].dtype == torch.float64 and bool(info["_prob"].all())


# ---------------------------------------------------------------------------------------------------------------------
# LunarLander-v3: the checker is oracle/lunar_lander.c (Box2D-subset restatement, parity with the real wheel unpinned)
def test_lunarlander_matches_oracle_bit_exact_random_policy():
    from oracle.lunar_lander import OracleLunarLander

    n, T, seed = 512, 400, 2024
    env = make("LunarLander-v3", n)
    ora = OracleLunarLander(n)
    o1, _ = env.reset(seed=seed)
    o2, _ = ora.reset(seed=seed)
    np.testing.assert_array_equal(o1, o2)
    rs = np.random.default_rng(4)
    n_term = 0
    for t in range(T):
        a = rs.integers(0, 4, n)
        x, y = env.step(a), ora.step(a)
        np.testing.assert_array_equal(x[0], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2], y[2])
        np.testing.assert_array_equal(x[3], y[3])
        n_term += int(y[2].sum())
    assert n_term > n  # every lane crashed (and was auto-reset) more than once on average
    assert not env.contact_overflow()


def test_lunarlander_heuristic_landing_on_gpu():
    """The reference's behavioural pin (tests/envs/test_env_implementation.py:12-16) driven through the engine, and
    bit-for-bit agreement with the oracle while legs rest on the ground (contacts, block solver, sleep)."""
    from oracle.lunar_lander import OracleLunarLander, heuristic

    seeds = [1, 0, 2, 3, 7, 11, 42, 5]
    n = len(seeds)
    env = make("LunarLander-v3", n)
    ora = OracleLunarLander(n)
    o1, _ = env.reset(seed=seeds)
    o2, _ = ora.reset(seed=seeds)
    np.testing.assert_array_equal(o1, o2)
    total = np.zeros(n)
    alive = np.ones(n, dtype=bool)
    for t in range(1000):
        a = np.array([heuristic(o) for o in o1])
        o1, r1, te1, tr1, _ = env.step(a)
        o2, r2, te2, tr2, _ = ora.step(a)
        np.testing.assert_array_equal(o1[alive], o2[alive], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(r1[alive], r2[alive])
        np.testing.assert_array_equal(te1, te2)
        total[alive] += r1[alive]
        alive &= ~(te1 | tr1)
        if not alive.any():
            break
    assert total[0] > 100, total  # seed=1, the reference test
    assert (total > 0).all(), total


def test_lunarlander_api():
    import torch

    env = make("LunarLander-v3", 6, output="torch")
    obs, info = env.reset(seed=3)
    assert obs.shape == (6, 8) and obs.dtype == torch.float32 and info == {}
    assert env.observation_space.shape == (6, 8) and env.action_space.shape == (6,)
    o, r, te, tr, _ = env.step(torch.zeros(6, dtype=torch.int64, device="cuda"))
    assert r.dtype == torch.float64 and te.dtype == torch.bool
    cont = make("LunarLander-v3", 2, continuous=True)  # lunar_lander.py:298-305
    assert cont.single_action_space.shape == (2,) and cont.action_space.shape == (2, 2)
    with pytest.raises(AssertionError):  # lunar_lander.py:232-234
        make("LunarLander-v3", 2, gravity=-13.0)
    # determinism + sharding invariance
    a = make("LunarLander-v3", 64)
    b = [make("LunarLander-v3", 32, env_offset=0), make("LunarLander-v3", 32, env_offset=32)]
    oa, _ = a.reset(seed=77)
    ob = np.concatenate([e.reset(seed=77)[0] for e in b])
    np.testing.assert_array_equal(oa, ob)
    rs = np.random.default_rng(1)
    for _ in range(120):
        act = rs.integers(0, 4, 64)
        xa = a.step(act)
        xb = [b[0].step(act[:32]), b[1].step(act[32:])]
        for k in range(4):
            np.testing.assert_array_equal(xa[k], np.concatenate([xb[0][k], xb[1][k]]))


# ---------------------------------------------------------------------------------------------------------------------
# Humanoid-v5: the checker is oracle/humanoid.c (MuJoCo-subset restatement, parity with the real wheel unpinned)
@pytest.mark.parametrize("impl", ["thread", "warp"])
def test_humanoid_matches_oracle_bit_exact(impl):
    from oracle.humanoid import OracleHumanoid

    n, T, seed = 48, 90, 31
    env = make("Humanoid-v5", n, impl=impl)
    ora = OracleHumanoid(n)
    o1, i1 = env.reset(seed=seed)
    o2, i2 = ora.reset(seed=seed)
    assert o1.shape == (n, 348) and o1.dtype == np.float64
    np.testing.assert_array_equal(o1, o2)
    np.testing.assert_array_equal(i1["x_position"], i2["x_position"])
    rs = np.random.default_rng(9)
    n_term = 0
    for t in range(T):
        a = rs.uniform(-0.4, 0.4, size=(n, 17)).astype(np.float32)
        x, y = env.step(a), ora.step(a)
        np.testing.assert_array_equal(x[0], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2], y[2])
        np.testing.assert_array_equal(x[3], y[3])
        for k in ("x_velocity", "y_velocity", "reward_survive", "reward_forward", "reward_ctrl", "reward_contact",
                  "distance_from_origin"):
            np.testing.assert_array_equal(x[4][k], y[4][k], err_msg=k)
        np.testing.assert_array_equal(x[4]["tendon_length"][:, 0], y[4]["tendon_length0"])
        np.testing.assert_array_equal(x[4]["tendon_velocity"][:, 1], y[4]["tendon_velocity1"])
        n_term += int(y[2].sum())
    assert n_term >= n // 2  # random actions make the humanoid fall within ~40-80 steps
    assert not env.buffer_overflow()


@pytest.mark.parametrize("mode", ["NextStep", "SameStep"])
def test_humanoid_warp_and_thread_mappings_agree(mode):
    """The two kernel mappings of the same physics must agree bit for bit, including through autoresets.  The warp mapping
    regroups envs into CTAs by the solver work of their last step (the thread mapping does not), so this also shows that
    the grouping is scheduling only; `order` must be a permutation of the env indices."""
    n, T = 1000, 70
    kw = dict(autoreset_mode=mode, max_episode_steps=40)
    a_env, b_env = make("Humanoid-v5", n, impl="thread", **kw), make("Humanoid-v5", n, impl="warp", **kw)
    o1, _ = a_env.reset(seed=5)
    o2, _ = b_env.reset(seed=5)
    np.testing.assert_array_equal(o1, o2)
    rs = np.random.default_rng(3)
    for t in range(T):
        a = rs.uniform(-0.4, 0.4, size=(n, 17)).astype(np.float32)
        x, y = a_env.step(a), b_env.step(a)
        for k in range(4):
            np.testing.assert_array_equal(x[k], y[k], err_msg=f"output {k} differs at step {t}")
        for k in x[4]:
            if isinstance(x[4][k], np.ndarray) and x[4][k].dtype != object:
                np.testing.assert_array_equal(x[4][k], y[4][k], err_msg=k)
    assert not a_env.buffer_overflow() and not b_env.buffer_overflow()
    order = b_env._s["order"].cpu().numpy()
    assert sorted(order.tolist()) == list(range(n))
    work = b_env._s["work"].cpu().numpy()
    assert (work >= -1).all() and work.max() > 0


def test_humanoid_reference_structural_pins_on_gpu():
    """The reference's own checks for this boundary (tests/envs/mujoco/test_mujoco_v5.py), through the engine."""
    import torch

    env = make("Humanoid-v5", 4, reset_noise_scale=0.0)
    obs, info = env.reset(seed=0)
    np.testing.assert_array_equal(obs[:, 0], 1.4)              # z of the noise-free init state (:693-710)
    assert set(info) >= {"x_position", "y_position", "tendon_length", "tendon_velocity", "distance_from_origin"}  # :454-476
    assert env.single_observation_space.shape == (348,) and env.single_action_space.shape == (17,)
    rs = np.random.default_rng(2)
    terminated_at = None
    for step in range(80):                                        # test_verify_reward_survive (:159-191)
        a = rs.uniform(-0.4, 0.4, size=(4, 17)).astype(np.float32)
        obs, r, te, tr, info = env.step(a)
        total = (info["reward_forward"] + info["reward_survive"]) + (info["reward_ctrl"] + info["reward_contact"])
        assert (r == total).all()                                  # exact, the reference's grouping (:248-254)
        if te[0]:
            assert info["reward_survive"][0] == 0 and not (1.0 < obs[0, 0] < 2.0)
            terminated_at = step
            break
        assert info["reward_survive"][0] == 5.0
    assert terminated_at is not None
    with pytest.raises(ValueError, match="Action dimension mismatch"):
        env.step(np.zeros((4, 16), dtype=np.float32))
    t = make("Humanoid-v5", 2, output="torch")
    o, _ = t.reset(seed=1)
    assert o.dtype == torch.float64 and o.shape == (2, 348)


# ---------------------------------------------------------------------------------------------------------------------
# CliffWalking-v1 / Taxi-v4 through the generic tabular kernel (pinned to the live reference)
@pytest.mark.parametrize("name", golden_files("cliffwalking") + golden_files("taxi"))
def test_toy_text_matches_reference_golden_bit_exact(name):
    g = golden(name)
    n = g["actions"].shape[1]
    mes = int(g["max_episode_steps"]) or None
    if name.startswith("taxi"):
        env = make("Taxi-v4", n, max_episode_steps=mes, is_rainy="rainy" in name, fickle_passenger="fickle" in name)
    else:
        env = make("CliffWalkingSlippery-v1" if "slippery" in name else "CliffWalking-v1", n, max_episode_steps=mes)
    out = replay_fixture(env, g)
    np.testing.assert_array_equal(out["obs"], g["obs"])
    np.testing.assert_array_equal(out["reward"], g["reward"])
    np.testing.assert_array_equal(out["terminated"], g["terminated"])
    np.testing.assert_array_equal(out["truncated"], g["truncated"])
    for t, info in enumerate(out["info"][1:]):
        ref = g["info_prob"][t]
        assert ((ref == info["prob"]) | (ref == np.floor(info["prob"]))).all()
        if name.startswith("taxi"):
            np.testing.assert_array_equal(info["action_mask"], g["info_action_mask"][t])
            assert info["action_mask"].dtype == np.int8


# ---------------------------------------------------------------------------------------------------------------------
# MountainCar-v0 / MountainCarContinuous-v0 / Pendulum-v1 / Acrobot-v1 (csrc/classic.cu), pinned to the live reference
CLASSIC = {"mountaincar_": "MountainCar-v0", "mountaincarcontinuous_": "MountainCarContinuous-v0",
           "pendulum_": "Pendulum-v1", "acrobot_": "Acrobot-v1"}


@pytest.mark.parametrize("name", sum((golden_files(p) for p in CLASSIC), []))
def test_classic_control_matches_reference_golden(name):
    import torch

    g = golden(name)
    env_id = next(v for k, v in CLASSIC.items() if name.startswith(k))
    n = g["actions"].shape[1]
    options = {"low": -0.7, "high": -0.3} if "bounds" in name else {"x_init": 1.0, "y_init": 0.5} if "init" in name else None
    chaotic_long = name.startswith("acrobot") and g["actions"].shape[0] > 300
    if not chaotic_long:  # free-running replay of the whole tape
        env = make(env_id, n, max_episode_steps=int(g["max_episode_steps"]))
        out = replay_fixture(env, g, options)
        np.testing.assert_array_equal(out["terminated"], g["terminated"])
        np.testing.assert_array_equal(out["truncated"], g["truncated"])
        assert out["obs"].dtype == np.float32 and out["reward"].dtype == np.float64
        np.testing.assert_allclose(out["obs"], g["obs"], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(out["reward"], g["reward"], rtol=RTOL, atol=ATOL)
        assert float(np.max(np.abs(out["obs"].astype(np.float64) - g["obs"]))) < 2e-6
    # step-wise ("teacher-forced") check of the one-step map: start every call from the reference's own float64 state, so
    # chaotic families (Acrobot is a double pendulum) cannot amplify last-ulp sin/cos differences over hundreds of steps
    env = make(env_id, n, max_episode_steps=int(g["max_episode_steps"]))
    obs, _ = env.reset(seed=int(g["seed"]), options=options)
    np.testing.assert_allclose(obs, g["obs"][0], rtol=0, atol=1e-7)
    worst_state = worst_obs = 0.0
    for t, a in enumerate(g["actions"]):
        env.set_state(g["state"][t])
        o, r, te, tr, _ = env.step(a)
        np.testing.assert_array_equal(te, g["terminated"][t])
        np.testing.assert_array_equal(tr, g["truncated"][t])
        worst_obs = max(worst_obs, float(np.max(np.abs(o.astype(np.float64) - g["obs"][t + 1]))))
        worst_state = max(worst_state, float(np.max(np.abs(env.state.cpu().numpy() - g["state"][t + 1]))))
        # 1e-9: the reference squares float32 torques with powf (pendulum.py:137), which is not always u*u to the last ulp
        np.testing.assert_allclose(r, g["reward"][t], rtol=1e-9, atol=1e-9)
    assert worst_obs < 5e-7 and worst_state < 1e-12, (worst_obs, worst_state)


def test_wrappers_run_on_device_without_host_sync():
    """RecordEpisodeStatistics + NormalizeObservation + NormalizeReward stacked on the engine, all tensors on the GPU;
    episode returns agree with an independent accumulation of the raw rewards."""
    import torch
    from gymnasium_b200 import wrappers as W

    n = 4096
    raw = make("CartPole-v1", n, output="torch")
    env = W.NormalizeReward(W.NormalizeObservation(W.RecordEpisodeStatistics(make("CartPole-v1", n, output="torch"))))
    o_raw, _ = raw.reset(seed=3)
    o, _ = env.reset(seed=3)
    assert o.is_cuda and o.dtype == torch.float32
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    prev = torch.zeros(n, dtype=torch.bool, device="cuda")
    gen = torch.Generator("cuda").manual_seed(0)
    total_done = 0
    for t in range(120):
        a = torch.randint(0, 2, (n,), device="cuda", generator=gen)
        _, r_raw, te_raw, tr_raw, _ = raw.step(a)
        o, r, te, tr, info = env.step(a)
        assert torch.equal(te, te_raw) and torch.equal(tr, tr_raw) and r.is_cuda
        ret = torch.where(prev, torch.zeros_like(ret), ret + r_raw)
        done = te | tr
        assert torch.equal(info["_episode"], done)
        assert torch.equal(info["episode"]["r"][done], ret[done])
        prev = done
        total_done += int(done.sum())
    assert abs(float(o.mean())) < 0.2 and 0.5 < float(o.std()) < 1.5
    assert env.env.env.episode_count == total_done and total_done > n


def test_dict_info_to_list_and_numpy_to_torch_on_the_engine():
    """§8f rank 1: DictInfoToList over FrozenLake's masked `prob` info and Humanoid's 11 info keys; NumpyToTorch turns an
    output="numpy" engine env into a torch one without a host round trip."""
    import torch
    from gymnasium_b200 import wrappers as W

    n = 64
    raw = make("FrozenLake-v1", n, map_name="8x8")
    env = W.DictInfoToList(make("FrozenLake-v1", n, map_name="8x8", output="torch"))
    (_, i0), (_, l0) = raw.reset(seed=1), env.reset(seed=1)
    assert isinstance(l0, list) and len(l0) == n and all(d["prob"] == 1 for d in l0)
    rs = np.random.default_rng(0)
    for t in range(40):
        a = rs.integers(0, 4, n)
        info, lst = raw.step(a)[4], env.step(a)[4]
        for i in range(n):
            assert ("prob" in lst[i]) == bool(info["_prob"][i])
            if info["_prob"][i]:
                assert lst[i]["prob"] == info["prob"][i]
    h = W.DictInfoToList(make("Humanoid-v5", 3))
    _, li = h.reset(seed=0)
    assert set(li[0]) >= {"x_position", "tendon_length"} and li[2]["tendon_length"].shape == (2,)
    t = W.NumpyToTorch(make("CartPole-v1", 16, output="numpy"))
    o, _ = t.reset(seed=0)
    o2, r, te, tr, _ = t.step(torch.zeros(16, dtype=torch.int64))
    assert o.is_cuda and o2.is_cuda and r.dtype == torch.float64 and te.dtype == torch.bool
    ref = make("CartPole-v1", 16)
    ref.reset(seed=0)
    np.testing.assert_array_equal(ref.step(np.zeros(16, dtype=np.int64))[0], o2.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# Blackjack-v1 (SURVEY §8f rank 3): Tuple observation, Generator.choice draws on PCG64's buffered 32-bit words
@pytest.mark.parametrize("name", golden_files("blackjack"))
def test_blackjack_matches_reference_golden_bit_exact(name):
    g = golden(name)
    n = g["actions"].shape[1]
    env = make("Blackjack-v1", n, natural=bool(g["natural"]), sab=bool(g["sab"]), autoreset_mode=str(g["mode"]))
    obs, info = env.reset(seed=int(g["seed"]))
    assert isinstance(obs, tuple) and len(obs) == 3 and obs[0].dtype == np.int64 and info == {}
    np.testing.assert_array_equal(np.stack(obs, axis=1), g["obs"][0])
    for t, a in enumerate(g["actions"]):
        o, r, te, tr, info = env.step(a)
        np.testing.assert_array_equal(np.stack(o, axis=1), g["obs"][t + 1], err_msg=f"obs at step {t}")
        np.testing.assert_array_equal(r, g["reward"][t])
        np.testing.assert_array_equal(te, g["terminated"][t])
        assert not tr.any()
        if str(g["mode"]) == "SameStep":
            done = te | tr
            np.testing.assert_array_equal(info["_final_obs"], done)
            np.testing.assert_array_equal(np.stack(info["final_obs"], axis=1)[done], g["final_obs"][t][done])


def test_blackjack_reseeding_and_reset_mask():
    """Re-seeding an env empties its 32-bit word buffer (a fresh numpy Generator has none); unmasked tables keep theirs."""
    n = 8
    env, ref = make("Blackjack-v1", n, sab=True), make("Blackjack-v1", n, sab=True)
    env.reset(seed=5)
    for t in range(7):
        env.step(np.ones(n, dtype=np.int64))          # leaves odd/even buffer states behind
    o1, _ = env.reset(seed=5)
    o2, _ = ref.reset(seed=5)
    for a, b in zip(o1, o2):
        np.testing.assert_array_equal(a, b)
    mask = np.array([True, False] * 4)
    seeds = [100 + i if m else None for i, m in enumerate(mask)]
    before = [x.copy() for x in o1]
    o3, _ = env.reset(seed=seeds, options={"reset_mask": mask})
    fresh, _ = make("Blackjack-v1", n, sab=True).reset(seed=[100 + i for i in range(n)])
    for k in range(3):
        np.testing.assert_array_equal(o3[k][mask], fresh[k][mask])
        np.testing.assert_array_equal(o3[k][~mask], before[k][~mask])
    assert env.single_observation_space.contains((int(o3[0][0]), int(o3[1][0]), int(o3[2][0])))


def test_async_call_api_and_attr_access():
    """AsyncVectorEnv's split calls (async_vector_env.py:310-521) and SyncVectorEnv.call/get_attr/set_attr
    (sync_vector_env.py:343-398) on the engine: same results as reset()/step(), same exception types and messages."""
    from gymnasium_b200 import errors

    for output in ("numpy", "torch"):
        a, b = make("CartPole-v1", 9, output=output), make("CartPole-v1", 9, output=output)
        with pytest.raises(errors.NoAsyncCallError, match="without any prior call to `reset_async`"):
            a.reset_wait()
        a.reset_async(seed=4)
        with pytest.raises(errors.AlreadyPendingCallError, match="pending call to `reset`"):
            a.step_async(np.zeros(9, dtype=np.int64))
        o1, i1 = a.reset_wait()
        o2, i2 = b.reset(seed=4)
        as_np = (lambda x: x.cpu().numpy()) if output == "torch" else (lambda x: x)
        np.testing.assert_array_equal(as_np(o1), as_np(o2))
        rs = np.random.default_rng(1)
        for t in range(40):
            act = rs.integers(0, 2, 9)
            a.step_async(act)
            with pytest.raises(errors.AlreadyPendingCallError, match="pending call to `step`"):
                a.reset_async()
            x, y = a.step_wait(), b.step(act)
            for k in range(4):
                np.testing.assert_array_equal(as_np(x[k]), as_np(y[k]))
        with pytest.raises(errors.NoAsyncCallError, match="without any prior call to `step_async`"):
            a.step_wait()
    bj = make("Blackjack-v1", 5)
    bj.reset_async(seed=2)
    o, _ = bj.reset_wait()
    assert isinstance(o, tuple) and len(o) == 3 and isinstance(o[0], np.ndarray)
    bj.step_async(np.ones(5, dtype=np.int64))
    assert isinstance(bj.step_wait()[0], tuple)
    fl = make("FrozenLake-v1", 4, map_name="8x8")
    mask = np.array([True, False, True, False])
    fl.reset(seed=0)
    fl.reset_async(seed=[7, None, 8, None], options={"reset_mask": mask})
    _, info = fl.reset_wait()
    np.testing.assert_array_equal(info["_prob"], mask)
    # attribute access
    h = make("Humanoid-v5", 3)
    assert h.get_attr("frame_skip") == (5, 5, 5) and h.call("elapsed_steps").shape == (3,)
    cp = make("CartPole-v1", 3)
    with pytest.raises(ValueError, match="same value for every sub-environment"):
        cp.set_attr("max_episode_steps", [1, 2, 3])
    with pytest.raises(ValueError, match="length equal to the number of environments"):
        cp.set_attr("max_episode_steps", [1, 2])
    cp.close()
    with pytest.raises(errors.ClosedEnvironmentError):
        cp.reset(seed=0)


@pytest.mark.gpu
def test_first_reset_with_mask_seeds_every_lane_and_np_random_seed_tracks_masked_reseeds():
    """A first reset() that carries a reset_mask must not leave the other lanes on all-zero PCG64 words (their autoresets
    would all draw u = 0.0), and np_random_seed must follow masked int / list re-seeds lane by lane."""
    mask = np.array([True, False, True, False, False, True])
    env = make("CartPole-v1", 6)
    env.reset(seed=100, options={"reset_mask": mask})
    words = env.rng_state()  # [2][n][2]
    assert (words[0].any(axis=1)).all() and (words[1].any(axis=1)).all()
    assert env.np_random_seed == tuple(100 + i for i in range(6))
    # masked lanes follow numpy exactly
    for i in np.nonzero(mask)[0]:
        st = np.random.PCG64(np.random.SeedSequence(100 + int(i))).state["state"]
        # four uniform draws were taken by the reset: advance the reference stream the same way
        g = np.random.Generator(np.random.PCG64(np.random.SeedSequence(100 + int(i))))
        g.uniform(-0.05, 0.05, size=4)
        s = g.bit_generator.state["state"]["state"]
        assert int(words[0][i][0]) | (int(words[0][i][1]) << 64) == s and st is not None
    env.reset(seed=500, options={"reset_mask": np.array([False, True, False, False, False, False])})
    assert env.np_random_seed == (100, 501, 102, 103, 104, 105)
    env.reset(seed=[1, 2, 3, 4, 5, 6], options={"reset_mask": np.array([False, False, False, True, False, False])})
    assert env.np_random_seed == (100, 501, 102, 4, 104, 105)
    # seed=None on a never-seeded batch with a mask: every lane still gets a (lazy) stream
    env2 = make("CartPole-v1", 6)
    env2.reset(options={"reset_mask": mask})
    w2 = env2.rng_state()
    assert (w2[0].any(axis=1)).all() and (w2[1].any(axis=1)).all()


@pytest.mark.gpu
def test_np_random_snapshots_continue_the_device_streams():
    """SyncVectorEnv.np_random (sync_vector_env.py:182-185): the Generators handed out reproduce the draws the env makes next."""
    env = make("CartPole-v1", 5)
    env.reset(seed=40)
    gens = env.np_random
    assert len(gens) == 5 and all(isinstance(g, np.random.Generator) for g in gens)
    for i, g in enumerate(gens):
        ref = np.random.Generator(np.random.PCG64(np.random.SeedSequence(40 + i)))
        ref.uniform(-0.05, 0.05, size=4)  # the reset's draws
        assert g.random() == ref.random()
    nxt = [g.uniform(-0.05, 0.05, size=4) for g in env.np_random]  # what the next reset of every lane will draw
    obs, _ = env.reset()
    np.testing.assert_array_equal(obs, np.asarray(nxt, dtype=np.float64).astype(np.float32))


@pytest.mark.gpu
def test_humanoid_observation_flags_select_columns():
    """include_*_in_observation / exclude_current_positions_from_observation (humanoid_v5.py:281-300, :436-470)."""
    full = make("Humanoid-v5", 6)
    o_full, i_full = full.reset(seed=9)
    a = np.random.default_rng(0).uniform(-0.4, 0.4, size=(3, 6, 17)).astype(np.float32)
    small = make("Humanoid-v5", 6, include_cinert_in_observation=False, include_cfrc_ext_in_observation=False)
    xy = make("Humanoid-v5", 6, exclude_current_positions_from_observation=False, include_cvel_in_observation=False,
              include_qfrc_actuator_in_observation=False)
    o_small, _ = small.reset(seed=9)
    o_xy, _ = xy.reset(seed=9)
    assert small.single_observation_space.shape == (348 - 130 - 78,) and xy.single_observation_space.shape == (348 - 78 - 17 + 2,)
    assert small.observation_structure["cinert"] == 0 and xy.observation_structure["skipped_qpos"] == 0

    def check(of, info, os_, ox):
        np.testing.assert_array_equal(os_, np.concatenate([of[:, :45], of[:, 175:270]], axis=1))
        np.testing.assert_array_equal(ox[:, 0], info["x_position"])
        np.testing.assert_array_equal(ox[:, 1], info["y_position"])
        np.testing.assert_array_equal(ox[:, 2:], np.concatenate([of[:, :175], of[:, 270:]], axis=1))

    check(o_full, i_full, o_small, o_xy)
    for t in range(3):
        of, rf, _, _, info = full.step(a[t])
        os_, rs_, _, _, _ = small.step(a[t])
        ox, rx, _, _, _ = xy.step(a[t])
        check(of, info, os_, ox)
        np.testing.assert_array_equal(rf, rs_)
        np.testing.assert_array_equal(rf, rx)
    t_env = make("Humanoid-v5", 4, include_cinert_in_observation=False, output="torch")
    o, _ = t_env.reset(seed=1)
    assert tuple(o.shape) == (4, 218) and o.is_cuda
