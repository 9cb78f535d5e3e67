"""Parity hardening for the two physics families whose third-party engines (Box2D, MuJoCo) cannot be installed here.

* config-size runs: LunarLander-v3 at BASELINE's N=16384 and Humanoid-v5 at N=8192 on the GPU, with a sampled set of 256
  GLOBAL env indices checked bit for bit against the C oracle (envs are independent: the oracle gets those indices as a seed
  list), through at least one autoreset per family;
* sharding invariance of Humanoid (env_offset), which the 8-GPU configuration depends on;
* analytic known-answer tests that do NOT depend on the repo's own oracle: closed forms of the engines' integrators in free
  flight (total-momentum balance), the numpy RNG draw order of reset(), zero actuation for zero control;
* the reference's own reward identity with its exact grouping and `==` (tests/envs/mujoco/test_mujoco_v5.py:248-254).
"""
import numpy as np
import pytest

import gymnasium_b200

pytestmark = pytest.mark.gpu


def make(env_id, n, **kw):
    kw.setdefault("output", "numpy")
    return gymnasium_b200.make_vec(env_id, num_envs=n, **kw)


# ---------------------------------------------------------------------------------------------------------------------
def test_lunarlander_config_size_sampled_lanes_match_oracle():
    """BASELINE configs[3]: 16384 envs.  256 sampled global indices vs oracle/lunar_lander.c, bit-exact, through autoresets."""
    from oracle.lunar_lander import OracleLunarLander

    n, T, seed = 16384, 320, 77
    rs = np.random.default_rng(10)
    idx = np.sort(rs.choice(n, size=256, replace=False))
    idx[0], idx[-1] = 0, n - 1
    env = make("LunarLander-v3", n)
    ora = OracleLunarLander(len(idx))
    o1, _ = env.reset(seed=seed)
    o2, _ = ora.reset(seed=[seed + int(i) for i in idx])
    np.testing.assert_array_equal(o1[idx], o2)
    resets = np.zeros(len(idx), dtype=np.int64)
    for t in range(T):
        a = rs.integers(0, 4, n)
        x, y = env.step(a), ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2][idx], y[2])
        np.testing.assert_array_equal(x[3][idx], y[3])
        resets += y[2] | y[3]
    assert (resets >= 1).mean() > 0.95 and resets.sum() > len(idx)  # (almost) every sampled lane went through an autoreset
    assert not env.contact_overflow()


@pytest.mark.parametrize("continuous,wind,n,T", [(True, True, 2048, 230), (True, False, 512, 200), (False, True, 512, 200)])
def test_lunarlander_continuous_and_wind_match_oracle_bit_exact(continuous, wind, n, T):
    """LunarLander(continuous=..., enable_wind=...) (lunar_lander.py:476-616, :401-403) against oracle/lunar_lander.c: throttled
    engines, fuel costs, the wind / turbulence pattern with its np_random.integers offsets, across autoresets."""
    from oracle.lunar_lander import OracleLunarLander

    seed = 41
    rs = np.random.default_rng(6)
    idx = np.arange(n) if n <= 512 else np.sort(rs.choice(n, size=256, replace=False))
    kw = dict(continuous=continuous, enable_wind=wind, wind_power=12.0, turbulence_power=1.0)
    env = make("LunarLander-v3", n, **kw)
    ora = OracleLunarLander(len(idx), **kw)
    o1, _ = env.reset(seed=seed)
    o2, _ = ora.reset(seed=[seed + int(i) for i in idx])
    np.testing.assert_array_equal(o1[idx], o2)
    if continuous:
        assert env.single_action_space.shape == (2,) and env.single_action_space.dtype == np.float32
    if wind:
        np.testing.assert_array_equal(env.wind_state().cpu().numpy()[idx], [ora.wind_state(i) for i in range(len(idx))])
    resets = np.zeros(len(idx), dtype=np.int64)
    for t in range(T):
        a = rs.uniform(-1.3, 1.3, size=(n, 2)).astype(np.float32) if continuous else rs.integers(0, 4, n)
        x, y = env.step(a), ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2][idx], y[2])
        np.testing.assert_array_equal(x[3][idx], y[3])
        resets += y[2] | y[3]
    assert (resets >= 1).mean() > 0.9  # the wind pattern was re-drawn and the 32-bit buffer carried across resets
    if wind:
        np.testing.assert_array_equal(env.wind_state().cpu().numpy()[idx], [ora.wind_state(i) for i in range(len(idx))])
    assert not env.contact_overflow()
    # a masked re-seed starts those lanes' streams (and their 32-bit buffers) afresh
    mask = np.zeros(n, dtype=bool)
    mask[idx[: len(idx) // 2]] = True
    o3, _ = env.reset(seed=seed + 1000, options={"reset_mask": mask})
    sub = np.zeros(len(idx), dtype=bool)
    sub[: len(idx) // 2] = True
    o4, _ = ora.reset(seed=[seed + 1000 + int(i) for i in idx], options={"reset_mask": sub})
    np.testing.assert_array_equal(o3[idx][sub], o4[sub])
    for t in range(30):
        a = rs.uniform(-1.3, 1.3, size=(n, 2)).astype(np.float32) if continuous else rs.integers(0, 4, n)
        x, y = env.step(a), ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t} after the masked re-seed")
        np.testing.assert_array_equal(x[1][idx], y[1])


def test_lunarlander_continuous_id_and_float64_actions():
    env = make("LunarLanderContinuous-v3", 64)
    assert env.continuous and env.single_action_space.shape == (2,)
    ref = make("LunarLander-v3", 64, continuous=True)
    np.testing.assert_array_equal(env.reset(seed=2)[0], ref.reset(seed=2)[0])
    rs = np.random.default_rng(0)
    for _ in range(40):
        a = rs.uniform(-1, 1, size=(64, 2)).astype(np.float32)
        x, y = env.step(a.astype(np.float64)), ref.step(a)  # float32-representable float64 actions: identical run
        for k in range(4):
            np.testing.assert_array_equal(x[k], y[k])
    with pytest.raises(ValueError):
        env.step(np.zeros(64, dtype=np.int64))


def test_humanoid_config_size_sampled_lanes_match_oracle():
    """BASELINE configs[4]: 8192 envs per GPU.  256 sampled global indices vs oracle/humanoid.c, bit-exact, through autoresets."""
    from oracle.humanoid import OracleHumanoid

    n, T, seed = 8192, 110, 5
    rs = np.random.default_rng(12)
    idx = np.sort(rs.choice(n, size=256, replace=False))
    idx[0], idx[-1] = 0, n - 1
    env = make("Humanoid-v5", n)
    ora = OracleHumanoid(len(idx))
    o1, _ = env.reset(seed=seed)
    o2, _ = ora.reset(seed=[seed + int(i) for i in idx])
    np.testing.assert_array_equal(o1[idx], o2)
    resets = np.zeros(len(idx), dtype=np.int64)
    for t in range(T):
        a = rs.uniform(-0.4, 0.4, size=(n, 17)).astype(np.float32)
        x, y = env.step(a), ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2][idx], y[2])
        np.testing.assert_array_equal(x[3][idx], y[3])
        for k in ("x_velocity", "reward_forward", "reward_contact"):
            np.testing.assert_array_equal(x[4][k][idx], y[4][k], err_msg=k)
        resets += y[2] | y[3]
    assert (resets >= 1).mean() > 0.9  # random actions make the humanoid fall within ~40-80 steps: autoresets were crossed
    assert not env.buffer_overflow()


def test_humanoid_sharding_is_invariant():
    """One 96-env batch == shards of 40 + 56 envs with env_offset (seeds use the GLOBAL env index), through autoresets."""
    whole = make("Humanoid-v5", 96, max_episode_steps=25)
    parts = [make("Humanoid-v5", 40, env_offset=0, max_episode_steps=25), make("Humanoid-v5", 56, env_offset=40, max_episode_steps=25)]
    ow, iw = whole.reset(seed=123)
    op = [p.reset(seed=123) for p in parts]
    np.testing.assert_array_equal(ow, np.concatenate([o for o, _ in op]))
    np.testing.assert_array_equal(iw["x_position"], np.concatenate([i["x_position"] for _, i in op]))
    rs = np.random.default_rng(8)
    for t in range(60):
        a = rs.uniform(-0.4, 0.4, size=(96, 17)).astype(np.float32)
        xw = whole.step(a)
        xp = [parts[0].step(a[:40]), parts[1].step(a[40:])]
        for k in range(4):
            np.testing.assert_array_equal(xw[k], np.concatenate([xp[0][k], xp[1][k]]), err_msg=f"output {k} at step {t}")
        for key in ("x_velocity", "reward_ctrl", "distance_from_origin"):
            np.testing.assert_array_equal(xw[4][key], np.concatenate([xp[0][4][key], xp[1][4][key]]))


# ---------------------------------------------------------------------------------------------------------------------
# analytic known answers (independent of oracle/*.c)
def _humanoid_momentum(obs):
    """Total linear momentum per unit mass from the observation alone: cinert rows carry (.., m*(xipos - com), m) and cvel rows
    the spatial velocity at the subtree COM, so a body's COM velocity is v + w x (xipos - com) (humanoid_v5.py:436-470)."""
    cin = obs[:, 45:175].reshape(-1, 13, 10)
    cvel = obs[:, 175:253].reshape(-1, 13, 6)
    m = cin[:, :, 9]
    off = cin[:, :, 6:9] / m[:, :, None]
    v = cvel[:, :, 3:6] + np.cross(cvel[:, :, 0:3], off)
    return (m[:, :, None] * v).sum(axis=1) / m.sum(axis=1)[:, None], m


def test_humanoid_free_fall_known_answer():
    """Noise-free reset, zero control: until the first contact the only external force is gravity, so the mass centre obeys
    v_com(t) = (0, 0, -9.81 t) whatever the limbs do (RK4 is exact for constant acceleration).  The stock model's joint
    armature (1.0, humanoid.xml:4) is rotor inertia outside the body masses, which limits the identity to ~1e-7; an error in
    kinematics, composite inertia, the factorisation, the bias forces or the integrator shows up at 1e-2.  Zero control must
    give exactly zero actuator forces (gear * ctrl), and the body masses must be the stock model's (mjModel.body_mass)."""
    n = 8
    env = make("Humanoid-v5", n, reset_noise_scale=0.0)
    obs, _ = env.reset(seed=0)
    np.testing.assert_array_equal(obs[:, 0], 1.4)
    act = np.zeros((n, 17), dtype=np.float32)
    free = 0
    for k in range(12):
        obs, r, te, tr, info = env.step(act)
        if np.abs(obs[:, 270:348]).max() > 0:  # cfrc_ext: the first contact has happened
            break
        t = (k + 1) * 5 * 0.003  # frame_skip 5 x timestep 0.003 (humanoid.xml:8, humanoid_v5.py:268)
        p, m = _humanoid_momentum(obs)
        np.testing.assert_allclose(p[:, 2], -9.81 * t, rtol=0, atol=2e-6)
        np.testing.assert_allclose(p[:, :2], 0.0, rtol=0, atol=1e-7)
        np.testing.assert_array_equal(obs[:, 253:270], 0.0)            # qfrc_actuator[6:] with zero ctrl
        np.testing.assert_array_equal(info["reward_ctrl"], 0.0)
        np.testing.assert_allclose(info["x_velocity"], 0.0, atol=1e-7)  # the COM does not move sideways in free fall
        assert (info["reward_survive"] == 5.0).all() and not te.any()
        free += 1
    assert free >= 8, f"only {free} free-fall steps before the first contact"
    # well-known mjModel.body_mass of the stock humanoid.xml (inertiafromgeom): torso 8.907, lwaist 2.262, pelvis 6.616, ...
    known = [8.90746237, 2.26194671, 6.61619413, 4.75175093, 2.75569617, 1.76714587, 4.75175093, 2.75569617, 1.76714587,
             1.66108048, 1.22954019, 1.66108048, 1.22954019]
    np.testing.assert_allclose(m[0], known, rtol=1e-7)


def test_lunarlander_free_flight_known_answer():
    """reset() then no-op steps: before any contact the only external forces on (lander + 2 legs) are gravity and the initial
    random force on the lander, applied during the world.Step embedded in reset() (lunar_lander.py:393-399, :447).  Box2D's
    semi-implicit Euler then gives the total momentum in closed form, P_k = h F + M h g (k + 1), with F read from numpy's own
    stream in the reference's draw order (12 terrain heights, then fx, fy).  Checked from the engine's body states; masses
    from the shoelace areas of the fixtures (density 5 / 1)."""
    n, seed = 64, 2024
    env = make("LunarLander-v3", n)
    obs, _ = env.reset(seed=seed)
    h, g = 1.0 / 50.0, -10.0
    poly = np.array([(-14, 17), (-17, 0), (-17, -10), (17, -10), (17, 0), (14, 17)], dtype=np.float64) / 30.0
    x, y = poly[:, 0], poly[:, 1]
    area = 0.5 * abs(np.dot(x, np.roll(y, -1)) - np.dot(y, np.roll(x, -1)))
    m_lander, m_leg = 5.0 * area, 1.0 * (2 * 2 / 30.0) * (2 * 8 / 30.0)
    M = m_lander + 2 * m_leg
    F = np.zeros((n, 2))
    for i in range(n):
        gen = np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed + i)))
        gen.uniform(0, 400 / 30.0 / 2, size=(12,))       # terrain heights (lunar_lander.py:344)
        F[i] = [gen.uniform(-1000.0, 1000.0), gen.uniform(-1000.0, 1000.0)]
    masses = np.array([m_lander, m_leg, m_leg])

    def momentum():
        b = env.body_state().cpu().numpy().astype(np.float64)  # (n, 3, 7): c.x c.y angle v.x v.y w sleep
        return (masses[None, :, None] * b[:, :, 3:5]).sum(axis=1)

    p = momentum()
    np.testing.assert_allclose(p[:, 0], h * F[:, 0], rtol=2e-5, atol=2e-4)
    np.testing.assert_allclose(p[:, 1], h * F[:, 1] + M * h * g, rtol=2e-5, atol=2e-4)
    # the observation's velocity entries are the lander's (vel * (W/2 or H/2) / FPS, lunar_lander.py:627-628); right after
    # reset the legs have barely pulled on it
    b = env.body_state().cpu().numpy()
    np.testing.assert_allclose(obs[:, 2], b[:, 0, 3] * (600 / 30.0 / 2) / 50, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(obs[:, 3], b[:, 0, 4] * (400 / 30.0 / 2) / 50, rtol=1e-6, atol=1e-7)
    a = np.zeros(n, dtype=np.int64)
    for k in range(1, 25):  # the lander starts at the top of the viewport: ~1 s of flight before anything can touch
        o, r, te, tr, _ = env.step(a)
        assert not te.any() and (o[:, 6:8] == 0).all()
        p = momentum()
        np.testing.assert_allclose(p[:, 0], h * F[:, 0], rtol=5e-5, atol=5e-4, err_msg=f"step {k}")
        np.testing.assert_allclose(p[:, 1], h * F[:, 1] + M * h * g * (k + 1), rtol=5e-5, atol=5e-4, err_msg=f"step {k}")


def test_humanoid_reward_identity_is_exact_with_the_reference_grouping():
    """tests/envs/mujoco/test_mujoco_v5.py:248-254 asserts `reward == (forward + survive) + (ctrl + contact)` with ==."""
    env = make("Humanoid-v5", 256)
    env.reset(seed=3)
    rs = np.random.default_rng(2)
    for _ in range(100):
        a = rs.uniform(-0.4, 0.4, size=(256, 17)).astype(np.float32)
        _, reward, te, tr, info = env.step(a)
        live = ~(info["reward_survive"] == 0) | te  # autoreset calls return reward 0 and zeroed terms: identity holds too
        total = (info["reward_forward"] + info["reward_survive"]) + (info["reward_ctrl"] + info["reward_contact"])
        assert (reward == total).all(), np.abs(reward - total).max()
        assert live.any()


@pytest.mark.parametrize("output", ["numpy", "torch"])
def test_humanoid_info_masks_follow_syncvectorenv(output):
    """NEXT_STEP: the call after a done is that lane's reset() -- SyncVectorEnv merges only the 5 reset-info keys for it, so
    the masks of the 6 step-only keys are False there (vector_env.py:277-338 `_add_info`); SAME_STEP: lanes that end an
    episode report their reset info as well."""
    env = gymnasium_b200.make_vec("Humanoid-v5", num_envs=32, max_episode_steps=4, output=output)
    env.reset(seed=0)
    a = np.zeros((32, 17), dtype=np.float32)
    prev = np.zeros(32, dtype=bool)
    for t in range(11):
        _, _, te, tr, info = env.step(a)
        te, tr = np.asarray(te.cpu() if output == "torch" else te), np.asarray(tr.cpu() if output == "torch" else tr)
        for k in ("x_position", "tendon_length", "distance_from_origin"):
            assert bool(np.asarray(info["_" + k].cpu() if output == "torch" else info["_" + k]).all())
        for k in ("x_velocity", "reward_survive", "reward_contact"):
            m = np.asarray(info["_" + k].cpu() if output == "torch" else info["_" + k])
            np.testing.assert_array_equal(m, ~prev, err_msg=f"{k} at step {t}")
        prev = te | tr
    assert prev.any() or t > 4
    same = gymnasium_b200.make_vec("Humanoid-v5", num_envs=8, max_episode_steps=3, autoreset_mode="SameStep", output="numpy")
    same.reset(seed=0)
    for t in range(4):
        _, _, te, tr, info = same.step(a[:8])
        np.testing.assert_array_equal(info["_reward_forward"], ~(te | tr))
        np.testing.assert_array_equal(info["_final_obs"], te | tr)


# ---------------------------------------------------------------------------------------------------------------------
# Hopper-v5 (SURVEY 8f rank 4: the Humanoid solver generalised to another MuJoCo robot); checker = oracle/hopper.c
@pytest.mark.parametrize("robot", ["Hopper-v5", "Walker2d-v5"])
@pytest.mark.parametrize("n,T,dtype", [(512, 130, np.float32), (8192, 70, np.float32), (64, 60, np.float64)])
def test_planar_robots_match_oracle_bit_exact(robot, n, T, dtype):
    from oracle.hopper import OracleHopper
    from oracle.walker2d import OracleWalker2d

    Oracle, nu, nobs = (OracleHopper, 3, 11) if robot == "Hopper-v5" else (OracleWalker2d, 6, 17)
    seed = 21
    rs = np.random.default_rng(3)
    idx = np.arange(n) if n <= 512 else np.sort(rs.choice(n, size=256, replace=False))
    env = make(robot, n)
    ora = Oracle(len(idx))
    o1, i1 = env.reset(seed=seed)
    o2, i2 = ora.reset(seed=[seed + int(i) for i in idx])
    assert o1.shape == (n, nobs) and o1.dtype == np.float64
    np.testing.assert_array_equal(o1[idx], o2)
    np.testing.assert_array_equal(i1["z_distance_from_origin"][idx], i2["z_distance_from_origin"])
    resets = np.zeros(len(idx), dtype=np.int64)
    for t in range(T):
        a = rs.uniform(-1.0, 1.0, size=(n, nu)).astype(dtype)
        x = env.step(a)
        if dtype == np.float64:  # the oracle's control cost is the float32 one; compare everything but reward_ctrl / reward
            y = ora.step(a[idx].astype(np.float32))
            if (a[idx].astype(np.float32).astype(np.float64) != a[idx]).any():
                np.testing.assert_array_equal(x[2][idx], y[2])
                break  # float64 actions that are not float32-representable drive a (slightly) different trajectory
        else:
            y = ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2][idx], y[2])
        np.testing.assert_array_equal(x[3][idx], y[3])
        for k in ("x_position", "x_velocity", "reward_forward", "reward_ctrl", "reward_survive"):
            np.testing.assert_array_equal(x[4][k][idx], y[4][k], err_msg=k)
        total = x[4]["reward_forward"] + x[4]["reward_survive"] + x[4]["reward_ctrl"]
        assert (x[1] == total).all()  # tests/envs/mujoco/test_mujoco_v5.py:236-241, exact
        resets += y[2] | y[3]
    if dtype == np.float32:
        assert (resets >= 1).mean() > 0.9  # random policies fall within ~25 steps: autoresets were crossed
    assert not env.buffer_overflow()


@pytest.mark.parametrize("n,T,dtype", [(512, 160, np.float32), (16384, 60, np.float32), (64, 40, np.float64)])
def test_inverted_pendulum_matches_oracle_bit_exact(n, T, dtype):
    """InvertedPendulum-v5 on the planar kernels against oracle/inverted_pendulum.c (itself pinned to the cart-pole equations
    of motion, tests/test_oracle_hopper.py): observations, rewards, flags and reward_survive, across autoresets."""
    from oracle.inverted_pendulum import OracleInvertedPendulum

    seed = 5
    rs = np.random.default_rng(9)
    idx = np.arange(n) if n <= 512 else np.sort(rs.choice(n, size=256, replace=False))
    env = make("InvertedPendulum-v5", n)
    ora = OracleInvertedPendulum(len(idx))
    o1, i1 = env.reset(seed=seed)
    o2, _ = ora.reset(seed=[seed + int(i) for i in idx])
    assert o1.shape == (n, 4) and o1.dtype == np.float64 and i1 == {}
    assert env.single_action_space.shape == (1,) and float(env.single_action_space.high[0]) == 3.0
    np.testing.assert_array_equal(o1[idx], o2)
    resets = np.zeros(len(idx), dtype=np.int64)
    prev_done = np.zeros(n, dtype=bool)
    for t in range(T):
        a = rs.uniform(-3.5, 3.5, size=(n, 1)).astype(dtype)  # beyond the control range on purpose: clamped like ctrllimited
        x = env.step(a)
        y = ora.step(a[idx].astype(np.float32))
        if dtype == np.float64 and (a[idx].astype(np.float32).astype(np.float64) != a[idx]).any():
            np.testing.assert_allclose(x[0][idx], y[0], rtol=0, atol=1e-4)  # float64 actions drive a slightly different run
            break
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        np.testing.assert_array_equal(x[2][idx], y[2])
        np.testing.assert_array_equal(x[3][idx], y[3])
        np.testing.assert_array_equal(x[4]["reward_survive"][idx][~prev_done[idx]], y[4]["reward_survive"][~prev_done[idx]])
        np.testing.assert_array_equal(x[4]["_reward_survive"], ~prev_done)  # lanes on their reset call report no step keys
        prev_done = x[2] | x[3]
        resets += y[2] | y[3]
    if dtype == np.float32:
        assert (resets >= 1).mean() > 0.9  # random pushes drop the pole within ~15 steps
    assert not env.buffer_overflow()


@pytest.mark.parametrize("n,T,limit", [(512, 110, 35), (8192, 50, 20)])
def test_half_cheetah_matches_oracle_bit_exact(n, T, limit):
    """HalfCheetah-v5 on the planar kernels (Euler integrator with implicit joint damping, joint springs, standard_normal reset
    noise from numpy's ziggurat) against oracle/half_cheetah.c: observations, rewards, flags and info, across TimeLimit
    autoresets (the env never terminates)."""
    from oracle.half_cheetah import OracleHalfCheetah

    seed = 17
    rs = np.random.default_rng(21)
    idx = np.arange(n) if n <= 512 else np.sort(rs.choice(n, size=256, replace=False))
    env = make("HalfCheetah-v5", n, max_episode_steps=limit)
    ora = OracleHalfCheetah(len(idx), max_episode_steps=limit)
    o1, i1 = env.reset(seed=seed)
    o2, i2 = ora.reset(seed=[seed + int(i) for i in idx])
    assert o1.shape == (n, 17) and o1.dtype == np.float64 and env.single_action_space.shape == (6,)
    np.testing.assert_array_equal(o1[idx], o2)
    np.testing.assert_array_equal(i1["x_position"][idx], i2["x_position"])
    for i in idx[:16]:  # reset_model's draws are numpy's: uniform(-0.1, 0.1, 9), then 0.1 * standard_normal(9)
        gen = np.random.Generator(np.random.PCG64(np.random.SeedSequence(seed + int(i))))
        qpos = gen.uniform(low=-0.1, high=0.1, size=9)
        np.testing.assert_array_equal(o1[i], np.concatenate([qpos[1:], 0.1 * gen.standard_normal(9)]))
    truncs = 0
    for t in range(T):
        a = rs.uniform(-1.0, 1.0, size=(n, 6)).astype(np.float32)
        x, y = env.step(a), ora.step(a[idx])
        np.testing.assert_array_equal(x[0][idx], y[0], err_msg=f"obs differ at step {t}")
        np.testing.assert_array_equal(x[1][idx], y[1], err_msg=f"reward differs at step {t}")
        assert not x[2].any()
        np.testing.assert_array_equal(x[3][idx], y[3])
        live = x[4]["_x_velocity"][idx]
        for k in ("x_velocity", "reward_forward", "reward_ctrl"):
            np.testing.assert_array_equal(x[4][k][idx][live], y[4][k][live], err_msg=k)
        assert (x[1][x[4]["_x_velocity"]] == (x[4]["reward_forward"] + x[4]["reward_ctrl"])[x[4]["_x_velocity"]]).all()
        truncs += int(y[3].sum())
    assert truncs >= 2 * len(idx) and not env.buffer_overflow()


def test_hopper_sharding_and_api():
    import torch

    whole = make("Hopper-v5", 96, max_episode_steps=30)
    parts = [make("Hopper-v5", 40, env_offset=0, max_episode_steps=30), make("Hopper-v5", 56, env_offset=40, max_episode_steps=30)]
    ow, _ = whole.reset(seed=8)
    np.testing.assert_array_equal(ow, np.concatenate([p.reset(seed=8)[0] for p in parts]))
    rs = np.random.default_rng(2)
    for t in range(70):
        a = rs.uniform(-1, 1, size=(96, 3)).astype(np.float32)
        xw = whole.step(a)
        xp = [parts[0].step(a[:40]), parts[1].step(a[40:])]
        for k in range(4):
            np.testing.assert_array_equal(xw[k], np.concatenate([xp[0][k], xp[1][k]]), err_msg=f"output {k} at step {t}")
    w = make("Walker2d-v5", 8)
    ow2, _ = w.reset(seed=3)
    assert ow2.shape == (8, 17) and w.single_action_space.shape == (6,)
    t_env = make("Hopper-v5", 4, output="torch")
    o, info = t_env.reset(seed=1)
    assert o.dtype == torch.float64 and tuple(o.shape) == (4, 11) and set(info) >= {"x_position", "_x_position"}
    assert t_env.single_action_space.shape == (3,) and float(t_env.single_action_space.high[0]) == 1.0
    with pytest.raises(ValueError, match="Action dimension mismatch"):
        t_env.step(np.zeros((4, 2), dtype=np.float32))
    same = make("Hopper-v5", 16, autoreset_mode="SameStep", max_episode_steps=9)
    same.reset(seed=0)
    for t in range(12):
        _, _, te, tr, info = same.step(np.zeros((16, 3), dtype=np.float32))
        np.testing.assert_array_equal(info["_final_obs"], te | tr)
        np.testing.assert_array_equal(info["_x_velocity"], ~(te | tr))
