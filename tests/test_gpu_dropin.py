"""Drop-in through Gymnasium's own registry, checked against the stock sync vectoriser's spaces and outputs stored in
tests/golden/dropin_*.npz (tests/golden/make_golden.py dropin).  Without Gymnasium installed, the same ids go through the
engine's standalone make_vec (gymnasium_b200/registration.py) and are checked against the same fixtures."""
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, golden, have_cuda

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not have_cuda(), reason="needs a CUDA device")]


def replay(env, g):
    """Reset with the fixture's seed, step its action tape, and compare every output (and its dtype) with the fixture."""
    np.testing.assert_array_equal(env.reset(seed=int(g["seed"]))[0], g["obs"][0])
    for t, a in enumerate(g["actions"]):
        x = env.step(a)
        if x[0].dtype == np.float32:
            np.testing.assert_allclose(x[0], g["obs"][t + 1], rtol=1e-5, atol=1e-5)
        else:
            np.testing.assert_array_equal(x[0], g["obs"][t + 1])
        for k, name in ((1, "reward"), (2, "terminated"), (3, "truncated")):
            np.testing.assert_array_equal(x[k], g[name][t])
            assert str(x[k].dtype) == str(g["step_dtypes"][k - 1])


def test_make_vec_through_the_registry():
    import gymnasium_b200

    g = golden("dropin_cartpole_n5_s123_T150.npz")
    if gymnasium_b200.HAVE_GYMNASIUM:
        import gymnasium as gym
        from gymnasium.vector import VectorEnv

        env = gym.make_vec("B200/CartPole-v1", num_envs=5, output="numpy")
        assert isinstance(env, VectorEnv)
        assert env.spec.id == "B200/CartPole-v1" and env.spec.kwargs["num_envs"] == 5
    else:
        env = gymnasium_b200.make_vec("B200/CartPole-v1", num_envs=5, output="numpy")
    assert isinstance(env, gymnasium_b200.B200VectorEnv)
    assert env.max_episode_steps == 500 and env.metadata["autoreset_mode"] is gymnasium_b200.AutoresetMode.NEXT_STEP
    for tag, sp in (("obs_space", env.observation_space), ("single_obs_space", env.single_observation_space)):
        # Box equality as gymnasium.spaces.Box.__eq__ defines it: shape, dtype, np.allclose bounds
        assert str(sp.dtype) == str(g[tag + "_dtype"]) and sp.shape == g[tag + "_low"].shape
        assert np.allclose(sp.low, g[tag + "_low"]) and np.allclose(sp.high, g[tag + "_high"])
    assert str(env.action_space.dtype) == str(g["action_space_dtype"])
    np.testing.assert_array_equal(env.action_space.nvec, g["action_space_nvec"])
    np.testing.assert_array_equal(env.action_space.start, g["action_space_start"])
    replay(env, g)
    env.close()


def test_install_routes_stock_ids():
    import gymnasium_b200

    g = golden("dropin_frozenlake8x8_n6_s5_T200.npz")
    if not gymnasium_b200.HAVE_GYMNASIUM:
        with pytest.raises(RuntimeError, match="gymnasium is not importable"):
            gymnasium_b200.install(["FrozenLake-v1"])
        env = gymnasium_b200.make_vec("FrozenLake-v1", num_envs=6, map_name="8x8", output="numpy")
        assert env.max_episode_steps == 100
        replay(env, g)
        return
    import gymnasium as gym

    gymnasium_b200.install(["FrozenLake-v1"])
    try:
        env = gym.make_vec("FrozenLake-v1", num_envs=6, map_name="8x8", output="numpy")
        assert isinstance(env, gymnasium_b200.B200VectorEnv) and env.max_episode_steps == 100
        replay(env, g)
    finally:
        gymnasium_b200.uninstall()


def test_compat_mode_without_gymnasium():
    """The engine also runs on a box without the host framework (stand-in VectorEnv/spaces, gymnasium_b200/_compat.py)."""
    import subprocess

    code = (
        "import sys, numpy as np\n"
        "import gymnasium_b200\n"
        "assert not gymnasium_b200.HAVE_GYMNASIUM and 'gymnasium' not in sys.modules\n"
        "e = gymnasium_b200.make_vec('CartPole-v1', num_envs=3, output='numpy')\n"
        "o, _ = e.reset(seed=42)\n"
        "assert abs(float(o[0, 0]) - 0.0273956) < 1e-7, o\n"
        "o, r, te, tr, _ = e.step(np.array([1, 0, 1]))\n"
        "assert abs(float(o[0, 1]) - 0.18847767) < 1e-6 and r.dtype == np.float64\n"
        "assert e.action_space.shape == (3,) and e.observation_space.shape == (3, 4)\n"
        "print('compat ok')\n"
    )
    env = dict(os.environ, B200ENV_FORCE_COMPAT="1", PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert p.returncode == 0 and "compat ok" in p.stdout, p.stderr[-2000:]
