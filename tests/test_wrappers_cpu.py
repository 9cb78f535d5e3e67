"""On-device vector wrappers (gymnasium_b200/wrappers.py) against the reference's NumPy wrappers, driven by the same
scripted vector env (CPU tensors: the wrappers are device-agnostic torch code).  The reference's outputs on these tapes
are stored in tests/golden/wrappers_reference.npz (tests/golden/make_golden_wrappers.py)."""
import functools

import numpy as np
import pytest
import torch

from conftest import golden

from gymnasium_b200 import wrappers as W
from gymnasium_b200._api import AutoresetMode, Box, Discrete, VectorEnv, batch_space


@functools.cache
def reference():
    return golden("wrappers_reference.npz")


class ScriptedEnv(VectorEnv):
    """Replays fixed (obs, reward, terminated, truncated) tapes with NEXT_STEP semantics; numpy or torch outputs."""

    def __init__(self, n, T, seed, as_torch, mode=AutoresetMode.NEXT_STEP):
        rs = np.random.default_rng(seed)
        self.num_envs = n
        self.metadata = {"autoreset_mode": mode}
        self.single_observation_space = Box(-np.inf, np.inf, (3,), np.float32)
        self.single_action_space = Discrete(2)
        self.observation_space = batch_space(self.single_observation_space, n)
        self.action_space = batch_space(self.single_action_space, n)
        self.obs = rs.normal(1.5, 2.0, size=(T + 1, n, 3)).astype(np.float32)
        self.rew = rs.normal(0.3, 1.0, size=(T, n))
        self.term = rs.random((T, n)) < 0.07
        self.trunc = rs.random((T, n)) < 0.04
        self.t, self.as_torch = 0, as_torch
        self.prev_done = np.zeros(n, dtype=bool)
        self.device = torch.device("cpu")

    def _cv(self, x):
        return torch.from_numpy(np.ascontiguousarray(x)) if self.as_torch else x

    def reset(self, *, seed=None, options=None):
        self.t = 0
        self.prev_done[:] = False
        return self._cv(self.obs[0]), {}

    def step(self, actions):
        t = self.t
        r, te, tr = self.rew[t].copy(), self.term[t].copy(), self.trunc[t].copy()
        if self.metadata["autoreset_mode"] == AutoresetMode.NEXT_STEP:
            r[self.prev_done] = 0.0; te[self.prev_done] = False; tr[self.prev_done] = False
        self.prev_done = te | tr
        self.t += 1
        return self._cv(self.obs[t + 1]), self._cv(r), self._cv(te), self._cv(tr), {}


@pytest.mark.parametrize("mode", [AutoresetMode.NEXT_STEP, AutoresetMode.SAME_STEP])
def test_record_episode_statistics_matches_reference(mode):
    REF, p = reference(), f"res_{mode.name.lower()}_"
    n, T = 6, 120
    mine = W.RecordEpisodeStatistics(ScriptedEnv(n, T, 1, True, mode), buffer_length=50)
    mine.reset()
    for t in range(T):
        a = np.zeros(n, dtype=np.int64)
        _, _, te2, tr2, mi = mine.step(a)
        done = REF[p + "done"][t]
        np.testing.assert_array_equal(mi["_episode"].numpy(), done)
        if done.any():
            assert REF[p + "ep_present"][t]
            np.testing.assert_allclose(mi["episode"]["r"].numpy(), REF[p + "ep_r"][t], rtol=0, atol=1e-12)
            np.testing.assert_array_equal(mi["episode"]["l"].numpy(), REF[p + "ep_l"][t])
            np.testing.assert_array_equal(REF[p + "ep_mask"][t], done)
        else:
            assert not REF[p + "ep_present"][t] and float(mi["episode"]["r"].abs().sum()) == 0.0
    assert mine.episode_count == int(REF[p + "episode_count"])
    np.testing.assert_allclose(np.sort(mine.return_queue.numpy()), np.sort(REF[p + "return_queue"]), atol=1e-12)
    np.testing.assert_array_equal(np.sort(mine.length_queue.numpy()), np.sort(REF[p + "length_queue"]))
    # a buffer smaller than the number of episodes (and than the finishers of one step): same entries, same (chronological)
    # order as the reference's deques
    mine = W.RecordEpisodeStatistics(ScriptedEnv(n, T, 1, True, mode), buffer_length=4)
    mine.reset()
    for t in range(T):
        mine.step(np.zeros(n, dtype=np.int64))
        k = int(REF[p + "q4_len"][t])
        np.testing.assert_allclose(mine.return_queue.numpy(), REF[p + "rq4"][t, :k], atol=1e-12, err_msg=f"step {t}")
        np.testing.assert_array_equal(mine.length_queue.numpy(), REF[p + "lq4"][t, :k])


def test_normalize_observation_and_reward_match_reference():
    REF = reference()
    n, T = 8, 90
    mo = W.NormalizeObservation(ScriptedEnv(n, T, 2, True))
    mr = W.NormalizeReward(ScriptedEnv(n, T, 3, True), gamma=0.97)
    o2, _ = mo.reset()
    np.testing.assert_allclose(o2.numpy(), REF["no_obs"][0], rtol=1e-4, atol=1e-5)
    mr.reset()
    for t in range(T):
        a = np.zeros(n, dtype=np.int64)
        o2, *_ = mo.step(a)
        assert o2.dtype == torch.float32
        np.testing.assert_allclose(o2.numpy(), REF["no_obs"][t + 1], rtol=1e-4, atol=1e-5)
        _, r2, *_ = mr.step(a)
        # the reference takes np.mean/np.var of a float32 array (float32 pairwise sums); ours reduces in float64
        np.testing.assert_allclose(r2.numpy(), REF["nr_rew"][t], rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(mo.obs_rms.mean.numpy(), REF["no_mean"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(float(mr.return_rms.var), float(REF["nr_var"]), rtol=2e-6)
    with pytest.raises(ValueError):
        W.NormalizeObservation(ScriptedEnv(2, 3, 0, True), epsilon=0)
    with pytest.raises(ValueError):
        W.NormalizeReward(ScriptedEnv(2, 3, 0, True), gamma=1.5)


class InfoEnv(ScriptedEnv):
    """ScriptedEnv whose infos carry masked arrays and a nested dict, as SyncVectorEnv builds them (vector_env.py:277-338)."""

    def _info(self, t):
        n = self.num_envs
        rs = np.random.default_rng(1000 + t)
        m1, m2 = rs.random(n) < 0.5, rs.random(n) < 0.3
        info = {"k": rs.normal(size=n), "_k": m1, "always": np.arange(n, dtype=np.int64) + t,
                "nest": {"z": rs.normal(size=n).astype(np.float32), "_z": m2}, "_nest": m2}
        if self.as_torch:
            info = {"k": torch.from_numpy(info["k"]), "_k": torch.from_numpy(m1), "always": torch.from_numpy(info["always"]),
                    "nest": {"z": torch.from_numpy(info["nest"]["z"]), "_z": torch.from_numpy(m2)}, "_nest": torch.from_numpy(m2)}
        return info

    def reset(self, *, seed=None, options=None):
        o, _ = super().reset(seed=seed, options=options)
        return o, self._info(0)

    def step(self, actions):
        out = super().step(actions)
        return out[:4] + (self._info(self.t),)


def reference_info_list(t):
    """The reference DictInfoToList's list of per-env dicts at call t, rebuilt from the stored presence masks and values
    (an entry "a.b" is key b of the nested dict under key a)."""
    REF = reference()
    paths =[str(s) for s in REF["dil_paths"]]
    out = []
    for i in range(REF["dil_present_" + paths[0]].shape[1]):
        d = {}
        for path in paths:
            if not REF["dil_present_" + path][t, i]:
                continue
            *parents, key = path.split(".")
            node = d
            for q in parents:
                node = node.setdefault(q, {})
            if "dil_value_" + path in REF:
                node[key] = REF["dil_value_" + path][t, i]
            else:
                node.setdefault(key, {})
        out.append(d)
    return out


def test_dict_info_to_list_matches_reference():
    n, T = 6, 12
    ours = W.DictInfoToList(InfoEnv(n, T, 3, True))
    _, ib = ours.reset(seed=0)
    for t in range(T + 1):
        ia = reference_info_list(t)
        assert isinstance(ib, list) and len(ib) == n == len(ia)
        for a, b in zip(ia, ib):
            assert set(a) == set(b)
            for k in a:
                if isinstance(a[k], dict):
                    assert set(a[k]) == set(b[k])
                    for kk in a[k]:
                        assert a[k][kk] == b[k][kk] and np.asarray(b[k][kk]).dtype == np.asarray(a[k][kk]).dtype
                else:
                    assert a[k] == b[k] and np.asarray(b[k]).dtype == np.asarray(a[k]).dtype
        if t < T:
            ib = ours.step(np.zeros(n, dtype=np.int64))[4]


def test_numpy_to_torch_outputs_are_the_numpy_env_outputs_as_tensors():
    """The reference wrapper (numpy_to_torch.py:15-80) needs `array_api_compat`, which is not installed here; its
    contract is "same values, torch types" (tests/wrappers/vector/test_numpy_to_torch.py), checked against the raw env."""
    n, T = 5, 8
    raw, ours = InfoEnv(n, T, 4, False), W.NumpyToTorch(InfoEnv(n, T, 4, True))
    (oa, ia), (ob, ib) = raw.reset(seed=0), ours.reset(seed=0)
    assert isinstance(ob, torch.Tensor) and np.array_equal(oa, ob.numpy()) and np.array_equal(ia["k"], ib["k"].numpy())
    for t in range(T):
        a = raw.step(np.zeros(n, dtype=np.int64))
        b = ours.step(torch.zeros(n, dtype=torch.int64))
        for x, y in zip(a[:4], b[:4]):
            assert isinstance(y, torch.Tensor) and np.array_equal(x, y.numpy()) and y.numpy().dtype == x.dtype
        assert np.array_equal(a[4]["nest"]["z"], b[4]["nest"]["z"].numpy()) and np.array_equal(a[4]["_k"], b[4]["_k"].numpy())


def test_numpy_to_torch_switches_a_numpy_engine_env_to_torch_outputs():
    class Fake(ScriptedEnv):
        output = "numpy"

        @property
        def unwrapped(self):
            return self

    e = Fake(3, 4, 0, False)
    w = W.NumpyToTorch(e)
    assert e.output == "torch"
    assert isinstance(w.reset()[0], torch.Tensor)  # host arrays a non-engine env still returns are converted
