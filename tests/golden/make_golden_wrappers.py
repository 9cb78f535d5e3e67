"""Generate tests/golden/wrappers_reference.npz from the reference's own NumPy vector wrappers (Gymnasium v1.4.0):
RecordEpisodeStatistics, NormalizeObservation, NormalizeReward and DictInfoToList, driven by the scripted envs of
tests/test_wrappers_cpu.py.  Needs the reference importable ahead of this repository:

    PYTHONPATH=<Gymnasium v1.4.0 source tree>:. python tests/golden/make_golden_wrappers.py
"""
import os
import sys

import numpy as np

import gymnasium as gym
from gymnasium.wrappers.vector import DictInfoToList, NormalizeObservation, NormalizeReward, RecordEpisodeStatistics

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from test_wrappers_cpu import AutoresetMode, InfoEnv, ScriptedEnv  # noqa: E402


def record_episode_statistics(out, mode):
    p = f"res_{mode.name.lower()}_"
    n, T = 6, 120
    ref = RecordEpisodeStatistics(ScriptedEnv(n, T, 1, False, mode), buffer_length=50)
    ref.reset()
    done, present = np.zeros((T, n), bool), np.zeros(T, bool)
    ep_r, ep_l, ep_mask = np.zeros((T, n)), np.zeros((T, n), np.int64), np.zeros((T, n), bool)
    for t in range(T):
        _, _, te, tr, ri = ref.step(np.zeros(n, dtype=np.int64))
        done[t] = te | tr
        if "episode" in ri:
            present[t] = True
            ep_r[t], ep_l[t], ep_mask[t] = ri["episode"]["r"], ri["episode"]["l"], ri["_episode"]
    out.update({p + "done": done, p + "ep_present": present, p + "ep_r": ep_r, p + "ep_l": ep_l, p + "ep_mask": ep_mask,
                p + "episode_count": np.int64(ref.episode_count), p + "return_queue": np.array(ref.return_queue),
                p + "length_queue": np.array(ref.length_queue, dtype=np.int64)})
    ref = RecordEpisodeStatistics(ScriptedEnv(n, T, 1, False, mode), buffer_length=4)
    ref.reset()
    q_len, rq, lq = np.zeros(T, np.int64), np.full((T, 4), np.nan), np.full((T, 4), -1, np.int64)
    for t in range(T):
        ref.step(np.zeros(n, dtype=np.int64))
        k = q_len[t] = len(ref.return_queue)
        rq[t, :k], lq[t, :k] = np.array(ref.return_queue), np.array(ref.length_queue)
    out.update({p + "q4_len": q_len, p + "rq4": rq, p + "lq4": lq})


def normalize(out):
    n, T = 8, 90
    ro = NormalizeObservation(ScriptedEnv(n, T, 2, False))
    rr = NormalizeReward(ScriptedEnv(n, T, 3, False), gamma=0.97)
    obs, rew = np.zeros((T + 1, n, 3), np.float32), np.zeros((T, n))
    obs[0], _ = ro.reset()
    rr.reset()
    for t in range(T):
        obs[t + 1] = ro.step(np.zeros(n, dtype=np.int64))[0]
        rew[t] = rr.step(np.zeros(n, dtype=np.int64))[1]
    out.update(no_obs=obs, nr_rew=rew, no_mean=np.asarray(ro.obs_rms.mean), nr_var=np.float64(rr.return_rms.var))


def dict_info_to_list(out):
    """Each per-env dict flattened to paths ("nest.z" = key z of the dict under key nest): a presence mask per path and,
    for leaves, the value in the dtype the reference returned."""
    n, T = 6, 12
    ref = DictInfoToList(InfoEnv(n, T, 3, False))
    infos = [ref.reset(seed=0)[1]] + [ref.step(np.zeros(n, dtype=np.int64))[4] for _ in range(T)]
    leaves = {}

    def walk(d, t, i, prefix=""):
        for k, v in d.items():
            path = prefix + k
            out.setdefault("dil_present_" + path, np.zeros((T + 1, n), bool))[t, i] = True
            if isinstance(v, dict):
                walk(v, t, i, path + ".")
            else:
                leaves.setdefault(path, np.zeros((T + 1, n), np.asarray(v).dtype))[t, i] = v

    for t, lst in enumerate(infos):
        for i, d in enumerate(lst):
            walk(d, t, i)
    out["dil_paths"] = np.array(sorted(k[len("dil_present_"):] for k in out if k.startswith("dil_present_")))
    out.update({"dil_value_" + k: v for k, v in leaves.items()})


if __name__ == "__main__":
    print("reference:", gym.__version__, gym.__file__, "numpy", np.__version__)
    out = {}
    for mode in (AutoresetMode.NEXT_STEP, AutoresetMode.SAME_STEP):
        record_episode_statistics(out, mode)
    normalize(out)
    dict_info_to_list(out)
    np.savez_compressed(os.path.join(HERE, "wrappers_reference.npz"), **out)
    print({k: v.shape for k, v in out.items()})
