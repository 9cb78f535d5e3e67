import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def golden_files(prefix):
    return sorted(os.path.basename(p) for p in glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def have_cuda():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def fixture_kwargs(name):
    """Constructor kwargs encoded in a golden fixture's file name (see tests/golden/make_golden.py)."""
    kw = {}
    if "samestep" in name:
        kw["autoreset_mode"] = "SameStep"
    if "disabled" in name:
        kw["autoreset_mode"] = "Disabled"
    if name.startswith("frozenlakecustom"):
        kw.update(desc=["SFFHF", "FHFFF", "FFSFH", "HFFFG"], map_name=None, success_rate=0.8, reward_schedule=(10, -5, -1))
        return kw
    if "sutton" in name:
        kw["sutton_barto_reward"] = True
    if name.startswith("frozenlake"):
        kw["map_name"] = "4x4" if "4x4" in name else "8x8"
        if "noslip" in name:
            kw["is_slippery"] = False
    return kw


def fixture_options(name):
    return {"low": -0.1, "high": 0.1} if "bounds" in name else None


def replay_fixture(env, g, options=None, disabled=False):
    """Drive `env` with a golden fixture's seed + action tape; in DISABLED mode finished lanes are reset by the caller
    exactly as tests/golden/make_golden.py did.  Returns stacked outputs (+ per-step infos and reset observations)."""
    obs, info = env.reset(seed=int(g["seed"]), options=options)
    out = dict(obs=[obs], reward=[], terminated=[], truncated=[], info=[info], reset_obs={})
    for t, a in enumerate(g["actions"]):
        o, r, te, tr, info = env.step(a)
        out["obs"].append(o); out["reward"].append(r); out["terminated"].append(te); out["truncated"].append(tr)
        out["info"].append(info)
        done = np.asarray(te) | np.asarray(tr)
        if disabled and done.any():
            o2, _ = env.reset(options={"reset_mask": done.copy()})
            out["reset_obs"][t] = (done.copy(), np.asarray(o2))
    for k in ("obs", "reward", "terminated", "truncated"):
        out[k] = np.stack(out[k])
    return out


def check_reset_obs(out, g, exact=True):
    for t, (mask, o2) in out["reset_obs"].items():
        ref = g["info_reset_obs"][t]
        if exact:
            np.testing.assert_array_equal(o2[mask].astype(np.float64), ref[mask])
        else:
            np.testing.assert_allclose(o2[mask], ref[mask], rtol=1e-5, atol=1e-5)
