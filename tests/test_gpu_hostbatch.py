"""The single host-side batch on a GPU: HostBatchPipeline (pinned H2D of actions -> fused step -> D2H of the outputs into the
page-locked shared batch, copies of step k overlapping the kernel of step k+1) must hand out exactly what the blocking
``step()`` returns.  world_size 1 here (one GPU per test box); the world_size-2 protocol runs on CPU in
tests/test_distributed_cpu.py and on GPUs in scripts/hostbatch_multi.py (gpurun --gpus 2)."""
import numpy as np
import pytest
import torch

import gymnasium_b200
from gymnasium_b200.distributed import HostBatchPipeline

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("fast", [True, False])
@pytest.mark.parametrize("env_id,n,steps", [("CartPole-v1", 4096, 40), ("Humanoid-v5", 64, 12), ("FrozenLake-v1", 2048, 30),
                                            ("LunarLander-v3", 512, 30), ("Hopper-v5", 256, 30)])
def test_pipeline_batches_equal_blocking_step(env_id, n, steps, fast):
    kw = {"map_name": "8x8"} if env_id.startswith("FrozenLake") else {}
    ref = gymnasium_b200.make_vec(env_id, num_envs=n, output="numpy", **kw)
    env = gymnasium_b200.make_vec(env_id, num_envs=n, copy=False, out_buffers=3, **kw)
    ref.reset(seed=11)
    env.reset(seed=11)
    rs = np.random.default_rng(5)
    if env_id == "Humanoid-v5":
        acts = rs.uniform(-0.4, 0.4, size=(steps, n, 17)).astype(np.float32)
    elif env_id == "Hopper-v5":
        acts = rs.uniform(-1.0, 1.0, size=(steps, n, 3)).astype(np.float32)
    else:
        acts = rs.integers(0, ref.single_action_space.n, size=(steps, n))
    pipe = HostBatchPipeline(env, 1, 0, tag=f"test_{env_id}_{int(fast)}", depth=3, fast=fast)
    expect = [ref.step(a) for a in acts]
    got = []
    for k in range(steps):
        t = pipe.submit(acts[k])
        if t >= 1:  # consume one step behind, as the bench loop does; release the slot after reading it
            got.append({key: v.copy() for key, v in pipe.consume(t - 1, ack=False).items()})
            pipe.release(t - 1)
    got.append({key: v.copy() for key, v in pipe.consume(steps - 1, ack=False).items()})
    pipe.release(steps - 1)
    assert bool(pipe._fast) == fast  # fast: every submit was ONE b2e_pipe_submit call replaying the recorded step
    pipe.close()
    for k in range(steps):
        o, r, te, tr, info = expect[k]
        np.testing.assert_array_equal(got[k]["obs"], o, err_msg=f"step {k}")
        np.testing.assert_array_equal(got[k]["reward"], r)
        np.testing.assert_array_equal(got[k]["terminated"], te)
        np.testing.assert_array_equal(got[k]["truncated"], tr)
    if env_id == "Humanoid-v5":
        assert got[-1]["info"].shape == (13, n)
        np.testing.assert_array_equal(got[-1]["info"][7], expect[-1][4]["x_velocity"])


@pytest.mark.parametrize("env_id,n", [("CartPole-v1", 4096), ("Humanoid-v5", 64), ("CartPole-v1", 1001)])
def test_pipeline_pinned_actions_and_landing_modes(env_id, n):
    """Page-locked action batches (no staging copy), rows landed by the landing kernel: same batches (n = 1001: rows that
    are not 16-byte multiples take the kernel's byte path)."""
    steps, depth = 25, 4
    ref = gymnasium_b200.make_vec(env_id, num_envs=n, output="numpy")
    env = gymnasium_b200.make_vec(env_id, num_envs=n, copy=False, out_buffers=depth)
    ref.reset(seed=3)
    env.reset(seed=3)
    rs = np.random.default_rng(8)
    pipe = HostBatchPipeline(env, 1, 0, tag=f"pin_{env_id}_{n}", depth=depth)
    pool = pipe.pinned_actions(depth + 1)
    expect, got = [], []
    for k in range(steps):
        a = pool[k % len(pool)]  # last used depth+1 steps ago: that step has been consumed
        if env_id == "Humanoid-v5":
            a[...] = rs.uniform(-0.4, 0.4, size=a.shape)
        else:
            a[...] = rs.integers(0, 2, size=a.shape)
        expect.append(ref.step(a.copy()))
        t = pipe.submit(a)
        if t >= 2:
            got.append({key: v.copy() for key, v in pipe.consume(t - 2, ack=False).items()})
            pipe.release(t - 2)
    for t in (steps - 2, steps - 1):
        got.append({key: v.copy() for key, v in pipe.consume(t, ack=False).items()})
        pipe.release(t)
    assert pipe._fast and pipe._slots[0].land is not None
    pipe.close()
    for k in range(steps):
        np.testing.assert_array_equal(got[k]["obs"], expect[k][0], err_msg=f"step {k}")
        np.testing.assert_array_equal(got[k]["reward"], expect[k][1])
        np.testing.assert_array_equal(got[k]["terminated"], expect[k][2])
        np.testing.assert_array_equal(got[k]["truncated"], expect[k][3])


def test_out_buffers_rotate_without_aliasing():
    env = gymnasium_b200.make_vec("CartPole-v1", num_envs=256, copy=False, out_buffers=3)
    env.reset(seed=1)
    a = torch.zeros(256, dtype=torch.int64, device=env.device)
    ptrs = [env.step(a)[0].data_ptr() for _ in range(6)]
    assert len(set(ptrs[:3])) == 3 and ptrs[:3] == ptrs[3:]
