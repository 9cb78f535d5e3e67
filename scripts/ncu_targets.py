"""Small deterministic launch sequence for ncu captures (never a bench number): HBM-cold ring of 65536-env CartPole
batches, the same step kernel at N=16M, the fused rollout kernel, FrozenLake-v1 8x8 at 1M envs."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import gymnasium_b200

dev = torch.device("cuda:0")
which = sys.argv[1] if len(sys.argv) > 1 else "all"
if which in ("all", "step"):
    ring = [gymnasium_b200.make_vec("CartPole-v1", num_envs=65536, copy=False, env_offset=j * 65536) for j in range(40)]
    acts = torch.randint(0, 2, (65536,), device=dev)
    for e in ring:
        e.reset(seed=0)
    for rep in range(3):
        for e in ring:
            e.step(acts)
    torch.cuda.synchronize()
    del ring
if which in ("all", "big"):
    e = gymnasium_b200.make_vec("CartPole-v1", num_envs=1 << 24, copy=False)
    e.reset(seed=0)
    a = torch.randint(0, 2, (1 << 24,), device=dev)
    for _ in range(6):
        e.step(a)
    torch.cuda.synchronize()
    del e, a
if which in ("all", "rollout"):
    e = gymnasium_b200.make_vec("CartPole-v1", num_envs=65536)
    e.reset(seed=0)
    for _ in range(4):
        e.rollout(64)
    torch.cuda.synchronize()
    e = gymnasium_b200.make_vec("CartPole-v1", num_envs=1 << 20)
    e.reset(seed=0)
    for _ in range(3):
        e.rollout(64)
    torch.cuda.synchronize()
    del e
if which in ("all", "lake"):
    fl = [gymnasium_b200.make_vec("FrozenLake-v1", num_envs=1 << 20, map_name="8x8", copy=False, env_offset=j << 20)
          for j in range(4)]
    a = torch.randint(0, 4, (1 << 20,), device=dev)
    for f in fl:
        f.reset(seed=0)
    for rep in range(3):
        for f in fl:
            f.step(a)
    f = fl[0]
    f.rollout(32)
    torch.cuda.synchronize()
if which in ("all", "lander"):
    ll = gymnasium_b200.make_vec("LunarLander-v3", num_envs=16384, copy=False)
    ll.reset(seed=0)
    for t in range(80):  # reach the mixed regime: some lanes flying, some on the ground, some resetting
        ll.step(torch.randint(0, 4, (16384,), device=dev))
    torch.cuda.synchronize()
if which in ("all", "humanoid"):
    hm = gymnasium_b200.make_vec("Humanoid-v5", num_envs=8192, copy=False)
    hm.reset(seed=0)
    for t in range(14):  # feet reach the floor around step 10: contacts + PGS active
        hm.step((torch.rand((8192, 17), device=dev) * 0.8 - 0.4).float())
    torch.cuda.synchronize()
if which in ("humanoid", "humanoid_warp", "humanoid_thread"):
    impl = "thread" if which == "humanoid_thread" else "warp"
    hn = int(os.environ.get("B2E_NCU_N", "8192"))
    h = gymnasium_b200.make_vec("Humanoid-v5", num_envs=hn, copy=False, impl=impl)
    h.reset(seed=0)
    g = torch.Generator(device=dev).manual_seed(1)
    for t in range(64):  # steady state: standing / falling / on the ground / resetting envs all present
        h.step(torch.rand((hn, 17), device=dev, generator=g) * 0.8 - 0.4)
    torch.cuda.synchronize()
