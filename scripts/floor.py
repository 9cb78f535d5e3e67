"""Launch-latency floor: graph-replayed chains of step launches at tiny and BASELINE batch sizes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gymnasium_b200

def chain(env, acts, L=64, reps=50):
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        env.step(acts); torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for _ in range(L):
                env.step(acts)
    for _ in range(5): g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): g.replay()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (reps * L)

for fam, kw, na in [("CartPole-v1", {}, 2), ("FrozenLake-v1", {"map_name": "8x8"}, 4)]:
    for n in [32, 4096, 65536, 262144]:
        env = gymnasium_b200.make_vec(fam, num_envs=n, copy=False, **kw)
        env.reset(seed=0)
        acts = torch.randint(0, na, (n,), device="cuda")
        print(fam, n, "us/launch in graph chain: %.3f" % chain(env, acts))
# torch elementwise kernel chain for comparison
x = torch.zeros(65536, device="cuda")
g = torch.cuda.CUDAGraph()
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    x.add_(1); torch.cuda.synchronize()
    with torch.cuda.graph(g, stream=s):
        for _ in range(64): x.add_(1)
for _ in range(5): g.replay()
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(50): g.replay()
b.record(); torch.cuda.synchronize()
print("torch x.add_(1) 65536 floats, us/launch in graph chain: %.3f" % (a.elapsed_time(b) * 1e3 / (50 * 64)))
