"""Where does the end-to-end time go?  Device-only stepping vs HostPipeline at several depths, full size and 84x84."""
import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from collections import deque
from gym_duckietown_b200.batched_env import BatchedDuckietownEnv, HostPipeline
N, K = 4096, 60
env = BatchedDuckietownEnv(N, "small_loop", camera_width=160, camera_height=120, seed=1000, auto_reset=True, device_reset=True)
env.reset()
dev = env.device
acts = torch.rand((K + 8, N, 2), device=dev) * 2 - 1
h_act = acts.cpu().pin_memory()
def dev_only():
    for t in range(5): env.step(acts[t])
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for t in range(K): env.step(acts[5 + t])
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / K * 1e3
def d2h_only(x):
    h = torch.empty(tuple(x.shape), dtype=x.dtype).pin_memory()
    h.copy_(x, non_blocking=True); torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(10): h.copy_(x, non_blocking=True)
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / 10 * 1e3
def piped(depth):
    pipe = HostPipeline(env, depth=depth)
    for t in range(3): pipe.result(pipe.submit(h_act[t]))
    torch.cuda.synchronize(); t0 = time.perf_counter(); pend = deque()
    for t in range(K):
        pend.append(pipe.submit(h_act[3 + t]))
        if len(pend) >= depth: pipe.result(pend.popleft())
    while pend: pipe.result(pend.popleft())
    return (time.perf_counter() - t0) / K * 1e3
for label, rs in (("160x120", None), ("84x84", (84, 84))):
    if rs: env.set_resize(*rs)
    print(label, "device-only %.3f ms/step" % dev_only(), " D2H of one obs batch %.3f ms (%.1f MB)" % (d2h_only(env.obs), env.obs.numel() / 1e6),
          " ".join("depth%d %.3f" % (d, piped(d)) for d in (1, 2, 3, 4)), flush=True)
