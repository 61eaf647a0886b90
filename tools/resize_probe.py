"""Device-only step time at full size and with the device ResizeWrapper to 84x84: what the resize costs per step."""
import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
N, K = 4096, 60
env = BatchedDuckietownEnv(N, "small_loop", camera_width=160, camera_height=120, seed=1000, auto_reset=True, device_reset=True)
env.reset()
acts = torch.rand((K + 8, N, 2), device=env.device) * 2 - 1
def dev_only():
    for t in range(5): env.step(acts[t])
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for t in range(K): env.step(acts[5 + t])
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / K * 1e3
base = dev_only()
env.set_resize(84, 84)
print("full size %.3f ms/step, 84x84 %.3f ms/step -> resize %.3f ms" % (base, (r := dev_only()), r - base), flush=True)
