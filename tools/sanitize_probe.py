"""A small tour of every kernel for compute-sanitizer (memcheck / racecheck / initcheck): meshes, fisheye at 640x480,
wrapper layouts, the device resize, device resets, the literal tile mode."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
def run(n, m, w, h, steps=3, fmt=None, resize=None, **kw):
    env = BatchedDuckietownEnv(n, m, camera_width=w, camera_height=h, seed=3, auto_reset=True, device_reset=True, **kw)
    if fmt: env.set_output_format(obs_layout=fmt[0], obs_dtype=fmt[1])
    if resize: env.set_resize(*resize)
    env.reset()
    a = torch.rand((steps, n, 2), device=env.device) * 2 - 1
    for t in range(steps): env.step(a[t])
    torch.cuda.synchronize(); env.check(); s = int(env.obs.sum().item()); env.close(); return s
print("meshes", run(96, "loop_obstacles", 160, 120))
print("odd size", run(33, "udem1", 84, 84, domain_rand=True))
print("fisheye", run(3, "udem1", 640, 480, domain_rand=True, distortion=True, steps=2))
print("chw u8", run(40, "small_loop", 160, 120, fmt=("chw", "uint8")))
print("cwh f32", run(40, "small_loop", 160, 120, fmt=("cwh", "float32")))
print("resize", run(40, "loop_obstacles", 160, 120, resize=(84, 84)))
print("literal tiles", run(16, "small_loop", 160, 120, tessellate_tiles=True))
print("dynamic", run(32, "loop_pedestrians", 160, 120, steps=4))
