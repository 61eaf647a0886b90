"""Print DTS_STATS counters of the raster kernel for the bench workload (needs a -DDTS_STATS build):

    DTS_NVCC_EXTRA=-DDTS_STATS=1 python gym-duckietown_b200/build.py --force
    python tools/raster_stats.py [map]
    python gym-duckietown_b200/build.py --force    # back to the product build
"""
import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
m = sys.argv[1] if len(sys.argv) > 1 else "small_loop"
env = BatchedDuckietownEnv(4096, m, camera_width=160, camera_height=120, domain_rand=False, seed=1000, auto_reset=True, device_reset=True)
env.reset(render=False)
a = torch.rand((30, 4096, 2), device=env.device) * 2 - 1
for t in range(30):
    env.step(a[t], render=False)
torch.cuda.synchronize()
c0 = env.sim.debug_counters().astype(np.int64)
env.render_obs(); torch.cuda.synchronize()
c = env.sim.debug_counters().astype(np.int64) - c0
names = {8: "coarse bins", 9: "  empty (cleared)", 10: "sum of list lengths (records)", 14: "coarse bins with > 32 records", 15: "  their records",
         11: "fine bins shaded", 13: "  simple (one covering prim, no visibility pass)", 12: "extra shading rounds (2nd..4th winner of edge pixels)",
         16: "warp-wide prim visits", 17: "  trivially accepted (no edge tests)", 20: "general bins holding only road tiles (coverage-only visibility)", 21: "  of those redone with depth (a sample covered twice)", 22: "coarse bins inside one prim (solo)", 23: "  their fine bins", 18: "tiny-triangle passes (fine bins)", 19: "  tiny triangles in them"}
for k, v in names.items():
    print(f"{v:60s} {c[k]:12d}  per env {c[k]/4096:10.1f}")
