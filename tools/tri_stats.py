"""Triangle statistics of the raster oracle (orr_stats_read) for a few maps: how many set-up triangles reach no sample."""
import os, sys, numpy as np, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import oracle as orc
from gym_duckietown_b200 import maps
orc.build(force=True)
L = orc.lib()
L.orr_stats_read.argtypes = [C.POINTER(C.c_longlong), C.c_int]
def poses(md, n, seed):
    rng = np.random.default_rng(seed); out = []
    for _ in range(n):
        i, j = md.drivable_tiles[rng.integers(len(md.drivable_tiles))]
        out.append(((i + rng.uniform()) * md.tile_size, (j + rng.uniform()) * md.tile_size, rng.uniform(-np.pi, np.pi)))
    return out
for name, W, H in [('small_loop', 160, 120), ('loop_obstacles', 160, 120), ('udem1', 160, 120), ('udem1', 640, 480)]:
    md = maps.load_map(name); sc = orc.OracleScene(md)
    buf = (C.c_longlong * 8)(); L.orr_stats_read(buf, 1)
    n = 32
    for x, z, a in poses(md, n, 5): sc.render(x, z, a, W=W, H=H)
    L.orr_stats_read(buf, 1)
    s = np.array(list(buf)) / n
    print(name, W, H, 'tris/frame %.0f  no-sample-in-bbox %.0f  no-covered-sample %.0f  <=2x2 %.0f  <=4x4 %.0f quads %.0f' % tuple(s[:6]))
