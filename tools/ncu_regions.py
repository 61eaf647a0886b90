"""Instruction / sample shares of k_raster by source region (line ranges found by marker comments in dts_render.cu)."""
import csv, os, sys, re
src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gym-duckietown_b200', 'csrc', 'dts_render.cu')).read().splitlines()
def find(pat, start=0):
    for i in range(start, len(src)):
        if pat in src[i]: return i + 1
    raise KeyError(pat)
marks = [
    ("shade (load + eval)", find("struct ShadeIn {"), find("// ---- bulk-async copy")),
    ("pack / store", find("__device__ __forceinline__ unsigned pack_rgb"), find("struct FrameMem {")),
    ("work item setup + producer", find("k_raster(const DState S"), find("    for (int cbx = 0; cbx < cbins_x; cbx++) {", find("k_raster(const DState S"))),
    ("coarse-bin control / empty bins", find("    for (int cbx = 0; cbx < cbins_x; cbx++) {", find("k_raster(const DState S")), find("          // ---- acquire this chunk")),
    ("chunk acquire + flags", find("          // ---- acquire this chunk"), find("          for (int f = (single ? 0 : g)")),
    ("fine-bin control + simple test", find("          for (int f = (single ? 0 : g)"), find("              // ---- visibility: everything else first")),
    ("visibility (warp-wide prim visits)", find("              // ---- visibility: everything else first"), find("              // ---- tiny triangles, ONE PER LANE") - 1),
    ("tiny triangles (lane per prim)", find("              // ---- tiny triangles, ONE PER LANE") - 1, find("            // ---- deferred shading")),
    ("deferred shading control + resolve", find("            // ---- deferred shading"), find("// ------------------------------------------------------------------------------------------------ k_resize")),
]
r = list(csv.reader(open(sys.argv[1])))
hi = [i for i, x in enumerate(r) if x and x[0] == "Line No"][0]
h = r[hi]; ix = {}
for i, n in enumerate(h): ix.setdefault(n, i)
def f(x):
    try: return float(x)
    except ValueError: return 0.0
rows = [x for x in r[hi + 1:] if len(x) == len(h) and x[2] == "-"]
ts = sum(f(x[ix["# Samples"]]) for x in rows); ti = sum(f(x[ix["Instructions Executed"]]) for x in rows)
acc = {m[0]: [0, 0] for m in marks}; other = [0, 0]
for x in rows:
    ln = int(x[0]); s_, i_ = f(x[ix["# Samples"]]), f(x[ix["Instructions Executed"]])
    for name, a, b in marks:
        if a <= ln < b: acc[name][0] += s_; acc[name][1] += i_; break
    else: other[0] += s_; other[1] += i_
print("warp-instructions %.4g  samples %d" % (ti, ts))
for name, a, b in marks: print("%-40s lines %4d-%4d  %5.1f%% inst  %5.1f%% samples  %.4g inst" % (name, a, b, 100 * acc[name][1] / ti, 100 * acc[name][0] / ts, acc[name][1]))
print("%-40s %17s %5.1f%% inst  %5.1f%% samples" % ("other (intrinsics headers, helpers)", "", 100 * other[1] / ti, 100 * other[0] / ts))
