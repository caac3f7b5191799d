import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from eirgrid_b200 import _lib
ctx = _lib.Context(0); ctx.map_load_dir(os.path.join(ROOT, "tests", "golden", "ireland_map"))
for half, step in ((25, 2000.0), (50, 1000.0), (100, 500.0)):
    ctx.location_analysis(True, half, step)
    t = time.perf_counter(); s = ctx.location_analysis(True, half, step); dt = time.perf_counter() - t
    n = (2 * half + 1) ** 2
    print("half %d: %d points x 15 types in %.2f ms -> %.2f M point-types/s, water points %.0f%%" % (half, n, dt * 1e3, n * 15 / dt / 1e6, 100 * (s[:, 1] > 0).mean()))
