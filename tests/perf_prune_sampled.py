import os, sys, time, torch, statistics, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from dusty_gan_b200 import _lib
from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
dev = torch.device("cuda:0")
lidar = bench.make_lidar(dev); head = bench.make_head(1, dev)
N = 1000
ref = bench.make_clouds(N, 2, head, lidar, dev, 1, False); gen = bench.make_clouds(N, 1, head, lidar, dev, 1, False)
def run(): return M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
base = run()
ms = statistics.median(bench.time_events(run, 3, 1))
print("dense   ", ms, "ms", 3 * N * N / ms * 1e3, "entries/s")
M.MERGE_ORIGIN_ABOVE = 1024
pr = run()
ms = statistics.median(bench.time_events(run, 3, 1))
cnt = C.c_uint64()
_lib.load().dusty_chamfer_count_pairs(1, None); run(); _lib.load().dusty_chamfer_count_pairs(0, C.byref(cnt))
print("pruned  ", ms, "ms", 3 * N * N / ms * 1e3, "entries/s; visited fraction", cnt.value / (2001000 * 2 * 2048 * 2048))
print("scores equal:", base == pr, {k: (base[k], pr[k]) for k in base if base[k] != pr[k]})
