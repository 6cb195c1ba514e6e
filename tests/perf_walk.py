"""Timing of the best-first walk on un-sampled clouds: matrix front end (configs[4] shape, env N) and batch front end
(8 pairs x 32768 points); not a test."""
import os, sys, statistics, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from dusty_gan_b200 import _lib
from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
from dusty_gan_b200.utils.metrics.distance import chamfer_distance
dev = torch.device("cuda:0")
lidar = bench.make_lidar(dev); head = bench.make_head(1, dev)
N = int(os.environ.get("N", 100))
ref = bench.make_clouds(N, 2, head, lidar, dev, 1, True); gen = bench.make_clouds(N, 1, head, lidar, dev, 1, True)
def run(): return M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
pr = run()
ms = statistics.median(bench.time_events(run, 3, 1))
cnt = C.c_uint64()
_lib.load().dusty_chamfer_count_pairs(1, None); run(); _lib.load().dusty_chamfer_count_pairs(0, C.byref(cnt))
kept = torch.cat([(c != 0).any(-1).sum(1) + ((c == 0).all(-1).any(1)).long() for c in (ref, gen)]).double()
kept_pairs = float((kept.sum() ** 2 + (kept ** 2).sum()) / 2) * 2
print("matrix N=%d: %.1f ms  %.0f entries/s  visited %.4f of kept pairs  %s" % (
    N, ms, 3 * N * N / ms * 1e3, cnt.value / kept_pairs,
    {k: pr[k] for k in ("mmd-cd", "cov-cd", "1-nn-accuracy-cd")}))
a, b = ref[:8].contiguous(), gen[:8].contiguous()
d = chamfer_distance(a, b)
ms = statistics.median(bench.time_events(lambda: chamfer_distance(a, b), 10, 3))
print("batch 8 x 32768: %.1f us  %.0f pairs/s  checksum %.9g %.9g" % (
    ms * 1e3, 8 / ms * 1e3, d[0].double().sum().item(), d[1].double().sum().item()))
