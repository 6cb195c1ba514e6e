"""Timing of the resident-pair kernel on the evaluation's shape (env: N, P, ABOVE); not a test."""
import os, sys, statistics, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from dusty_gan_b200 import _lib
from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
dev = torch.device("cuda:0")
lidar = bench.make_lidar(dev); head = bench.make_head(1, dev)
N = int(os.environ.get("N", 1000)); P = int(os.environ.get("P", 2048))
bench.N_POINTS = P
ref = bench.make_clouds(N, 2, head, lidar, dev, 1, False); gen = bench.make_clouds(N, 1, head, lidar, dev, 1, False)
def run(): return M.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
M.MERGE_ORIGIN_ABOVE = int(os.environ.get("ABOVE", 1024))
pr = run()
ms = statistics.median(bench.time_events(run, 3, 1))
cnt = C.c_uint64()
_lib.load().dusty_chamfer_count_pairs(1, None); run(); _lib.load().dusty_chamfer_count_pairs(0, C.byref(cnt))
E2 = N * (2 * N + 1)
print("N=%d P=%d: %.1f ms  %.0f entries/s  visited %.4f  scores %s" % (
    N, P, ms, 3 * N * N / ms * 1e3, cnt.value / (E2 * 2 * P * P), pr))
