import os, sys, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, bench
from dusty_gan_b200.utils.metrics.distance import chamfer_distance
dev = torch.device("cuda:0")
lidar = bench.make_lidar(dev); head = bench.make_head(1, dev)
B = int(os.environ.get("B", 8))
ref = bench.make_clouds(B, 2, head, lidar, dev, 1, True)
gen = bench.make_clouds(B, 1, head, lidar, dev, 1, True)
d = chamfer_distance(ref, gen)
ms = statistics.median(bench.time_events(lambda: chamfer_distance(ref, gen), 10, 3))
print("batch %d x 32768: %.1f us" % (B, ms * 1e3))
