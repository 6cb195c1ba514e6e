import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from dusty_gan_b200 import pipeline
dev = torch.device("cuda:0")
lidar = bench.make_lidar(dev); head = bench.make_head(1, dev)
d, c = bench.backbone_like(256, 1, 11, dev)
def run(): return pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar, tol=0.0, compact=True)
for _ in range(3): run()
torch.cuda.synchronize()
run(); torch.cuda.synchronize()
