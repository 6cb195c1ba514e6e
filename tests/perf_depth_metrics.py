"""Reconstruction-metric timings on the B200; prints one JSON line.

    python tests/perf_depth_metrics.py

64x512 tanh-space range images (dropped pixels at -1: 30 % of the predictions, 45 % of the targets), batches of 32,
256 and 5000 scans. Per batch:
* dusty_depth_metrics (sums only) device-timed with CUDA events around each call, the L2 overwritten by a 512 MB write
  before every timed call (32 and 256 scans would otherwise be read from the 126 MB L2), median of the calls; its
  algorithmic bytes (two f32 images read once) over that time against the data-sheet HBM bandwidth of one B200;
* the same with the two metre images written (8 more bytes per pixel);
* compute_depth_metrics end to end (host clock around a call that ends in the host-side finalisation);
* the torch chain on the same GPU and inputs (oracle/depth.py: metres_torch on both images, then sums_torch, masked
  float64 reductions), timed like the kernel.
At 5000 scans two more inputs separate the bounds: every pixel valid on both sides (the float64 work, two logs and a
division per pixel, is done everywhere) and every target pixel dropped (S is empty: the same bytes, no float64 work).
The card's name, power limit and clocks are read in the same run.
"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import depth as od  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
H, W = 64, 512


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                                       str(torch.cuda.current_device())], text=True)
        return dict(zip(q.split(","), [s.strip() for s in out.strip().split(",")]))
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}


_FLUSH = None


def timed(fn, reps):
    """Median device time (ms) of fn over reps calls, each after a 512 MB write that evicts the L2."""
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(128 << 20, dtype=torch.float32, device="cuda")
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        _FLUSH.fill_(1.0)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def wall(fn, reps):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t) * 1e3)
    return statistics.median(times)


def images(b, seed, dropped):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.tanh(torch.randn(b, 1, H, W, generator=g, device="cuda") * 0.8 - 0.2)
    return torch.where(torch.rand(b, 1, H, W, generator=g, device="cuda") < dropped, torch.full_like(x, -1.0), x)


def kernel_ms(x, y, lidar, reps, metres=False):
    from dusty_gan_b200.utils.metrics.depth import depth_sums
    return timed(lambda: depth_sums(x, y, lidar, return_depth=metres), reps)


def run(b, lidar, reps):
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics, depth_sums
    x, y = images(b, 1, 0.3), images(b, 2, 0.45)
    npix = b * H * W
    k_ms = kernel_ms(x, y, lidar, reps)
    km_ms = kernel_ms(x, y, lidar, reps, metres=True)
    e2e_ms = wall(lambda: compute_depth_metrics(x, y, lidar), reps)

    def chain():
        mx, vx = od.metres_torch(x, lidar.min_depth, lidar.max_depth)
        my, vy = od.metres_torch(y, lidar.min_depth, lidar.max_depth)
        return od.sums_torch(mx, vx, my, vy)
    ref_ms = timed(chain, max(3, reps // 4))
    got, want = depth_sums(x, y, lidar), chain()
    worst = float(((got - want).abs() / want.abs().clamp(min=1e-300))[:, 3:6].max())
    out = {"scans": b, "pixels": npix,
           "kernel_ms": round(k_ms, 4), "kernel_bytes": 8 * npix,
           "kernel_tb_per_s": round(8 * npix / k_ms / 1e9, 3),
           "kernel_share_of_hbm_datasheet": round(8 * npix / k_ms / 1e-3 / HBM_BYTES_PER_S, 3),
           "kernel_with_metres_ms": round(km_ms, 4),
           "kernel_with_metres_tb_per_s": round(16 * npix / km_ms / 1e9, 3),
           "compute_depth_metrics_ms": round(e2e_ms, 4),
           "torch_chain_ms": round(ref_ms, 3), "speedup_vs_torch_chain": round(ref_ms / k_ms, 1),
           "counts_equal_torch_chain": bool(torch.equal(got[:, [0, 1, 2, 7, 8, 9]], want[:, [0, 1, 2, 7, 8, 9]])),
           "max_rel_diff_sums_vs_torch_chain": worst}
    if b == 5000:
        valid_ms = kernel_ms(x.clamp(min=-0.9), y.clamp(min=-0.9), lidar, reps)
        empty_ms = kernel_ms(x, torch.full_like(y, -1.0), lidar, reps)
        out.update({"all_valid_kernel_ms": round(valid_ms, 4), "all_valid_tb_per_s": round(8 * npix / valid_ms / 1e9, 3),
                    "no_overlap_kernel_ms": round(empty_ms, 4),
                    "no_overlap_tb_per_s": round(8 * npix / empty_ms / 1e9, 3)})
    return out


def main():
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    torch.cuda.set_device(0)
    lidar = LiDAR(H, W, 0.9, 120.0, angle=synthetic_hdl64e_angles()).cuda()
    runs = [run(b, lidar, reps) for b, reps in ((32, 50), (256, 30), (5000, 10))]
    print(json.dumps({"card": card(), "runs": runs}))


if __name__ == "__main__":
    main()
