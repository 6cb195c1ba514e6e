"""The flow of the reference's evaluate_synthesis.py (:20-195) on the B200 kernels, with synthetic stand-ins
for what this container lacks (KITTI scans, a trained checkpoint): raw scans -> real cache -> generated
range images -> clouds -> JSD + MMD / COV / 1-NNA, printed as the reference's score dict.

    python examples/evaluate_synthesis.py --num-test 200 --num-points 2048 [--dusty 2] [--tol 0.0]

Every stage is one call of this package where the reference script calls its own modules:
    preprocess_reals + cache loop (:49-57, :76-97)   pipeline.build_real_cache
    [skip:limit:skip] subsampling (:102-110)         pipeline.subsample_time_series
    G(latent) -> maskout (:157-158)                  a stand-in backbone + DUSty1/DUSty2.maskout fused with
    project_2d_to_3d (:59-64)                        pipeline.generate_points
    compute_jsd (:174-177)                           utils.metrics.jsd.compute_jsd
    compute_cov_mmd_1nna (:178-183)                  utils.metrics.cov_mmd_1nna.compute_cov_mmd_1nna
(SWD, :169-173, is a 2-D image metric outside the path.)
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dusty_gan_b200 import pipeline  # noqa: E402
from dusty_gan_b200.models.dusty import DUSty1, DUSty2  # noqa: E402
from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles  # noqa: E402
from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_cov_mmd_1nna  # noqa: E402
from dusty_gan_b200.utils.metrics.jsd import compute_jsd  # noqa: E402

H, W = 64, 512


class StandInBackbone(torch.nn.Module):
    """Random smooth range images in tanh space + confidence logits: the role of the reference's
    DCGAN-eqlr generator (models/gans/dcgan_eqlr.py), which stays PyTorch and is not the product."""

    def __init__(self, channels):
        super().__init__()
        self.channels = channels

    def forward(self, latent):
        B = latent.shape[0]
        low = latent[:, :128].view(B, 1, 4, 32)
        z = torch.nn.functional.interpolate(low, size=(H, W), mode="bilinear", align_corners=False)
        z = z + 0.35 * torch.randn(B, 1, H, W, device=latent.device)
        z = (z - z.mean()) / z.std()
        return {"depth": torch.tanh(0.68 * z - 1.72), "confidence": 2.0 * torch.randn(B, self.channels, H, W, device=latent.device)}


def synthetic_scan_batches(n, batch, device, seed):
    """Raw (64,2048,4) scans as process_kitti.py stores them; a slowly drifting scene (a 'time series')."""
    g = torch.Generator(device=device).manual_seed(seed)
    elev = torch.deg2rad(torch.linspace(2.0, -24.8, 64, device=device))[:, None]
    azim = torch.linspace(np.pi, -np.pi, 2049, device=device)[:-1][None, :]
    base = torch.randn(1, 1, 4, 32, generator=g, device=device)
    for i in range(0, n, batch):
        b = min(batch, n - i)
        base = base + 0.2 * torch.randn(b, 1, 4, 32, generator=g, device=device).cumsum(0)[-1:]
        low = base + 0.3 * torch.randn(b, 1, 4, 32, generator=g, device=device)
        r = torch.nn.functional.interpolate(low, size=(64, 2048), mode="bilinear", align_corners=False)[:, 0]
        r = (20 + 14 * r + 2 * torch.randn(b, 64, 2048, generator=g, device=device)).abs() + 0.5
        r = r * (torch.rand(b, 64, 2048, generator=g, device=device) > 0.3)
        yield torch.stack([r * torch.cos(elev) * torch.cos(azim), r * torch.cos(elev) * torch.sin(azim),
                           r * torch.sin(elev), torch.rand(b, 64, 2048, generator=g, device=device)], dim=-1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-test", type=int, default=200)
    ap.add_argument("--num-points", type=int, default=2048)
    ap.add_argument("--tol", type=float, default=0.0)
    ap.add_argument("--batch-size", type=int, default=32)       # cfg.solver.batch_size
    ap.add_argument("--dusty", type=int, default=1, choices=[1, 2])
    ap.add_argument("--metrics", default="cd", help="comma-separated subset of cd,emd for MMD/COV/1-NNA")
    args = ap.parse_args()
    metrics = tuple(m.strip() for m in args.metrics.split(",") if m.strip())
    if not metrics or any(m not in ("cd", "emd") for m in metrics):
        ap.error(f"--metrics: expected a subset of cd,emd, got {args.metrics!r}")
    torch.set_grad_enabled(False)
    device = torch.device("cuda")
    torch.manual_seed(0)

    lidar = LiDAR(num_ring=H, num_points=W, min_depth=0.9, max_depth=120.0, angle=synthetic_hdl64e_angles()).to(device)
    G = (DUSty1 if args.dusty == 1 else DUSty2)(StandInBackbone(args.dusty), tau=1.0, drop_const=-1).to(device).eval()
    # utils.setup(fix_noise=True), reference utils/__init__.py:141-149: freeze the first logistic draw
    for m in G.modules():
        if m.__class__.__name__ == "GumbelSigmoid" and m.pixelwise:
            m.fixed_noise = m.logistic_noise(torch.empty(1, 1, H, W, device=device))[[0]]

    t0 = time.perf_counter()
    reals = pipeline.build_real_cache(synthetic_scan_batches(2 * args.num_test + 3, args.batch_size, device, 7), lidar, args.num_points)
    reals = {k: pipeline.subsample_time_series(v, args.num_test) for k, v in reals.items()}
    torch.cuda.synchronize(); t1 = time.perf_counter()

    N_test = len(reals["2d"])
    fakes = {"2d": [], "3d": []}
    for _ in range(0, N_test, args.batch_size):
        latent = torch.randn(args.batch_size, 512, device=device)
        points, out = pipeline.generate_points(G, G.backbone(latent), lidar, args.num_points, tol=args.tol)
        fakes["2d"].append(out["depth"]); fakes["3d"].append(points)
    fakes = {k: torch.cat(v, dim=0)[:N_test] for k, v in fakes.items()}
    torch.cuda.synchronize(); t2 = time.perf_counter()

    scores = {"jsd": compute_jsd(pcs_gen=fakes["3d"] / 2.0, pcs_ref=reals["3d"] / 2.0)}
    scores.update(compute_cov_mmd_1nna(pcs_gen=fakes["3d"], pcs_ref=reals["3d"], batch_size=512, metrics=metrics))
    torch.cuda.synchronize(); t3 = time.perf_counter()
    scores["#test"] = args.num_test
    scores["#points"] = args.num_points
    print(json.dumps(scores, ensure_ascii=False, indent=4, sort_keys=True))
    print(f"real cache {t1 - t0:.3f} s | synthesis {t2 - t1:.3f} s | metrics {t3 - t2:.3f} s  ({N_test} vs {N_test} clouds)",
          file=sys.stderr)


if __name__ == "__main__":
    main()
