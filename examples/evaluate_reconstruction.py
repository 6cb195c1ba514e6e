"""The flow of the reference's evaluate_reconstruction.py on the B200 kernels, with synthetic stand-ins for what this
tree lacks (KITTI scans, a trained checkpoint, the reference's inversion loss): raw scans -> real range images and
un-sampled clouds -> latents fitted to each scan -> reconstruction scores, printed as one JSON dict.

    python examples/evaluate_reconstruction.py --num-test 256 --steps 50 [--dusty 2] [--tol 0.0]

Every stage is one call of this package where the reference script calls its own modules:
    raw scans -> inv, points                 pipeline.preprocess_reals
    G(latent) -> maskout, postprocess        pipeline.maskout_and_project (differentiable=True inside the inversion)
    depth metrics + compute_cd (:124-131)    pipeline.reconstruction_scores
The inversion here is a STAND-IN: a few Adam steps on the stand-in backbone's latents against a masked L1 loss on the
inverse depth. The reference's inversion loss and optimiser are not in this tree and are not rebuilt.
"""
import argparse
import json
import math
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dusty_gan_b200 import pipeline  # noqa: E402
from dusty_gan_b200.models.dusty import DUSty1, DUSty2  # noqa: E402
from dusty_gan_b200.utils import tanh_to_sigmoid  # noqa: E402
from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles  # noqa: E402
from dusty_gan_b200.utils.metrics.depth import KEYS  # noqa: E402
from evaluate_synthesis import synthetic_scan_batches  # noqa: E402

H, W = 64, 512
LATENT = 256


class StandInBackbone(torch.nn.Module):
    """A deterministic, differentiable latent -> {depth, confidence} map (the role of the reference's generator, which
    stays PyTorch and is not the product): each half of the latent is a 4x32 grid, upsampled to the range image."""

    def __init__(self, channels):
        super().__init__()
        self.channels = channels

    def forward(self, latent):
        b = latent.shape[0]
        grid = latent.view(b, 2, 4, 32)
        up = torch.nn.functional.interpolate(grid, size=(H, W), mode="bilinear", align_corners=False)
        conf = 2.0 + 4.0 * up[:, 1:]
        return {"depth": torch.tanh(up[:, :1]), "confidence": conf.expand(b, self.channels, H, W).contiguous()}


def invert(G, real_inv, lidar, steps, lr, tol):
    """Stand-in inversion: Adam on the latents, masked L1 between the generated and real inverse depth in [0, 1]."""
    z = torch.zeros(real_inv.shape[0], LATENT, device=real_inv.device, requires_grad=True)
    opt = torch.optim.Adam([z], lr=lr)
    target = tanh_to_sigmoid(real_inv)
    mask = (real_inv > -1).float()
    loss = torch.full((), math.nan)
    for _ in range(steps):
        out = pipeline.maskout_and_project(G, G.backbone(z), lidar, tol=tol, differentiable=True)
        loss = ((tanh_to_sigmoid(out["depth"]) - target).abs() * mask).sum() / mask.sum().clamp(min=1)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
    return z.detach(), float(loss)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--num-test", type=int, default=256)
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--steps", type=int, default=50, help="stand-in inversion steps per batch")
    ap.add_argument("--lr", type=float, default=0.1)
    ap.add_argument("--tol", type=float, default=0.0)
    ap.add_argument("--dusty", type=int, default=1, choices=[1, 2])
    args = ap.parse_args()
    device = torch.device("cuda")
    torch.manual_seed(0)

    lidar = LiDAR(num_ring=H, num_points=W, min_depth=0.9, max_depth=120.0, angle=synthetic_hdl64e_angles()).to(device)
    G = (DUSty1 if args.dusty == 1 else DUSty2)(StandInBackbone(args.dusty), tau=1.0, drop_const=-1).to(device).eval()
    for m in G.modules():         # utils.setup(fix_noise=True): freeze the first logistic draw
        if m.__class__.__name__ == "GumbelSigmoid" and m.pixelwise:
            m.fixed_noise = m.logistic_noise(torch.empty(1, 1, H, W, device=device))[[0]]

    t0 = time.perf_counter()
    totals, n_depth, n_cd, last_loss = dict.fromkeys(KEYS + ("cd",), 0.0), 0, 0, math.nan
    for scans in synthetic_scan_batches(args.num_test, args.batch_size, device, 7):
        real_inv, _, real_points = pipeline.preprocess_reals(scans, lidar)
        z, last_loss = invert(G, real_inv, lidar, args.steps, args.lr, args.tol)
        with torch.no_grad():
            s = pipeline.reconstruction_scores(G, G.backbone(z), real_inv, real_points, lidar, tol=args.tol)
        b = s.pop("#scans")
        kept = b - s.pop("#empty")
        cd = s.pop("cd")
        if kept:                      # depth keys: means over the scans with a non-empty overlap
            for k, v in s.items():
                totals[k] += v * kept
        totals["cd"] += cd * b
        n_depth, n_cd = n_depth + kept, n_cd + b
    torch.cuda.synchronize()
    t1 = time.perf_counter()

    scores = {k: (v / (n_cd if k == "cd" else n_depth)) if (n_cd if k == "cd" else n_depth) else math.nan
              for k, v in totals.items()}
    scores["#scans"] = n_cd
    scores["#empty"] = n_cd - n_depth
    scores["inversion_loss"] = last_loss
    print(json.dumps(scores, ensure_ascii=False, indent=4, sort_keys=True))
    print(f"inversion + scores {t1 - t0:.3f} s ({n_cd} scans, {args.steps} steps per batch)", file=sys.stderr)


if __name__ == "__main__":
    main()
