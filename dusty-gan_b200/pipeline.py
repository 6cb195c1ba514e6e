"""Fused generate -> points entry: what evaluate_synthesis.py does between ``G.backbone(latent)`` and
``compute_cov_mmd_1nna`` (reference evaluate_synthesis.py:59-64,151-163; trainers/dcgan_amp.py:344-349).

    backbone output {depth, confidence}
      -> maskout + tanh_to_sigmoid + clamp + inv_to_xyz + flatten/transpose      (one kernel)
      -> downsample_point_clouds                                                  (one kernel)

and the real-data side of the same script (evaluate_synthesis.py:49-57, 69-110):

    raw (64,2048,4) scans -> preprocess_reals (one kernel) -> downsample_point_clouds -> {"2d","3d"} cache
"""
import contextlib

import torch

from .datasets.kitti import preprocess_scans
from .models.dusty import _head_call
from .utils.sampling.fps import downsample_point_clouds


def maskout_and_project(head, output, lidar, tol=0.0, threshold=0.5, compact=False, buffers=None,
                        differentiable=False):
    """``head`` is a DUSty1/DUSty2 module, ``output`` the backbone's dict. Returns the dict updated like
    ``maskout`` plus ``points`` (B,H*W,3) -- the contiguous layout FPS consumes -- and, with
    ``compact=True``, ``valid_count`` (B,), ``valid_index`` (B,H*W) and ``valid_points`` (B,H*W,3):
    the valid pixels of each image in ascending pixel order (what ``points[i][valid[i]]`` selects).

    Runs under ``no_grad`` unless ``differentiable=True``; then ``depth``, ``mask`` and ``points`` carry gradients
    to ``output["depth"]`` and ``output["confidence"]`` (the inversion loss of demo.py:510-515 back-propagates a
    Chamfer loss on the points to the latent). Compaction outputs have no gradient, so ``compact=True`` is refused
    there."""
    if differentiable and compact:
        raise ValueError("maskout_and_project: compact=True has no gradient; use differentiable=False")
    with contextlib.nullcontext() if differentiable else torch.no_grad():
        out, points, count, index, compacted = _head_call(head, output, threshold, lidar=lidar, tol=tol,
                                                          points_layout=1, compact=compact, buffers=buffers)
    out["points"] = points
    if compact:
        out["valid_count"], out["valid_index"], out["valid_points"] = count, index, compacted
    return out


@torch.no_grad()
def generate_points(head, output, lidar, num_points, tol=0.0, threshold=0.5):
    """range images -> FPS-sampled clouds (B,num_points,3): project_2d_to_3d of the reference."""
    out = maskout_and_project(head, output, lidar, tol=tol, threshold=threshold)
    return downsample_point_clouds(out["points"], num_points), out


@torch.no_grad()
def preprocess_reals(scans, lidar, drop_const=-1):
    """Raw scans (B,Hs,Ws,C) on the GPU -> (inv, mask, points) of evaluate_synthesis.py:49-57; ``lidar``
    supplies the range-image shape and the depth limits (LiDAR(num_ring, num_points, min_depth, max_depth))."""
    out = preprocess_scans(scans, (lidar.H, lidar.W), lidar.min_depth, lidar.max_depth, drop_const)
    return out["inv"], out["mask"], out["points"]


@torch.no_grad()
def build_real_cache(scan_batches, lidar, num_points, drop_const=-1, device="cuda"):
    """The ``reals[subset]`` dict evaluate_synthesis.py:76-97 builds and ``torch.save``s as
    ``data/cache_<dataset>_<subset>_<num_points>.pt``: {"2d": (N,1,H,W) inverse-depth images,
    "3d": (N,num_points,3) FPS-sampled clouds}. ``scan_batches`` yields (B,Hs,Ws,C) float tensors (or
    the dataset's collated {"scan": ...} dicts); two kernels per batch."""
    two_d, three_d = [], []
    for batch in scan_batches:
        scans = batch["scan"] if isinstance(batch, dict) else batch
        inv, _, points = preprocess_reals(scans.to(device, non_blocking=True), lidar, drop_const)
        two_d.append(inv)
        three_d.append(downsample_point_clouds(points, num_points))
    return {"2d": torch.cat(two_d, dim=0), "3d": torch.cat(three_d, dim=0)}


def subsample_time_series(t, num_test):
    """Every ``len(t)//num_test``-th sample (evaluate_synthesis.py:102-110); -1 keeps everything."""
    if num_test == -1:
        return t
    skip = len(t) // num_test
    limit = skip * num_test + 1
    return t[skip:limit:skip]
