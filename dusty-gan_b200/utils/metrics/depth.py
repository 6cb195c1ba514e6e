"""Reconstruction metrics of range images on libdustyb200 (mirror of reference utils/metrics/depth.py, called by
evaluate_reconstruction.py).

The reference's depth.py is not in this tree; only its outline is known ("RMSE / abs-rel / delta accuracy"). The
contract is therefore the standard set of Eigen et al. (2014) in the form monodepth2's ``compute_depth_errors`` uses,
computed per scan and averaged over the scans (DESIGN.md §2.8). Every formula that turns the kernel's per-scan sums
into a metric lives in ``finalise`` below, so if the reference's file differs, the change is made there.

Both images go through the reference's postprocess chain: ``inv = clamp((x + 1) / 2, 0, 1)``, ``valid = |inv| > tol``
(a NaN pixel is not valid), depth in metres ``revert_depth(inv, norm=False)``. With S the pixels valid in both images
and p, t the predicted and target depths on S (in float64, from the float32 depths):

    abs_rel = mean |p - t| / t          rmse     = sqrt(mean (p - t)^2)
    sq_rel  = mean (p - t)^2 / t        rmse_log = sqrt(mean (log p - log t)^2)
    a1, a2, a3 = fraction of S with max(p / t, t / p) < 1.25, 1.25^2, 1.25^3

A scan with empty S gives NaN for these keys. The mask scores are an addition that the reference's outline does not
list: the agreement of the two validity masks, mask_precision = |S| / |pred valid|, mask_recall = |S| / |target
valid| and mask_iou = |S| / |pred valid or target valid| (NaN where the denominator is 0). They come from the counts
the means need anyway, and the drop mask is what a point-drop model is trained to get right.
"""
import ctypes

import numpy as np
import torch

from ... import _lib

KEYS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "mask_precision", "mask_recall", "mask_iou")
REDUCTIONS = ("mean", "none")


def _check(depth_gen, depth_ref, lidar, reduction):
    if reduction not in REDUCTIONS:
        raise ValueError(f"reduction={reduction!r}: expected one of {REDUCTIONS}")
    for name, x in (("depth_gen", depth_gen), ("depth_ref", depth_ref)):
        if not isinstance(x, torch.Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if x.dim() != 4 or x.shape[1] != 1:
            raise ValueError(f"{name}: expected (B,1,H,W), got {tuple(x.shape)}")
    if depth_gen.shape != depth_ref.shape:
        raise ValueError(f"depth_gen and depth_ref differ in shape: {tuple(depth_gen.shape)} vs {tuple(depth_ref.shape)}")
    _, _, h, w = depth_gen.shape
    if (h, w) != (lidar.H, lidar.W):
        raise ValueError(f"images are {h}x{w}, the LiDAR's range image is {lidar.H}x{lidar.W}")
    if w % 4:
        raise ValueError(f"W={w} must be a multiple of 4")
    if lidar.drop_const != 0:
        raise NotImplementedError("the kernel implements the LiDAR drop value 0 used by every caller "
                                  "(reference utils/lidar.py:12,121-125)")
    _lib.require_cuda(depth_gen, "depth_gen")
    _lib.require_cuda(depth_ref, "depth_ref")
    if depth_gen.device != depth_ref.device:
        raise ValueError(f"depth_gen and depth_ref are on different devices: {depth_gen.device} and {depth_ref.device}")


def depth_sums(depth_gen, depth_ref, lidar, tol=0.0, return_depth=False):
    """The kernel's (B, 10) float64 per-scan sums on the images' device (columns: |S|, |pred valid|, |target valid|,
    sum |d|/t, sum d^2/t, sum d^2, sum (log p - log t)^2, #a1, #a2, #a3), and with ``return_depth`` the two (B,1,H,W)
    float32 depth images in metres (0 where invalid). Arguments are those of ``compute_depth_metrics``."""
    from ...models.dusty import _projection_fields
    _check(depth_gen, depth_ref, lidar, "none")
    pred, target = depth_gen.contiguous(), depth_ref.contiguous()
    b, _, h, w = pred.shape
    p = _lib.HeadParams()
    p.b, p.h, p.w, p.conf_channels = b, h, w, 1
    _projection_fields(p, lidar, tol)
    sums = torch.empty(b, 10, dtype=torch.float64, device=pred.device)
    metres = (torch.empty_like(pred), torch.empty_like(target)) if return_depth else (None, None)
    lib = _lib.load()
    ws = _lib.workspace(lib.dusty_depth_metrics_workspace_bytes(b, h, w), pred.device)
    with torch.cuda.device(pred.device):
        _lib.check(lib.dusty_depth_metrics(ctypes.byref(p), _lib.ptr(pred), _lib.ptr(target), _lib.ptr(sums),
                                           _lib.ptr(metres[0]), _lib.ptr(metres[1]), _lib.ptr(ws), ws.numel(),
                                           _lib.stream_of(pred)), "dusty_depth_metrics")
    return (sums, *metres) if return_depth else sums


def finalise(s):
    """(B, 10) float64 numpy sums of ``depth_sums`` -> {key: (B,) float64 array}, the metrics of each scan."""
    n, pv, tv = s[:, 0], s[:, 1], s[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        return {
            "abs_rel": s[:, 3] / n,
            "sq_rel": s[:, 4] / n,
            "rmse": np.sqrt(s[:, 5] / n),
            "rmse_log": np.sqrt(s[:, 6] / n),
            "a1": s[:, 7] / n,
            "a2": s[:, 8] / n,
            "a3": s[:, 9] / n,
            "mask_precision": n / pv,
            "mask_recall": n / tv,
            "mask_iou": n / (pv + tv - n),
        }


@torch.no_grad()
def compute_depth_metrics(depth_gen, depth_ref, lidar, tol=0.0, reduction="mean", return_depth=False):
    """Reconstruction metrics of (B,1,H,W) float32 CUDA range images in the generator's tanh space (dropped pixels at
    -1): ``depth_gen`` the reconstructions, ``depth_ref`` the real scans, paired scan by scan. ``lidar`` supplies H, W
    and the depth limits; ``tol`` is the validity tolerance of ``inv_to_xyz``. Every argument is checked before the
    one library call.

    ``reduction="mean"``: a dict of Python floats, each key's mean over the scans whose S is not empty, plus
    ``"#scans"`` and ``"#empty"`` (NaN values when every S is empty). ``reduction="none"``: a dict of (B,) float64 CPU
    tensors. With ``return_depth=True`` the result is ``(scores, pred_metres, target_metres)``, the two (B,1,H,W)
    float32 depth images in metres (0 where invalid) on the images' device."""
    _check(depth_gen, depth_ref, lidar, reduction)
    out = depth_sums(depth_gen, depth_ref, lidar, tol, return_depth)
    sums, metres = (out[0], out[1:]) if return_depth else (out, ())
    s = sums.cpu().numpy()
    per_scan = finalise(s)
    if reduction == "none":
        scores = {k: torch.from_numpy(v) for k, v in per_scan.items()}
    else:
        keep = s[:, 0] > 0
        scores = {k: float(v[keep].mean()) if keep.any() else float("nan") for k, v in per_scan.items()}
        scores["#scans"] = int(len(keep))
        scores["#empty"] = int((~keep).sum())
    return (scores, *metres) if return_depth else scores
