"""Reconstruction-metric references (test and measurement infrastructure only; the product never imports this).

metres_torch    the reference's postprocess chain in torch on the images' device: tanh_to_sigmoid, clamp,
                revert_depth(norm=False) and the valid multiply. Run on the GPU it is the same-device rounding the
                kernel must match bit for bit.
sums_numpy      the ten per-scan sums of dusty_depth_metrics in float64 numpy, from the f32 depths and validity masks.
sums_torch      the same sums as a torch chain of masked float64 reductions on the images' device (what a user would
                write without the kernel; the comparison arm of tests/perf_depth_metrics.py).
finalise_numpy  the metrics of each scan from the sums; mean_numpy the average over scans with non-empty S.
The contract is Eigen et al.'s metric set as monodepth2's compute_depth_errors computes it (DESIGN.md §2.8).
"""
import numpy as np
import torch

from oracle.head_projection import tanh_to_sigmoid_clamped

KEYS = ("abs_rel", "sq_rel", "rmse", "rmse_log", "a1", "a2", "a3", "mask_precision", "mask_recall", "mask_iou")


def metres_torch(x, min_depth, max_depth, tol=0.0):
    """(B,1,H,W) tanh-space images -> (depth in metres with invalid pixels multiplied by 0, valid mask)."""
    inv = tanh_to_sigmoid_clamped(x)
    valid = torch.abs(inv - 0) > tol
    disp = inv * (1 / min_depth - 1 / max_depth) + 1 / max_depth       # denormalize_minmax(inv, 1/max, 1/min)
    depth = 1 / disp
    return depth * valid, valid


def sums_numpy(p, vp, t, vt):
    """(B,10) float64: |S|, |pred valid|, |target valid|, sum |d|/t, sum d^2/t, sum d^2, sum (log p - log t)^2, #a1,
    #a2, #a3 over S = vp & vt, with p, t the f32 depths widened to float64 and d = p - t."""
    b = p.shape[0]
    p, t = p.reshape(b, -1).astype(np.float64), t.reshape(b, -1).astype(np.float64)
    vp, vt = vp.reshape(b, -1).astype(bool), vt.reshape(b, -1).astype(bool)
    out = np.zeros((b, 10))
    for i in range(b):
        s = vp[i] & vt[i]
        P, T = p[i][s], t[i][s]
        d = P - T
        ratio = np.maximum(P / T, T / P)
        out[i] = [s.sum(), vp[i].sum(), vt[i].sum(), np.sum(np.abs(d) / T), np.sum(d * d / T), np.sum(d * d),
                  np.sum((np.log(P) - np.log(T)) ** 2), np.sum(ratio < 1.25), np.sum(ratio < 1.25 ** 2),
                  np.sum(ratio < 1.25 ** 3)]
    return out


def sums_torch(p, vp, t, vt):
    """sums_numpy as a torch chain on the tensors' device."""
    b = p.shape[0]
    P, T = p.reshape(b, -1).double(), t.reshape(b, -1).double()
    vp, vt = vp.reshape(b, -1), vt.reshape(b, -1)
    s = vp & vt
    zero = torch.zeros((), dtype=torch.float64, device=p.device)
    d = P - T
    ratio = torch.maximum(P / T, T / P)
    lg = torch.log(P) - torch.log(T)

    def masked(x):
        return torch.where(s, x, zero).sum(dim=1)
    cols = [s.sum(dim=1).double(), vp.sum(dim=1).double(), vt.sum(dim=1).double(), masked(d.abs() / T),
            masked(d * d / T), masked(d * d), masked(lg * lg), (s & (ratio < 1.25)).sum(dim=1).double(),
            (s & (ratio < 1.25 ** 2)).sum(dim=1).double(), (s & (ratio < 1.25 ** 3)).sum(dim=1).double()]
    return torch.stack(cols, dim=1)


def finalise_numpy(sums):
    """{key: (B,) float64} from (B,10) sums; NaN where a denominator is 0."""
    s = np.asarray(sums, dtype=np.float64)
    n, pv, tv = s[:, 0], s[:, 1], s[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        vals = [s[:, 3] / n, s[:, 4] / n, np.sqrt(s[:, 5] / n), np.sqrt(s[:, 6] / n), s[:, 7] / n, s[:, 8] / n,
                s[:, 9] / n, n / pv, n / tv, n / (pv + tv - n)]
    return dict(zip(KEYS, vals))


def mean_numpy(sums):
    """Each key's mean over the scans with non-empty S, plus "#scans" and "#empty"."""
    s = np.asarray(sums, dtype=np.float64)
    keep = s[:, 0] > 0
    per = finalise_numpy(s)
    out = {k: float(v[keep].mean()) if keep.any() else float("nan") for k, v in per.items()}
    out["#scans"], out["#empty"] = int(len(s)), int((~keep).sum())
    return out
