"""Restatement of the JSD occupancy metric -- TEST INFRASTRUCTURE ONLY.

Follows reference utils/metrics/jsd.py: unit_cube_grid_point_cloud (:10-20), the brute-force voting of
entropy_of_occupancy_grid (:42-84, distances as (p-g).pow(2).sum(-1) in f32, argmin = first minimum),
_entropy (:95-107, including its in-place ``p += eps``) and _jensen_shannon_divergence (:110-121).
Pinned by tests/golden/jsd_cpu.npz (the reference's own compute_jsd / grid_counters).
"""
import numpy as np
import torch


def grid_points(resolution, clip_sphere=True, device="cpu"):
    """The reference builds its grid on the points' device; on a GPU, torch.norm may round a point that lies exactly
    on the sphere (odd resolutions only) to the other side of 0.5 than on the CPU."""
    spacing = 1.0 / float(resolution - 1)
    steps = torch.arange(resolution, device=device)
    grid = torch.stack(torch.meshgrid(steps, steps, steps, indexing="ij"), dim=-1) * spacing - 0.5
    grid = grid.reshape(-1, 3)
    if clip_sphere:
        grid = grid[torch.norm(grid, dim=1) <= 0.5]
    return grid.cpu().numpy().astype(np.float32), spacing


def vote(pcs, resolution=28, in_sphere=True):
    """-> (grid_counters (Ng,), clouds_touching (Ng,)) as int64."""
    grid, _ = grid_points(resolution, in_sphere)
    pcs = np.asarray(pcs, np.float32)
    B, Np, _ = pcs.shape
    counters = np.zeros(len(grid), np.int64)
    touching = np.zeros(len(grid), np.int64)
    for b in range(B):
        idx = np.empty(Np, np.int64)
        for j in range(0, Np, 256):
            d = pcs[b, j:j + 256, None, :] - grid[None, :, :]          # f32
            d = d * d
            dist = (d[..., 0] + d[..., 1]) + d[..., 2]
            idx[j:j + 256] = dist.argmin(axis=1)
        np.add.at(counters, idx, 1)
        touching[np.unique(idx)] += 1
    return counters, touching


def nearest_torch(points, grid, max_bytes=1 << 30):
    """(dist, idx) of the nearest grid point to each of ``points`` (n,3) on their device: vote()'s arithmetic as
    separate element-wise f32 ops (no ``.sum(-1)`` or matmul form, which may reorder the sum), first minimum on
    ties, in chunks of points so that no intermediate exceeds about ``max_bytes``."""
    points = points.reshape(-1, 3)
    grid = grid.to(points.device)
    dist = torch.empty(len(points), dtype=torch.float32, device=points.device)
    idx = torch.empty(len(points), dtype=torch.int64, device=points.device)
    chunk = max(1, max_bytes // (12 * max(len(grid), 1)))
    for j in range(0, len(points), chunk):
        d = points[j:j + chunk, None, :] - grid[None, :, :]
        d = d * d
        dj = (d[..., 0] + d[..., 1]) + d[..., 2]
        dist[j:j + chunk], idx[j:j + chunk] = dj.amin(dim=1), dj.argmin(dim=1)
    return dist, idx


def vote_torch(pcs, resolution=28, in_sphere=True, grid_device=None):
    """vote() in torch on ``pcs``'s device (a CUDA tensor for the evaluation's sizes) -> (counters, touching) as
    int64 tensors there. The grid is built on ``grid_device``, by default the points' device as in the reference.
    Pinned to vote() by tests/test_gpu_jsd_edges.py."""
    pcs = torch.as_tensor(pcs, dtype=torch.float32)
    B, Np, _ = pcs.shape
    grid = torch.from_numpy(grid_points(resolution, in_sphere, grid_device or pcs.device)[0])
    ng = len(grid)
    if B * Np == 0:
        zero = torch.zeros(ng, dtype=torch.int64, device=pcs.device)
        return zero, zero.clone()
    _, idx = nearest_torch(pcs, grid)
    counters = torch.bincount(idx, minlength=ng)
    touched = torch.zeros(B, ng, dtype=torch.bool, device=pcs.device)
    touched.scatter_(1, idx.view(B, Np), True)
    return counters, touched.sum(0)


def _entropy(p, base2=True, eps=np.float32(1e-8)):
    p += eps                                                           # in place, like the reference
    log_p = np.log2(p) if base2 else np.log(p)
    return (-p * log_p).sum(dtype=np.float32)


def jsd_from_counts(P, Q):
    P = np.asarray(P, np.float32); Q = np.asarray(Q, np.float32)
    P_ = P / P.sum(dtype=np.float32); Q_ = Q / Q.sum(dtype=np.float32)
    e1 = _entropy(P_); e2 = _entropy(Q_)
    e_sum = _entropy((P_ + Q_) / np.float32(2.0))
    return float(e_sum - ((e1 + e2) / np.float32(2.0)))


_EPS64 = float(np.float32(1e-8))       # the reference adds 1e-8 to f32 tensors: the f32 value of 1e-8


def _entropy64(p, log):
    return -(p * log(p)).sum()


def jsd_from_counts_f64(P, Q):
    """_jensen_shannon_divergence in float64 from exact counts, with the reference's eps placement: _entropy adds eps
    to P_ and Q_ in place, so e_sum sees it twice. -> (jsd, e_sum, e1, e2)."""
    P = np.asarray(P, np.float64); Q = np.asarray(Q, np.float64)
    p = P / P.sum() + _EPS64
    q = Q / Q.sum() + _EPS64
    e1, e2 = _entropy64(p, np.log2), _entropy64(q, np.log2)
    e_sum = _entropy64((p + q) / 2.0 + _EPS64, np.log2)
    return e_sum - (e1 + e2) / 2.0, e_sum, e1, e2


def acc_entropy_f64(touching, n_clouds, ng):
    """entropy_of_occupancy_grid's acc_entropy (reference jsd.py:23-92: natural log, eps added once) in float64
    from exact touching counts."""
    t = np.asarray(touching, np.float64)
    p = t[t > 0] / n_clouds
    return _entropy64(np.concatenate([p, 1.0 - p]) + _EPS64, np.log) / ng


def compute_jsd(pcs_gen, pcs_ref, resolution=28):
    return jsd_from_counts(vote(pcs_gen, resolution)[0], vote(pcs_ref, resolution)[0])
