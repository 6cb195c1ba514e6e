"""Sliced Wasserstein distance references (test and measurement infrastructure only; the product never imports this).

swd_torch   the published op chain (swd-pytorch's compute_swd, the contract of DESIGN.md §2.7) in plain torch f32, on
            the images' device. Its draws come from torch's global CPU generator in the published order, per level:
            randperm, then n_repeat_projection normalised randn blocks. Patches are extracted on the images' device
            (the published code copies the pyramids to the host first; the values are the same).
swd_numpy   the same steps in float64 numpy, given the positions and directions; returns the per-level values.
"""
import numpy as np
import torch
import torch.nn.functional as F

_BINOM = np.float32([1, 4, 6, 4, 1])
KERNEL = (np.outer(_BINOM, _BINOM) / 256).astype(np.float32)


def default_pyramids(h):
    return int(np.rint(np.log2(h // 16)))


def _kernel(x):
    return torch.from_numpy(KERNEL).to(x.device).view(1, 1, 5, 5)


def _pyramid_down(x):
    k = _kernel(x)
    return torch.cat([F.conv2d(x[:, i:i + 1], k, padding=2, stride=2) for i in range(x.size(1))], dim=1)


def _pyramid_up(x):
    k = _kernel(x)
    up = F.interpolate(x, scale_factor=2)
    return torch.cat([F.conv2d(up[:, i:i + 1], k, padding=2) for i in range(x.size(1))], dim=1)


def laplacian_pyramid(x, n_pyramids):
    g = [x]
    for _ in range(n_pyramids):
        g.append(_pyramid_down(g[-1]))
    return [g[i] - _pyramid_up(g[i + 1]) for i in range(n_pyramids)] + [g[-1]]


def extract_patches(layer, indices, slice_size=7, unfold_batch_size=128):
    """(n * n_desc, C * 49) rows normalised per channel over the set, as the published extract_patches."""
    n, c = layer.shape[:2]
    parts = []
    for s in range(0, n, unfold_batch_size):
        x = layer[s:s + unfold_batch_size].unfold(2, slice_size, 1).unfold(3, slice_size, 1)
        x = x.reshape(x.size(0), c, -1, slice_size, slice_size)[:, :, indices.to(layer.device)]
        parts.append(x.permute(0, 2, 1, 3, 4))
    x = torch.cat(parts, dim=0)
    std, mean = torch.std_mean(x, dim=(0, 1, 3, 4), keepdim=True)
    x = (x - mean) / (std + 1e-8)
    return x.reshape(-1, c * slice_size * slice_size)


@torch.no_grad()
def swd_torch(image1, image2, n_pyramids=None, slice_size=7, n_descriptors=128, n_repeat_projection=128,
              proj_per_repeat=4, return_by_resolution=False, draws=None):
    """Published compute_swd. ``draws``: a list that receives (indices, directions (C*49, D)) per level."""
    assert image1.size() == image2.size() and image1.ndim == 4
    if n_pyramids is None:
        n_pyramids = default_pyramids(image1.size(2))
    pyr1 = laplacian_pyramid(image1, n_pyramids)
    pyr2 = laplacian_pyramid(image2, n_pyramids)
    result = []
    for level in range(n_pyramids + 1):
        n = (pyr1[level].size(2) - 6) * (pyr1[level].size(3) - 6)
        indices = torch.randperm(n)[:n_descriptors]
        p1 = extract_patches(pyr1[level], indices, slice_size)
        p2 = extract_patches(pyr2[level], indices, slice_size)
        distances, blocks = [], []
        for _ in range(n_repeat_projection):
            rand = torch.randn(p1.size(1), proj_per_repeat)
            rand = rand / torch.std(rand, dim=0, keepdim=True)
            blocks.append(rand)
            rand = rand.to(image1.device)
            proj1, _ = torch.sort(torch.matmul(p1, rand), dim=0)
            proj2, _ = torch.sort(torch.matmul(p2, rand), dim=0)
            distances.append(torch.mean(torch.abs(proj1 - proj2)))
        if draws is not None:
            draws.append((indices, torch.cat(blocks, dim=1)))
        result.append(torch.mean(torch.stack(distances)))
    result = torch.stack(result) * 1e3
    return result.cpu() if return_by_resolution else torch.mean(result).cpu()


def _down64(x):
    n, c, h, w = x.shape
    p = np.pad(x, ((0, 0), (0, 0), (2, 2), (2, 2)))
    out = np.zeros((n, c, h // 2, w // 2))
    for i in range(5):
        for j in range(5):
            out += float(KERNEL[i, j]) * p[:, :, i:i + h:2, j:j + w:2]
    return out


def _up64(x):
    up = x.repeat(2, axis=2).repeat(2, axis=3)
    n, c, h, w = up.shape
    p = np.pad(up, ((0, 0), (0, 0), (2, 2), (2, 2)))
    out = np.zeros_like(up)
    for i in range(5):
        for j in range(5):
            out += float(KERNEL[i, j]) * p[:, :, i:i + h, j:j + w]
    return out


def pyramid_numpy(images, n_pyramids):
    g = [np.asarray(images, dtype=np.float64)]
    for _ in range(n_pyramids):
        g.append(_down64(g[-1]))
    return [g[i] - _up64(g[i + 1]) for i in range(n_pyramids)] + [g[-1]]


def descriptors_numpy(layer, positions):
    """Unnormalised (n * n_desc, C * 49) rows of one level at the given top-left positions."""
    n, c, h, w = layer.shape
    py, px = np.divmod(np.asarray(positions, dtype=np.int64), w - 6)
    ky, kx = np.divmod(np.arange(49), 7)
    rows = layer[:, :, py[:, None] + ky[None, :], px[:, None] + kx[None, :]]      # (n, c, n_desc, 49)
    return rows.transpose(0, 2, 1, 3).reshape(n * len(positions), c * 49)


def normalise_numpy(rows, c):
    x = rows.reshape(rows.shape[0], c, 49)
    mean = x.mean(axis=(0, 2), keepdims=True)
    std = x.std(axis=(0, 2), ddof=1, keepdims=True)
    return ((x - mean) / (std + 1e-8)).reshape(rows.shape)


def swd_numpy(image1, image2, positions, directions, n_pyramids):
    """Per-level SWD (already x 1e3) in float64. positions[l]: (n_desc,) ints; directions[l]: (C*49, D)."""
    c = image1.shape[1]
    pyr1, pyr2 = pyramid_numpy(image1, n_pyramids), pyramid_numpy(image2, n_pyramids)
    out = []
    for level in range(n_pyramids + 1):
        pos = np.asarray(positions[level])
        dirs = np.asarray(directions[level], dtype=np.float64)
        a = normalise_numpy(descriptors_numpy(pyr1[level], pos), c) @ dirs
        b = normalise_numpy(descriptors_numpy(pyr2[level], pos), c) @ dirs
        out.append(np.abs(np.sort(a, axis=0) - np.sort(b, axis=0)).mean() * 1e3)
    return np.array(out)


def range_images(n, c, h, w, seed, dropped=0.3):
    """Calibrated DUSty-like images: tanh-space inverse depth, smooth along each row, with a fraction of pixels dropped
    to exactly -1 (the heavy ties of real range images)."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(n, c, h, w, generator=g).cumsum(dim=3) / (w ** 0.5)
    img = torch.tanh(base * 1.2 - 0.3 + 0.2 * torch.randn(n, c, h, w, generator=g))
    drop = torch.rand(n, c, h, w, generator=g) < dropped
    return torch.where(drop, torch.full_like(img, -1.0), img)
