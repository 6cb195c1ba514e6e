"""Sliced Wasserstein distance between two sets of range images on libdustyb200 (mirror of reference
utils/metrics/swd.py, called at evaluate_synthesis.py:169-173). The algorithm is swd-pytorch's, step by step; the
random draws, the direction normalisation and the default level count live here, not in the kernels (DESIGN.md §2.7).
"""
import numpy as np
import torch

from ... import _lib, sharding


def default_pyramids(h):
    """The published default: int(rint(log2(H // 16))), 2 for 64-row images."""
    if h // 16 < 1:
        raise ValueError(f"n_pyramids has no default for H={h} < 16; pass it explicitly")
    return int(np.rint(np.log2(h // 16)))


def draw(h, w, c, n_pyramids, n_descriptors=128, n_repeat_projection=128, proj_per_repeat=4):
    """The published draws from torch's global CPU generator, in its order: per level, finest first,
    ``randperm((h_l-6)(w_l-6))[:n_descriptors]`` and then ``n_repeat_projection`` blocks of ``randn(c*49,
    proj_per_repeat)``, each divided by its own unbiased std over dim 0. Returns [(positions, directions (c*49, D))]."""
    out = []
    for level in range(n_pyramids + 1):
        hl, wl = h >> level, w >> level
        positions = torch.randperm((hl - 6) * (wl - 6))[:n_descriptors]
        blocks = []
        for _ in range(n_repeat_projection):
            rand = torch.randn(c * 49, proj_per_repeat)
            blocks.append(rand / torch.std(rand, dim=0, keepdim=True))
        out.append((positions, torch.cat(blocks, dim=1)))
    return out


def _check(image1, image2, n_pyramids, slice_size, n_descriptors, n_repeat_projection, proj_per_repeat):
    if image1.dim() != 4 or image2.dim() != 4:
        raise ValueError(f"expected (N,C,H,W) images, got {tuple(image1.shape)} and {tuple(image2.shape)}")
    if image1.shape != image2.shape:
        raise ValueError(f"image sets differ in shape: {tuple(image1.shape)} vs {tuple(image2.shape)}")
    if slice_size != 7:
        raise ValueError(f"slice_size={slice_size}: only 7x7 patches are supported")
    n, c, h, w = image1.shape
    if n_pyramids is None:
        n_pyramids = default_pyramids(h)
    levels = n_pyramids + 1
    if not 1 <= c <= 4:
        raise ValueError(f"C={c}: 1 to 4 channels are supported")
    if n_pyramids < 0 or levels > 16:
        raise ValueError(f"n_pyramids={n_pyramids}: 0 to 15 are supported")
    if min(n_descriptors, n_repeat_projection, proj_per_repeat, n) < 1:
        raise ValueError("n_descriptors, n_repeat_projection, proj_per_repeat and N must be positive")
    f = 1 << n_pyramids
    if h % f or w % f:
        raise ValueError(f"{h}x{w} is not divisible by 2^n_pyramids = {f}")
    hl, wl = h >> n_pyramids, w >> n_pyramids
    if hl < 7 or wl < 7:
        raise ValueError(f"the coarsest level is {hl}x{wl}, smaller than the 7x7 patch")
    if (hl - 6) * (wl - 6) < n_descriptors:
        raise ValueError(f"the coarsest level has {(hl - 6) * (wl - 6)} patch positions, fewer than "
                         f"n_descriptors={n_descriptors}")
    if n * n_descriptors > 1 << 30 or h * w > 2 ** 31 - 1 or n_repeat_projection * proj_per_repeat > 2 ** 31 - 1:
        raise ValueError("sizes overflow the kernels' indexing")
    if image1.device != image2.device:
        raise ValueError(f"image sets are on different devices: {image1.device} and {image2.device}")
    _lib.require_cuda(image1, "image1")
    _lib.require_cuda(image2, "image2")
    return n_pyramids


def descriptors(images, positions, levels, n_desc):
    """Stage A: ((levels, N*n_desc, C*49) f32 descriptors, (levels, C, 2) f64 mean / std) on the images' device."""
    x = images.contiguous()
    n, c, h, w = x.shape
    desc = torch.empty(levels, n * n_desc, c * 49, dtype=torch.float32, device=x.device)
    stats = torch.empty(levels, c, 2, dtype=torch.float64, device=x.device)
    lib = _lib.load()
    ws = _lib.workspace(lib.dusty_swd_descriptors_workspace_bytes(n, c, h, w, levels, n_desc), x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.dusty_swd_descriptors(_lib.ptr(x), n, c, h, w, levels, _lib.ptr(positions), n_desc,
                                             _lib.ptr(desc), _lib.ptr(stats), _lib.ptr(ws), ws.numel(),
                                             _lib.stream_of(x)), "dusty_swd_descriptors")
    return desc, stats


def sliced_sums(desc1, stats1, desc2, stats2, directions, dir_begin=0, dir_stride=1):
    """Stage B: (levels, D) f64 sums of |sorted1 - sorted2| for directions d = dir_begin + k dir_stride; the other
    entries are 0. directions: (levels, C*49, D) f32 on the descriptors' device."""
    levels, rows, k = desc1.shape
    c, d = k // 49, directions.shape[2]
    sums = torch.zeros(levels, d, dtype=torch.float64, device=desc1.device)
    lib = _lib.load()
    ws = _lib.workspace(lib.dusty_swd_sliced_workspace_bytes(rows, c, d), desc1.device)
    with torch.cuda.device(desc1.device):
        for level in range(levels):
            _lib.check(lib.dusty_swd_sliced(_lib.ptr(desc1[level]), _lib.ptr(desc2[level]), _lib.ptr(stats1[level]),
                                            _lib.ptr(stats2[level]), rows, c, _lib.ptr(directions[level]), d,
                                            dir_begin, d, dir_stride, _lib.ptr(sums[level]), _lib.ptr(ws), ws.numel(),
                                            _lib.stream_of(desc1)), "dusty_swd_sliced")
    return sums


def upload_draws(draws, device):
    """Positions (levels, n_desc) i32 and directions (levels, C*49, D) f32 on ``device`` in one host-to-device copy."""
    positions = torch.stack([p for p, _ in draws]).to(torch.int32)
    directions = torch.stack([dirs for _, dirs in draws]).float()
    packed = torch.cat([directions.reshape(-1), positions.reshape(-1).view(torch.float32)])
    dev = packed.pin_memory().to(device, non_blocking=True)
    nd = directions.numel()
    return dev[nd:].view(torch.int32).view(positions.shape), dev[:nd].view(directions.shape)


@torch.no_grad()
def compute_swd(image1, image2, n_pyramids=None, slice_size=7, n_descriptors=128, n_repeat_projection=128,
                proj_per_repeat=4, device=None, return_by_resolution=False, pyramid_batchsize=128):
    """SWD between two (N, C, H, W) f32 CUDA image sets, x 1e3 and averaged over the Laplacian levels; a 0-d CPU float32
    tensor, or the (levels,) per-level values with ``return_by_resolution``. The draws come from torch's global CPU
    generator exactly as the published code makes them, so ``torch.manual_seed(s)`` reproduces its positions and
    directions. ``device`` and ``pyramid_batchsize`` only shaped the published code's memory use and have no effect
    here: everything runs on the images' device.

    With torch.distributed initialised every rank must pass the same images: each rank computes the descriptors and
    the sums of the directions d = rank (mod world size), one all-gather collects the (levels, D) sums, and every rank
    reduces them in the same order, so the score is bit-identical for any number of ranks."""
    n_pyramids = _check(image1, image2, n_pyramids, slice_size, n_descriptors, n_repeat_projection, proj_per_repeat)
    n, c, h, w = image1.shape
    levels = n_pyramids + 1
    positions, directions = upload_draws(draw(h, w, c, n_pyramids, n_descriptors, n_repeat_projection,
                                              proj_per_repeat), image1.device)
    desc1, stats1 = descriptors(image1, positions, levels, n_descriptors)
    desc2, stats2 = descriptors(image2, positions, levels, n_descriptors)
    rank, world = sharding.world(None)
    sums = sliced_sums(desc1, stats1, desc2, stats2, directions, rank, world)
    d = directions.shape[2]
    if world > 1:
        gathered = sharding._all_gather_flat(sums, None).view(world, levels, d)
        owner = torch.arange(d, device=sums.device) % world
        sums = gathered.gather(0, owner.view(1, 1, d).expand(1, levels, d))[0]
    per_level = sums.cpu().numpy().sum(axis=1) / (float(d) * float(n * n_descriptors)) * 1e3
    result = torch.from_numpy(per_level.astype(np.float32))
    return result if return_by_resolution else torch.mean(result)
