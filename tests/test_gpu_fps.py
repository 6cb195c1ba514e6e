"""FPS kernel: indices bit-exact against the oracle's thread-by-thread replay of the reference
kernel and against the reference's own CUDA kernel (its stored outputs, plus a live run on this GPU
when oracle/_ref is present)."""
import numpy as np
import pytest
import torch

from helpers import lidar_like_clouds
from oracle import native, refload

pytestmark = pytest.mark.gpu


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def fps_gpu(x, m):
    from dusty_gan_b200.utils.sampling.fps import furthest_point_sampling
    idx = furthest_point_sampling(cuda(x), m)
    torch.cuda.synchronize()
    assert idx.dtype == torch.int32
    return idx.cpu().numpy()


def test_full_resolution_clouds_bit_exact():
    x = lidar_like_clouds(3, 32768, 7)                  # 64x512 range images, ~60 % eligible
    assert np.array_equal(fps_gpu(x, 2048), native.fps(x, 2048))


@pytest.mark.parametrize("n,m", [(1, 1), (1, 4), (2, 2), (3, 3), (31, 8), (33, 33), (511, 64), (512, 512), (513, 100),
                                 (1000, 1000), (2048, 512), (5000, 300), (20000, 128)])
def test_sizes_bit_exact(n, m):
    x = lidar_like_clouds(2, n, 1000 + n, dropped=0.2, near=0.1)
    assert np.array_equal(fps_gpu(x, m), native.fps(x, m))


def test_all_points_eligible_dense_cloud():
    x = lidar_like_clouds(2, 32768, 8, dropped=0.0, near=0.0)      # exceeds the smem staging capacity
    assert np.array_equal(fps_gpu(x, 512), native.fps(x, 512))


def test_more_points_than_register_capacity():
    x = lidar_like_clouds(1, 40000, 9, dropped=0.1, near=0.05)
    assert np.array_equal(fps_gpu(x, 96), native.fps(x, 96))


def test_degenerate_inputs():
    # literal random-init generator: every range inside the exclusion radius => index 0 repeated (trap T1)
    x = (np.random.default_rng(3).standard_normal((2, 4096, 3)) * 0.005).astype(np.float32)
    assert np.all(fps_gpu(x, 64) == 0)
    # dropped seed pixel, coincident points, fewer distinct points than samples: the tie rule decides
    n = 1500
    x = np.zeros((1, n, 3), np.float32)
    x[0, [5, 77, 517, 1101, 300, 1401]] = [0.3, 0.1, 0.05]
    x[0, 300] = [0.5, -0.2, 0.01]
    assert np.array_equal(fps_gpu(x, 9), native.fps(x, 9))
    # exact ties between different positions (mirror-symmetric pairs at equal distance from the seed)
    rng = np.random.default_rng(4)
    half = rng.uniform(0.05, 0.5, (600, 3)).astype(np.float32)
    x = np.concatenate([half, half * np.array([1, -1, 1], np.float32)])[None]
    x[0, 0] = [0.2, 0.0, 0.1]
    assert np.array_equal(fps_gpu(x, 200), native.fps(x, 200))


def test_downsample_and_gather():
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds, gather_operation, furthest_point_sampling
    x = lidar_like_clouds(2, 8192, 12)
    t = cuda(x)
    sub = downsample_point_clouds(t, 256)
    ref_sub, ref_idx = native.downsample_point_clouds(x, 256)
    assert sub.shape == (2, 256, 3) and np.array_equal(sub.cpu().numpy(), ref_sub)
    idx = furthest_point_sampling(t, 256)
    feats = t.transpose(1, 2).contiguous().requires_grad_(True)
    g = gather_operation(feats, idx)
    assert np.array_equal(g.detach().cpu().numpy(), native.gather_points(x.transpose(0, 2, 1), ref_idx))
    w = torch.rand_like(g)
    (g * w).sum().backward()
    expect = torch.zeros_like(feats).scatter_add_(2, idx.long()[:, None, :].expand(-1, 3, -1), w)
    assert torch.allclose(feats.grad, expect)


def reference_kernel_cases(golden):
    """(clouds, samples, the reference CUDA kernel's indices): every case it ran on a B200 for
    tests/golden/gpu_reference_kernels.npz (oracle/gen_golden_gpu.py) and, when oracle/_ref holds the
    compiled reference, three more run live on this GPU."""
    g = golden("gpu_reference_kernels.npz")
    i = 0
    while f"fps{i}_case" in g:
        b, n, m, seed, dropped, near = [int(v) for v in g[f"fps{i}_case"]]
        yield lidar_like_clouds(b, n, seed, dropped=dropped / 1000, near=near / 1000), m, g[f"fps{i}_idx"]
        i += 1
    yield g["fps_deg_input"], 200, g["fps_deg_idx"]
    ref = refload.load("dustyref_fps")
    if ref is not None:
        for n, m, seed in ((32768, 2048, 21), (5000, 512, 22), (700, 64, 23)):
            x = lidar_like_clouds(3, n, seed)
            r = ref.furthest_point_sampling(cuda(x), m)
            torch.cuda.synchronize()
            yield x, m, r.cpu().numpy()


def test_against_reference_cuda_kernel(golden):
    for x, m, want in reference_kernel_cases(golden):
        assert np.array_equal(fps_gpu(x, m), want), (x.shape, m)
        assert np.array_equal(native.fps(x, m), want), (x.shape, m)     # pins the oracle too


def test_against_reference_cuda_golden(golden):
    """The committed outputs of the reference's CUDA kernel (oracle/gen_golden_gpu.py on a B200)."""
    g = golden("gpu_reference_kernels.npz")
    i = 0
    while f"fps{i}_case" in g:
        b, n, m, seed, dropped, near = [int(v) for v in g[f"fps{i}_case"]]
        x = lidar_like_clouds(b, n, seed, dropped=dropped / 1000, near=near / 1000)
        assert np.array_equal(fps_gpu(x, m), g[f"fps{i}_idx"]), g[f"fps{i}_case"]
        i += 1
    assert np.array_equal(fps_gpu(g["fps_deg_input"], 200), g["fps_deg_idx"])


def test_duplicate_points_tie_inside_one_lane():
    """Exact duplicates that land next to each other after the spatial sort: one lane then holds two
    candidates with the same distance, the path where the tie key decides (and must stay warp-uniform)."""
    base = lidar_like_clouds(2, 4000, 31, dropped=0.1, near=0.05)
    x = np.repeat(base, 3, axis=1)                     # every point three times
    assert np.array_equal(fps_gpu(x, 300), native.fps(x, 300))
    y = lidar_like_clouds(300, 2048, 32, dropped=0.3, near=0.1)   # more clouds than SMs
    y[:, 1::2] = y[:, ::2]                             # pairs of duplicates
    assert np.array_equal(fps_gpu(y, 128), native.fps(y, 128))


def kitti_like_dense(clouds, seed):
    """Un-sampled 64x512 clouds with ~28 k eligible points (|p|^2 > 1e-3), what real KITTI scans give (SURVEY.md H3):
    more than the 17 792 points whose coordinates fit one SM's shared memory and more than the 16 384 running
    distances the throughput variant keeps on chip."""
    return lidar_like_clouds(clouds, 32768, seed, dropped=0.12, near=0.03)


def test_kitti_like_28k_eligible_points_every_variant(monkeypatch):
    x = kitti_like_dense(3, 41)
    elig = ((x.astype(np.float64) ** 2).sum(-1) > 1e-3).sum(1)
    assert elig.min() > 27000
    want = native.fps(x, 2048)
    assert np.array_equal(fps_gpu(x, 2048), want)                      # one cloud per SM, tail of the coordinates in L2
    ref = refload.load("dustyref_fps")
    if ref is not None:
        assert np.array_equal(ref.furthest_point_sampling(cuda(x), 2048).cpu().numpy(), want)
    many = np.concatenate([x, kitti_like_dense(150, 42)])              # > 148 clouds: three per SM, distances on chip + overflow
    got = fps_gpu(many, 512)
    assert np.array_equal(got[:3], native.fps(x, 512))
    assert np.array_equal(got[3:60], fps_gpu(many[3:60], 512))         # same indices from the one-cloud-per-SM variant
