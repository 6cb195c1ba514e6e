"""Parity at the shapes of BASELINE.json configs[3] and configs[4] (the 8-GPU configurations), on clouds made
by the product's own head / projection / FPS kernels, every matrix entry against the oracle."""
import numpy as np
import pytest
import torch

from helpers import head_inputs, lidar_like_clouds
from oracle import metrics as om
from oracle import native

pytestmark = pytest.mark.gpu
ULP = 2.0 ** -23
H, W = 64, 512


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def make_head(kind):
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    lidar = LiDAR(H, W, 0.9, 120.0, angle=synthetic_hdl64e_angles()).cuda()
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=1.0).cuda().eval()
    return head, lidar


def head_clouds(kind, n, seed, num_points=None):
    """n clouds through the fused head + projection (+ FPS to num_points; None keeps all H*W points, dropped
    pixels at the origin: what evaluate_reconstruction.py:124-131 feeds compute_cd)."""
    from dusty_gan_b200 import pipeline
    head, lidar = make_head(kind)
    depth, conf, u1, u2 = head_inputs(n, kind, H, W, seed, "cuda")
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    gate.fixed_noise = gate._logistic_from_uniform(u1, u2)
    if num_points is None:
        return pipeline.maskout_and_project(head, {"depth": depth, "confidence": conf}, lidar, tol=0.0)["points"]
    return pipeline.generate_points(head, {"depth": depth, "confidence": conf}, lidar, num_points, tol=0.0)[0]


def assert_matrix(M, O):
    M = M.cpu().numpy() if isinstance(M, torch.Tensor) else M
    bad = np.abs(M.astype(np.float64) - O) > ULP * np.abs(O)
    assert not bad.any(), f"{bad.sum()} of {bad.size} entries off by more than one ulp; worst rel {np.abs(M - O).max() / O.max():.2e}"


def test_configs3_dusty2_clouds_64_vs_64_every_entry_and_score():
    """configs[3] in miniature: DUSty-II head (pixel x image gates) -> projection -> FPS to 2048 -> the three
    matrices and the fused scores, 64 vs 64 clouds (the full shape is 5000 vs 5000 of the same clouds)."""
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_cov_mmd_1nna, pairwise_matrices
    gen, ref = head_clouds(2, 64, 301, 2048), head_clouds(2, 64, 302, 2048)
    Mrr, Mrg, Mgg = pairwise_matrices(gen, ref)
    g, r = gen.cpu().numpy(), ref.cpu().numpy()
    Orr, Org, Ogg = native.pairwise_cd(r, None), native.pairwise_cd(r, g), native.pairwise_cd(g, None)
    assert_matrix(Mrr, Orr); assert_matrix(Mrg, Org); assert_matrix(Mgg, Ogg)
    scores = compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
    expect = om.scores_from_matrices(Orr, Org, Ogg)
    for k, v in expect.items():
        assert scores[k] == pytest.approx(v, rel=1e-6, abs=1e-12), k
    for k in ("cov-cd", "1-nn-tp-cd", "1-nn-fp-cd", "1-nn-fn-cd", "1-nn-tn-cd"):
        assert scores[k] == expect[k], k


def test_configs4_unsampled_clouds_through_the_sorted_and_pruned_path():
    """configs[4] shape: un-sampled 64x512 clouds (32 768 points, dropped pixels at the origin) through
    chamfer_matrix's default path for them: origin points merged, kept points in k-d order, chunks pruned by
    box distance. 3 vs 2 clouds from the DUSty-I head, every entry against the oracle on all 32 768 points."""
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
    a, b = head_clouds(1, 3, 401), head_clouds(1, 2, 402)
    assert a.shape == (3, H * W, 3)
    zeros = (a == 0).all(-1).sum(1)
    assert int(zeros.min()) > 1000                        # dropped pixels are really there
    M = chamfer_matrix(a, b)
    assert_matrix(M, native.pairwise_cd(a.cpu().numpy(), b.cpu().numpy()))
    S = chamfer_matrix(a)
    assert torch.equal(S, S.t()) and bool((S.diagonal() == 0).all())
    assert_matrix(S, native.pairwise_cd(a.cpu().numpy(), None))
    # the same entries with merging off: both paths agree to the ulp
    for kw in (dict(merge_origin=False),):
        assert_matrix(chamfer_matrix(a, b, **kw), native.pairwise_cd(a.cpu().numpy(), b.cpu().numpy()))


@pytest.mark.parametrize("points,nonzero", [(32768, 32768), (32768, 32767), (32769, 32769), (32769, 30000), (32767, 32767)])
def test_sort_capacity_and_packed_index_edges(points, nonzero):
    """The shared-memory sort holds at most 32 768 keys with a 15-bit index packed in the key: clouds with
    exactly 32 768 non-zero points, one fewer (+ one origin point), and 32 769 points (which must leave the
    sorted path) -- against a smaller second set so that the oracle stays cheap."""
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
    a = lidar_like_clouds(2, points, 500 + points + nonzero, dropped=0.0, near=0.05)
    if nonzero < points:
        a[:, nonzero:] = 0.0
        a[1] = a[1][np.random.default_rng(7).permutation(points)]      # zeros anywhere, not only at the end
    b = lidar_like_clouds(2, 8192, 600 + points, dropped=0.3)
    assert_matrix(chamfer_matrix(cuda(a), cuda(b)), native.pairwise_cd(a, b))
    assert_matrix(chamfer_matrix(cuda(b), cuda(a)), native.pairwise_cd(b, a))
    assert_matrix(chamfer_matrix(cuda(a)), native.pairwise_cd(a, None))


def test_compute_cd_on_unsampled_pairs():
    """The reference's real call site for un-sampled clouds: compute_cd(points_ref, points_gen) on a batch of
    (B, H*W, 3) pairs (evaluate_reconstruction.py:124-131) through the batch front end."""
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_cd
    from dusty_gan_b200.utils.metrics.distance import chamfer_distance
    a, b = head_clouds(1, 3, 411), head_clouds(1, 3, 412)
    d1, d2 = chamfer_distance(a, b)
    o1, o2, j1, j2 = native.chamfer_forward(a.cpu().numpy(), b.cpu().numpy(), rounding="cuda")
    assert np.array_equal(d1.cpu().numpy(), o1) and np.array_equal(d2.cpu().numpy(), o2)
    # arg-mins through the sorted path's maps back to the original order: dropped pixels (zero points) report the
    # FIRST zero point of the other cloud, as the reference's lowest-index rule does
    from test_gpu_chamfer import run_forward
    _, _, i1, i2 = run_forward(a.cpu().numpy(), b.cpu().numpy())
    assert np.array_equal(i1, j1) and np.array_equal(i2, j2)
    cd = compute_cd(a, b).cpu().numpy()
    want = (o1.astype(np.float64).mean(1) + o2.astype(np.float64).mean(1))
    assert np.all(np.abs(cd - want) <= 4 * ULP * want)
