"""Chamfer kernels (through the Python mirror -> C ABI) against the oracle, the golden vectors and the
reference's own CUDA kernel (its stored outputs, plus a live run on the same GPU when oracle/_ref is present)."""
import numpy as np
import pytest
import torch

from helpers import lidar_like_clouds, rel_err, sampled_clouds
from oracle import native, refload

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5      # north_star: Chamfer within 1e-5 relative (FP32) -- the bar against the reference's CPU twin
ULP = 2.0 ** -23    # matrix entries against the CUDA-rounding oracle: per-point distances are bit-equal, the two
                    # double-accumulated means can differ in the last place of their f32 rounding


def assert_entries_equal(M, O):
    """Every entry within one ulp of the oracle's (exactly equal almost everywhere)."""
    assert np.all(np.abs(M.astype(np.float64) - O) <= ULP * np.abs(O)), np.abs(M - O).max()


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_forward(xyz1, xyz2):
    from dusty_gan_b200.utils.metrics.distance.cd.chamfer_distance import ChamferDistanceFunction
    from dusty_gan_b200 import _lib
    a, b = cuda(xyz1), cuda(xyz2)
    B, n, _ = a.shape
    m = b.shape[1]
    d1 = torch.empty(B, n, device="cuda"); d2 = torch.empty(B, m, device="cuda")
    i1 = torch.empty(B, n, dtype=torch.int32, device="cuda"); i2 = torch.empty(B, m, dtype=torch.int32, device="cuda")
    lib = _lib.load()
    nbytes = lib.dusty_chamfer_forward_workspace_bytes(B, n, m)
    ws = _lib.workspace(nbytes, a.device)
    _lib.check(lib.dusty_chamfer_forward(_lib.ptr(a), _lib.ptr(b), B, n, m, _lib.ptr(d1), _lib.ptr(d2), _lib.ptr(i1),
                                         _lib.ptr(i2), _lib.ptr(ws), nbytes, _lib.stream_of(a)), "fwd")
    torch.cuda.synchronize()
    return d1.cpu().numpy(), d2.cpu().numpy(), i1.cpu().numpy(), i2.cpu().numpy()


def check_against_oracle(xyz1, xyz2):
    """Distances AND arg-mins bit-equal to the reference CUDA kernel's restatement: the |b|^2 - 2 a.b search
    only proposes, every returned value is the reference formula's minimum (csrc/chamfer.cu, guard)."""
    d1, d2, i1, i2 = run_forward(xyz1, xyz2)
    o1, o2, j1, j2 = native.chamfer_forward(xyz1, xyz2, rounding="cuda")
    for d, o, i, j in ((d1, o1, i1, j1), (d2, o2, i2, j2)):
        assert np.array_equal(d, o), (np.abs(d - o).max(), (d != o).mean())
        assert np.array_equal(i, j), (i != j).mean()
    return d1, d2, i1, i2


def test_forward_matches_golden_inputs(golden):
    g = golden("chamfer_cpu.npz")
    d1, d2, i1, i2 = check_against_oracle(g["xyz1"], g["xyz2"])
    # the reference's CPU twin (unfused squares) agrees to rounding
    assert np.allclose(d1, g["dist1"], rtol=2e-6, atol=1e-12) and np.allclose(d2, g["dist2"], rtol=2e-6, atol=1e-12)
    assert i1[2, 0] == 149 and d1[2, 0] == 0.0           # exact hit
    assert i2[0, 3] == g["idx2"][0, 3]


@pytest.mark.parametrize("n,m", [(1, 1), (1, 40), (31, 33), (32, 64), (255, 257), (2047, 2049), (2048, 2048),
                                 (5000, 700), (700, 5000), (4097, 4100)])
def test_forward_sizes(n, m):
    rng = np.random.default_rng(n * 7919 + m)
    check_against_oracle(rng.standard_normal((2, n, 3)).astype(np.float32) * 0.3,
                         rng.standard_normal((2, m, 3)).astype(np.float32) * 0.3)


def test_forward_lidar_clouds_with_dropped_pixels():
    # un-sampled clouds keep dropped pixels as (0,0,0) points on both sides (SURVEY.md S7)
    a = lidar_like_clouds(3, 4096, 21)
    b = lidar_like_clouds(3, 4096, 22)
    d1, d2, i1, i2 = check_against_oracle(a, b)
    zero_a = np.all(a == 0, -1)
    first_zero_b = [int(np.argmax(np.all(b[k] == 0, -1))) for k in range(3)]
    for k in range(3):
        assert np.all(d1[k][zero_a[k]] == 0) and np.all(i1[k][zero_a[k]] == first_zero_b[k])


def test_forward_empty_sides():
    a = np.zeros((2, 0, 3), np.float32)
    b = np.random.default_rng(0).standard_normal((2, 17, 3)).astype(np.float32)
    d1, d2, i1, i2 = run_forward(a, b)
    assert d1.shape == (2, 0) and np.all(d2 == 0) and np.all(i2 == 0)      # outputs left zero like the reference


def reference_forward_cases(golden):
    """(xyz1, xyz2, (dist1, dist2, idx1, idx2) of the reference CUDA kernel): every case it ran on a B200 for
    tests/golden/gpu_reference_kernels.npz (oracle/gen_golden_gpu.py) and, when oracle/_ref holds the compiled
    reference, one more run live on this GPU."""
    g = golden("gpu_reference_kernels.npz")
    for i in range(3):
        b, n, m, seed = [int(v) for v in g[f"cd{i}_case"]]
        yield (sampled_clouds(b, n, seed), lidar_like_clouds(b, m, seed + 1),
               tuple(g[f"cd{i}_{k}"] for k in ("dist1", "dist2", "idx1", "idx2")))
    cd = refload.load("dustyref_cd")
    if cd is not None:
        a = sampled_clouds(4, 2048, 31); b = sampled_clouds(4, 2048, 32)
        r1 = torch.zeros(4, 2048, device="cuda"); r2 = torch.zeros(4, 2048, device="cuda")
        k1 = torch.zeros(4, 2048, dtype=torch.int32, device="cuda"); k2 = torch.zeros(4, 2048, dtype=torch.int32, device="cuda")
        cd.forward_cuda(cuda(a), cuda(b), r1, r2, k1, k2)
        torch.cuda.synchronize()
        yield a, b, tuple(t.cpu().numpy() for t in (r1, r2, k1, k2))


def test_forward_against_reference_cuda_kernel(golden):
    for a, b, want in reference_forward_cases(golden):
        for got in (run_forward(a, b),
                    native.chamfer_forward(a, b, rounding="cuda")):    # the oracle's CUDA-rounding restatement IS the reference kernel, bit for bit
            for x, r in zip(got, want):
                assert np.array_equal(x, r), (a.shape, b.shape)


def test_autograd_wrapper_and_backward(golden):
    from dusty_gan_b200.utils.metrics.distance import chamfer_distance
    g = golden("chamfer_cpu.npz")
    a = cuda(g["xyz1"]).requires_grad_(True); b = cuda(g["xyz2"]).requires_grad_(True)
    d1, d2 = chamfer_distance(a, b)
    ((d1 * cuda(g["w1"])).sum() + (d2 * cuda(g["w2"])).sum()).backward()
    o1, o2, j1, j2 = native.chamfer_forward(g["xyz1"], g["xyz2"], rounding="cuda")
    gx1, gx2 = native.chamfer_backward(g["xyz1"], g["xyz2"], g["w1"], g["w2"], j1, j2)
    assert np.allclose(a.grad.cpu().numpy(), gx1, rtol=1e-5, atol=1e-7)
    assert np.allclose(b.grad.cpu().numpy(), gx2, rtol=1e-5, atol=1e-7)
    assert np.allclose(a.grad.cpu().numpy(), g["grad1"], rtol=1e-4, atol=1e-6)


def test_rejects_cpu_tensors():
    from dusty_gan_b200.utils.metrics.distance import chamfer_distance
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        chamfer_distance(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))


# ------------------------------------------------------------------ pairwise matrix ----------------
def matrix(a, b=None, **kw):
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
    M = chamfer_matrix(cuda(a), None if b is None else cuda(b), **kw)
    torch.cuda.synchronize()
    return M.cpu().numpy()


@pytest.mark.parametrize("P", [128, 512, 600, 2048])
def test_matrix_against_oracle(P):
    a = sampled_clouds(7, P, 100 + P); b = sampled_clouds(5, P, 200 + P)
    M = matrix(a, b)
    assert_entries_equal(M, native.pairwise_cd(a, b, rounding="cuda"))
    S = matrix(a)
    assert np.array_equal(S, S.T) and np.all(np.diag(S) == 0)
    assert_entries_equal(S, native.pairwise_cd(a, None, rounding="cuda"))


def test_matrix_unequal_point_counts_and_multi_tile():
    a = sampled_clouds(3, 5000, 301); b = sampled_clouds(4, 2500, 302)
    M = matrix(a, b)
    assert_entries_equal(M, native.pairwise_cd(a, b, rounding="cuda"))


@pytest.mark.parametrize("shape", [(3, 4, 5000, 5000), (2, 3, 6000, 4500), (2, 2, 333, 70)])
def test_matrix_merged_origin_points(shape):
    """Un-sampled clouds (SURVEY.md S7): collapsing every cloud's (0,0,0) points into one weighted point
    must give the matrix of the plain kernel (values within double-sum reassociation, i.e. <= 1 ulp of f32)
    and the oracle's within the tolerance. Includes clouds without zeros, all zeros, -0.0 and one zero."""
    na, nb, pa, pb = shape
    a = lidar_like_clouds(na, pa, 601, dropped=0.5); b = lidar_like_clouds(nb, pb, 602, dropped=0.35)
    a[0][np.all(a[0] == 0, axis=1)] = lidar_like_clouds(1, pa, 603, dropped=0.0)[0][np.all(a[0] == 0, axis=1)]  # no zeros
    b[0] = 0.0                                                                                                # only zeros
    b[1][np.all(b[1] == 0, axis=1)] *= -1.0                                                                   # -0.0 is the origin too
    if na > 2:
        a[2, 1:] = lidar_like_clouds(1, pa, 604, dropped=0.0)[0, 1:]; a[2, 0] = 0.0                           # a single zero
    plain = matrix(a, b, merge_origin=False)
    merged = matrix(a, b, merge_origin=True)
    O = native.pairwise_cd(a, b, rounding="cuda")
    assert np.all(np.abs(merged - plain) <= ULP * np.abs(plain))
    assert np.all(np.abs(merged - O) <= ULP * np.abs(O)) and np.all(np.abs(plain - O) <= ULP * np.abs(O))
    if pa == pb:
        S0 = matrix(a, merge_origin=False); S1 = matrix(a, merge_origin=True)
        assert np.array_equal(S1, S1.T) and np.all(np.diag(S1) == 0)
        assert np.all(np.abs(S1 - S0) <= 2.0 ** -23 * np.abs(S0))
        # row shards take the same path: bit-identical to the full launch
        from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
        sub = chamfer_matrix(cuda(a), cuda(b), rows=(1, na, 2), merge_origin=True).cpu().numpy()
        assert np.array_equal(sub[1::2], merged[1::2])


def test_matrix_sorted_search_is_the_default_above_256_points():
    from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
    assert M.MERGE_ORIGIN_ABOVE == 256
    a = lidar_like_clouds(2, 4100, 611, dropped=0.5)
    assert np.array_equal(matrix(a), matrix(a, merge_origin=True))
    s = sampled_clouds(3, 2048, 612)                        # the evaluation's own shape: k-d order + resident-pair kernel
    S1, S0 = matrix(s), matrix(s, merge_origin=False)
    assert np.array_equal(S1, matrix(s, merge_origin=True))
    assert np.all(np.abs(S1 - S0) <= ULP * S0)              # same distances, the two means summed in another order
    small = sampled_clouds(3, 256, 613)                     # at and below 256 points: the brute-force kernel
    assert np.array_equal(matrix(small), matrix(small, merge_origin=False))


@pytest.mark.parametrize("pa,pb,dropped", [(257, 300, 0.0), (512, 512, 0.0), (1000, 777, 0.3), (2047, 2048, 0.0),
                                            (2048, 2048, 0.4), (2048, 65, 0.5), (33, 2048, 0.2), (2048, 2049, 0.0)])
def test_matrix_resident_pair_kernel_against_oracle(pa, pb, dropped):
    """Clouds of at most 2048 points with merged origins: k-d ordered by prep_sort_kernel<true>, searched by
    nn_pair_split_kernel (both clouds in shared memory, best-first chunk walk). Every entry against the CUDA-rounding
    oracle, for point counts that are not multiples of the 32-row groups or the 32-candidate chunks, clouds with
    and without dropped (0,0,0) points, degenerate clouds, and 2049 points (one past the kernel's capacity: the
    two-level walk nn_walk_split_kernel). Two runs are bit-identical although warps take their row groups dynamically."""
    a = lidar_like_clouds(4, pa, 700 + pa, dropped=dropped); b = lidar_like_clouds(3, pb, 800 + pb, dropped=dropped)
    b[1] = b[1][0]                                           # every point the same
    if dropped:
        a[1] = 0.0                                           # only origin points
    M = matrix(a, b, merge_origin=True)
    assert_entries_equal(M, native.pairwise_cd(a, b, rounding="cuda"))
    assert np.array_equal(M, matrix(a, b, merge_origin=True))
    if pa == pb:
        S = matrix(a, merge_origin=True)
        assert np.array_equal(S, S.T) and np.all(np.diag(S) == 0)
        assert_entries_equal(S, native.pairwise_cd(a, None, rounding="cuda"))
        from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
        sub = chamfer_matrix(cuda(a), None, rows=(1, 4, 2), compact_rows=True, merge_origin=True).cpu().numpy()
        assert np.array_equal(sub[0, 1:], S[1, 1:]) and np.array_equal(sub[1, 3:], S[3, 3:])


def test_matrix_resident_pair_kernel_on_clustered_and_collinear_clouds():
    """k-d splits on clouds whose boxes degenerate: all points on a line (two zero-extent axes), many duplicates (equal
    sort keys broken by index), two far-apart clusters (empty space inside the top-level boxes)."""
    rng = np.random.default_rng(9)
    line = np.zeros((2, 1024, 3), np.float32); line[:, :, 0] = rng.uniform(-1, 1, (2, 1024))
    dup = np.repeat(rng.uniform(-0.5, 0.5, (2, 16, 3)).astype(np.float32), 64, axis=1)
    two = np.concatenate([rng.normal(0.8, 0.01, (2, 700, 3)), rng.normal(-0.8, 0.01, (2, 324, 3))], axis=1).astype(np.float32)
    for a, b in ((line, dup), (dup, two), (two, line)):
        assert_entries_equal(matrix(a, b, merge_origin=True), native.pairwise_cd(a, b, rounding="cuda"))


def test_matrix_golden_reference_driver(golden):
    g = golden("metrics_cpu.npz")
    assert rel_err(matrix(g["ref"], g["gen"]), g["M_rg"]).max() <= REL_TOL
    Mrr = matrix(g["ref"])
    assert rel_err(Mrr, g["M_rr"])[~np.eye(12, dtype=bool)].max() <= REL_TOL and np.all(np.diag(Mrr) == 0)
    Md = matrix(g["ref"], g["gen_dup"])
    assert Md[5, 3] == 0.0


def test_matrix_row_shards_are_bit_identical():
    a = sampled_clouds(23, 512, 401)
    full = matrix(a)
    G = 4
    parts = []
    for r in range(G):
        cap = (23 + G - 1) // G
        blk = torch.zeros(cap, 23, device="cuda")
        from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
        chamfer_matrix(cuda(a), None, rows=(r, 23, G), compact_rows=True, out=blk)
        parts.append(blk)
    from dusty_gan_b200 import sharding
    S = sharding.assemble_symmetric(torch.stack(parts), 23).cpu().numpy()
    assert np.array_equal(S, full)
    b = sampled_clouds(9, 512, 402)
    rect = matrix(a, b)
    sub = matrix(a, b, rows=(4, 17, 3))
    rows = list(range(4, 17, 3))
    assert np.array_equal(sub[rows], rect[rows]) and np.all(np.delete(sub, rows, 0) == 0)


def test_matrix_full_size_properties():
    """Config 3 shape (1000 vs 1000 clouds, 2048 points): the stacked symmetric matrix in one launch,
    checked through size-independent properties plus spot checks against the oracle."""
    ref = sampled_clouds(1000, 2048, 501); gen = sampled_clouds(1000, 2048, 502)
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import pairwise_matrices
    Mrr, Mrg, Mgg = [m.cpu().numpy() for m in pairwise_matrices(cuda(gen), cuda(ref))]
    assert Mrr.shape == Mrg.shape == Mgg.shape == (1000, 1000)
    for S in (Mrr, Mgg):
        assert np.array_equal(S, S.T) and np.all(np.diag(S) == 0)
        assert np.all(S[~np.eye(1000, dtype=bool)] > 0)
    assert np.all(np.isfinite(Mrg)) and np.all(Mrg > 0)
    rng = np.random.default_rng(9)
    for _ in range(6):
        i, j = rng.integers(0, 1000, 2)
        o = native.pairwise_cd(ref[i:i + 1], gen[j:j + 1], rounding="cuda")[0, 0]
        assert abs(Mrg[i, j] - o) <= ULP * o
        o = native.pairwise_cd(gen[i:i + 1], gen[j:j + 1], rounding="cuda")[0, 0]
        assert abs(Mgg[i, j] - o) <= ULP * o


def test_forward_against_reference_cuda_golden(golden):
    g = golden("gpu_reference_kernels.npz")
    for i in range(3):
        b, n, m, seed = [int(v) for v in g[f"cd{i}_case"]]
        a = sampled_clouds(b, n, seed); c = lidar_like_clouds(b, m, seed + 1)
        d1, d2, i1, i2 = run_forward(a, c)
        for d, r, ix, k in ((d1, g[f"cd{i}_dist1"], i1, g[f"cd{i}_idx1"]), (d2, g[f"cd{i}_dist2"], i2, g[f"cd{i}_idx2"])):
            assert np.array_equal(d, r) and np.array_equal(ix, k)      # the reference kernel's own output on a B200


@pytest.mark.parametrize("P,merge", [(700, True), (3000, True), (700, False)])
def test_matrix_prepared_flag_reuses_the_scan_copies(P, merge):
    """DUSTY_MATRIX_PREPARED: a second call on the same workspace skips the scan-format / k-d preparation of the clouds
    (resident-pair kernel at 700 points, walk kernel at 3000, brute-force kernel without the merge flag)."""
    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import chamfer_matrix
    a, b = cuda(lidar_like_clouds(5, P, 901, dropped=0.3)), cuda(lidar_like_clouds(4, P, 902, dropped=0.3))
    lib = _lib.load()
    flags = _lib.MATRIX_MERGE_ORIGIN if merge else 0
    nbytes = lib.dusty_chamfer_matrix_workspace_bytes(5, P, 4, P)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    M = torch.zeros(5, 4, device="cuda")
    launches = _lib.launch_count()
    _lib.check(lib.dusty_chamfer_matrix(_lib.ptr(a), 5, P, _lib.ptr(b), 4, P, 0, 2, 1, flags, _lib.ptr(M), 4, _lib.ptr(ws), nbytes,
                                        _lib.stream_of(a)), "first")
    first = _lib.launch_count() - launches
    _lib.check(lib.dusty_chamfer_matrix(_lib.ptr(a), 5, P, _lib.ptr(b), 4, P, 2, 5, 1, flags | _lib.MATRIX_PREPARED, _lib.ptr(M), 4,
                                        _lib.ptr(ws), nbytes, _lib.stream_of(a)), "second")
    assert _lib.launch_count() - launches - first == 1 and first >= 2      # the second call is the search kernel alone
    torch.cuda.synchronize()
    assert torch.equal(M, chamfer_matrix(a, b, merge_origin=merge))
