"""FPS at the evaluation's shape, at every capacity edge of csrc/fps.cu and on degenerate clouds, on each kernel.

Indices must be bit-equal to ``oracle.native.fps``, the thread-by-thread replay of the reference kernel that
``test_gpu_fps.py::test_against_reference_cuda_golden`` pins to the reference's CUDA kernel, and, when oracle/_ref
holds the compiled reference, to that kernel run live. Every case is written down as data: eligible points E, points
per cloud n, samples m, clouds per launch b and the kernel ``dusty_fps`` launches for them. A failure names all five.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from conftest import ROOT
from helpers import lidar_like_clouds
from oracle import native, refload
from test_gpu_fps import kitti_like_dense

pytestmark = pytest.mark.gpu

# Capacities of csrc/fps.cu. Each edge below is written in terms of the constant it belongs to, so that a change
# to a constant moves the edge with it.
BUCKET = 128          # BUCKET: points per bucket of the pruned and multi kernels (32 lanes x 4)
MT_DCAP = 14336       # MT_DCAP: running distances fps_multi_kernel<true> keeps in shared memory
PR_CAP = 17792        # PR_CAP: coordinates fps_pruned_kernel stages in shared memory
SMEM_CAP = 18432      # SMEM_CAP: coordinates fps_flat_kernel stages in shared memory
ELIST = 1536          # PR_ELIST / MT_ELIST: winners kept in shared memory; later samples go through idx[]
REG_CAP = 32768       # REG_CAP: register-resident distances; larger clouds take fps_flat_kernel<false>
NUM_SMS = 148         # kNumSMs: more clouds than this take fps_multi_kernel
TIE_BLOCK = 512       # the reference's block size: tie key block T = min(2^floor(log2 n), TIE_BLOCK)

EVAL_M = 2048         # samples per cloud of the evaluation (bench.py configs 2 and 3)

# Exact eligible counts, each at the edge of the constant it names.
E_EDGES = [
    0, 1, 2,                                   # no eligible point (index 0 throughout), one, two
    BUCKET - 1, BUCKET, BUCKET + 1,            # one bucket, partly and exactly full, then a second one
    MT_DCAP - 1, MT_DCAP, MT_DCAP + 1,         # multi kernel: last distance on chip, first one in the workspace
    REG_CAP // 2,                              # 16 384 = 128 buckets: half the register-resident capacity
    PR_CAP - 1, PR_CAP, PR_CAP + 1,            # pruned kernel: last coordinate in shared memory, first one in L2
    SMEM_CAP - 1, SMEM_CAP, SMEM_CAP + 1,      # flat kernel: the same for its staging buffer
]
# Points per cloud for the exact-count clouds: the register capacity, one above it (flat kernel with distances in the
# workspace), and two sizes that are not multiples of BUCKET.
N_EDGES = [REG_CAP, REG_CAP + 1, 2049, 16383]
# Sample counts around the on-chip winner list, plus the smallest ones.
M_EDGES = [1, 2, ELIST - 1, ELIST, ELIST + 1, EVAL_M]
# Points per cloud where the tie-block size T = min(2^floor(log2 n), TIE_BLOCK) changes (T = 256, 512, 512 and
# 512 throughout the second triple: the key's second digit, k div T, gains a value).
T_EDGES = [TIE_BLOCK - 1, TIE_BLOCK, TIE_BLOCK + 1, 2 * TIE_BLOCK - 1, 2 * TIE_BLOCK, 2 * TIE_BLOCK + 1]


def kernel_for(b, n, algo=None):
    """The kernel dusty_fps launches for b clouds of n points, with DUSTY_FPS_ALGO=algo."""
    if n > REG_CAP:
        return "fps_flat_kernel<false>"
    if algo == "flat":
        return "fps_flat_kernel<true>"
    if algo == "l2":
        return "fps_multi_kernel<false>"
    if algo == "multi" or (algo != "single" and b > NUM_SMS):
        return "fps_multi_kernel<true>"
    return "fps_pruned_kernel"


def eligible(x):
    """Eligible points per cloud, (double)|p|^2 > 1e-3, in float64 (exact counts only away from the threshold)."""
    return ((np.asarray(x, np.float64) ** 2).sum(-1) > 1e-3).sum(-1)


def fps(x, m):
    """Indices (b, m) from the library; x is a numpy array or a CUDA tensor."""
    from dusty_gan_b200.utils.sampling.fps import furthest_point_sampling
    t = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x)).cuda()
    idx = furthest_point_sampling(t, m)
    assert idx.dtype == torch.int32 and idx.shape == (t.shape[0], m)
    return idx.cpu().numpy()


def oracle(x, m):
    """oracle.native.fps, one cloud per thread (the C replay releases the GIL; it takes ~0.3 s per 32 768 x 2048)."""
    x = np.ascontiguousarray(x, np.float32)
    native.lib()
    with ThreadPoolExecutor(max(1, min(len(x), os.cpu_count() or 1))) as pool:
        return np.concatenate(list(pool.map(lambda c: native.fps(x[c:c + 1], m), range(len(x)))))


def case(E, n, m, b, kernel, what=""):
    return f"E={E} n={n} m={m} b={b} expected kernel {kernel}" + (f" ({what})" if what else "")


def check(got, want, labels, against="oracle"):
    """got/want (clouds, m); labels: one case() string per cloud, or one for all of them."""
    assert got.shape == want.shape, (got.shape, want.shape, labels if isinstance(labels, str) else labels[0])
    bad = np.flatnonzero((got != want).any(1))
    if len(bad):
        c = bad[0]
        j = int(np.flatnonzero(got[c] != want[c])[0])
        label = labels if isinstance(labels, str) else labels[c]
        raise AssertionError(f"{label}: {len(bad)} of {len(got)} clouds differ from the {against}; first: cloud {c}, "
                             f"sample {j}: got index {got[c, j]}, {against} {want[c, j]}")


def check_alone_and_in_149(x, m, want, what="", E=None):
    """Clouds x (b <= 148) on their own, where dusty_fps runs fps_pruned_kernel, and as the last b clouds of a batch of
    149, where it runs fps_multi_kernel<true> (the last of them is the 149th CTA). Both must give `want`; the filler
    clouds in front must give what the pruned kernel gives for them."""
    b, n, _ = x.shape
    assert b <= NUM_SMS
    E = eligible(x) if E is None else E
    got = fps(x, m)
    check(got, want, [case(E[c], n, m, b, kernel_for(b, n), what) for c in range(b)])
    fill = lidar_like_clouds(NUM_SMS + 1 - b, n, 7 * n + m)
    big = np.concatenate([fill, x])
    got = fps(big, m)
    B = len(big)
    check(got[len(fill):], want, [case(E[c], n, m, B, kernel_for(B, n), what + f", cloud {len(fill) + c} of {B}")
                                  for c in range(b)])
    check(got[:len(fill)], fps(fill, m), case("~", n, m, B, kernel_for(B, n), "filler clouds"), "pruned kernel")


# ---------------------------------------------------------------------------------------------------------------------
# cloud makers
# ---------------------------------------------------------------------------------------------------------------------
def exact_eligible_clouds(counts, n, seed):
    """One cloud per entry of `counts`: a cloud of n eligible points (lidar_like_clouds without dropped or near
    points: |p|^2 >= 0.035^2, 22 % above the threshold) in which all but E randomly chosen points are zeroed."""
    x = lidar_like_clouds(len(counts), n, seed, dropped=0.0, near=0.0)
    rng = np.random.default_rng(seed)
    for c, E in enumerate(counts):
        drop = np.ones(n, bool)
        drop[rng.choice(n, E, replace=False)] = False
        x[c, drop] = 0.0
    assert np.array_equal(eligible(x), counts)
    return x


def lattice_clouds(b, n, seed):
    """Points on a grid of step 1/64: every coordinate, difference and squared distance is exact in float32, so
    different points at the same distance from a centre, duplicates and ties across buckets are common. The grid
    points nearest the origin are not eligible."""
    g = np.random.default_rng(seed).integers(-20, 21, (b, n, 3))
    return (g / 64.0).astype(np.float32)


def few_distinct_clouds(b, n, distinct, seed):
    """n points drawn from `distinct` eligible ones, so m > distinct samples end in ties that only the key decides."""
    base = lidar_like_clouds(b, distinct, seed, dropped=0.0, near=0.0)
    pick = np.random.default_rng(seed).integers(0, distinct, (b, n))
    pick[:, :distinct] = np.arange(distinct)
    return np.take_along_axis(base, pick[..., None], 1)


def paired_clouds(b, n, seed):
    """Every point twice (the copies at random positions): ties inside and across buckets from the first sample on."""
    half = lidar_like_clouds(b, (n + 1) // 2, seed, dropped=0.1, near=0.05)
    perm = np.random.default_rng(seed).permuted(np.tile(np.arange(half.shape[1]), (b, 2)), axis=1)[:, :n]
    return np.take_along_axis(half, perm[..., None], 1)


def t1_clouds(b, n, seed):
    """An untrained generator (SURVEY trap T1): every point inside the exclusion radius."""
    return (np.random.default_rng(seed).standard_normal((b, n, 3)) * 0.004).astype(np.float32)


def threshold_points():
    """(above, below): points whose reference-rounded magnitude fmaf(z,z,fmaf(x,x,y*y)) is the smallest float32
    above 1e-3 (in double) and the largest one at or below it. The first are eligible, the second are not; comparing
    the magnitude with 1e-3f (= the first value) instead of 1e-3 in double would drop the first ones.

    Points (x, 0, z) with z = k 2^-20: x*x is exact in double, z*z + round(x*x) too (31 significant bits), so one
    rounding of each double value to float32 is the kernel's fmaf. Each (x, z) gives eight points (x or y axis, signs).
    """
    above = np.float32(1e-3)
    below = np.nextafter(above, np.float32(0))
    assert float(below) <= 1e-3 < float(above)
    found = {above: [], below: []}
    x0 = np.float32(np.sqrt(1e-3))
    for i in range(400):
        x = np.float32(x0 - i * np.spacing(x0))
        inner = np.float32(np.float64(x) * np.float64(x))
        for k in range(1, 1024):
            z = np.float32(k * 2.0 ** -20)
            mag = np.float32(np.float64(z) * np.float64(z) + np.float64(inner))
            if mag in found and len(found[mag]) < 24:
                found[mag].append((x, z))
    out = []
    for key in (above, below):
        assert len(found[key]) == 24, key
        pts = []
        for x, z in found[key]:
            for s in (1, -1):
                for t in (1, -1):
                    pts += [(s * x, 0.0, t * z), (0.0, s * x, t * z)]
        out.append(np.array(pts, np.float32))
    return out


def threshold_clouds(b, n, seed):
    """Dropped pixels at the origin (index 0 among them), 192 points just above the eligibility threshold, 192 just at
    or below it, and 100 ordinary points, at random positions. Returns (clouds, above mask, below mask)."""
    above, below = threshold_points()
    rng = np.random.default_rng(seed)
    x = np.zeros((b, n, 3), np.float32)
    is_above = np.zeros((b, n), bool)
    is_below = np.zeros((b, n), bool)
    far = lidar_like_clouds(b, 100, seed, dropped=0.0, near=0.0)
    for c in range(b):
        pos = 1 + rng.permutation(n - 1)[: len(above) + len(below) + 100]
        a, w, f = np.split(pos, [len(above), len(above) + len(below)])
        x[c, a], x[c, w], x[c, f] = above, below, far[c]
        is_above[c, a] = True
        is_below[c, w] = True
    return x, is_above, is_below


COINCIDENT = np.array([0.2, 0.1, -0.05], np.float32)


def dropped_seed_clouds(b, n, seed):
    """S5 on every cloud: index 0 dropped (still the first centre), one point that is picked first and eight
    coincident eligible points at random positions, a pure tie that only the key decides for the second pick."""
    rng = np.random.default_rng(seed)
    x = np.zeros((b, n, 3), np.float32)
    for c in range(b):
        ks = 1 + rng.choice(n - 1, 9, replace=False)
        x[c, ks[:8]] = COINCIDENT
        x[c, ks[8]] = [-0.3, 0.2, 0.1]
    return x


def tie_key(k, n):
    T = min(1 << (n.bit_length() - 1), TIE_BLOCK)
    L = T.bit_length() - 1
    return (int(format(k % T, f"0{L}b")[::-1], 2) if L else 0, k // T)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the evaluation's shape: 1000 clouds of 32 768 points -> 2048 on fps_multi_kernel<true>
# ---------------------------------------------------------------------------------------------------------------------
EVAL_CLOUDS = 1000
# the first and last clouds, both sides of each wave of CTAs (148 SMs; three multi CTAs per SM: 444 per wave)
EVAL_SAMPLE = [0, 1, 147, 148, 149, 150, 295, 296, 297, 443, 444, 445, 591, 592, 887, 888, 998, 999]
KITTI_CLOUDS = 300
KITTI_SAMPLE = [0, 1, 147, 148, 149, 150, 295, 296, 297, 298, 299]


def bench_clouds(n_clouds):
    """Un-sampled 64x512 clouds made the way bench.py makes them: backbone-like outputs through the DUSty-I head and
    the projection (about 15.6 k eligible points per cloud, more than MT_DCAP)."""
    import bench
    dev = torch.device("cuda")
    return bench.make_clouds(n_clouds, 4, bench.make_head(1, dev), bench.make_lidar(dev), dev, full_resolution=True)


@pytest.mark.parametrize("source", ["bench", "kitti_like"])
def test_evaluation_shape(source):
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    if source == "bench":
        x, sample = bench_clouds(EVAL_CLOUDS), EVAL_SAMPLE
    else:                                                     # ~28 k eligible: beyond PR_CAP and MT_DCAP
        x, sample = torch.from_numpy(kitti_like_dense(KITTI_CLOUDS, 43)).cuda(), KITTI_SAMPLE
    B, n, _ = x.shape
    assert n == REG_CAP and B > NUM_SMS
    idx = fps(x, EVAL_M)
    xs = x[sample].cpu().numpy()
    E = eligible(xs)
    assert (E > MT_DCAP).any(), E                            # distances overflow into the workspace
    want = oracle(xs, EVAL_M)
    check(idx[sample], want, [case(E[c], n, EVAL_M, B, kernel_for(B, n), f"cloud {s}") for c, s in enumerate(sample)])
    ref = refload.load("dustyref_fps")
    if ref is not None:
        live = ref.furthest_point_sampling(x[sample].contiguous(), EVAL_M).cpu().numpy()
        check(idx[sample], live, case("~", n, EVAL_M, B, kernel_for(B, n)), "reference kernel")
    # every cloud against the one-cloud-per-SM kernel, in launches of at most NUM_SMS clouds
    for c0 in range(0, B, NUM_SMS):
        part = x[c0:c0 + NUM_SMS]
        check(idx[c0:c0 + NUM_SMS], fps(part, EVAL_M),
              case("~", n, EVAL_M, B, kernel_for(B, n), f"clouds {c0}.. against {kernel_for(len(part), n)}"),
              "pruned kernel")
    # the fused gather returns exactly the sampled points
    pts = downsample_point_clouds(x, EVAL_M)
    gathered = torch.gather(x, 1, torch.from_numpy(idx).cuda().long()[..., None].expand(-1, -1, 3))
    assert torch.equal(pts, gathered)


# ---------------------------------------------------------------------------------------------------------------------
# 2. exact eligible counts at every capacity edge, on both default kernels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", N_EDGES)
def test_exact_eligible_counts(n):
    counts = [E for E in E_EDGES if E <= n]
    x = exact_eligible_clouds(counts, n, 100 + n)
    want = oracle(x, EVAL_M)
    check_alone_and_in_149(x, EVAL_M, want, "exact eligible count", np.array(counts))
    for c, E in enumerate(counts):                 # fewer eligible points than samples: all of them, then repeats
        if 0 < E < EVAL_M:
            assert len(np.unique(want[c])) == E + (x[c, 0] == 0).all(), case(E, n, EVAL_M, len(counts), "oracle")


# ---------------------------------------------------------------------------------------------------------------------
# 3. sample counts and ties
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lidar_2048():
    """Three evaluation-sized clouds and the oracle's first 2048 samples; FPS with fewer samples is a prefix."""
    x = np.concatenate([lidar_like_clouds(2, REG_CAP, 51), kitti_like_dense(1, 52)])
    return x, oracle(x, EVAL_M)


@pytest.mark.parametrize("m", M_EDGES)
def test_sample_counts(lidar_2048, m):
    x, want = lidar_2048
    check_alone_and_in_149(x, m, want[:, :m], "sample-count edge")


@pytest.mark.parametrize("n,E,m", [(300, 300, 1000),           # m > n, every point eligible
                                   (1000, 300, 1200),          # m > n > E
                                   (5000, 37, EVAL_M),         # m > E
                                   (REG_CAP, BUCKET + 1, ELIST + 1)])
def test_more_samples_than_points(n, E, m):
    x = exact_eligible_clouds([E, E, 0], n, n + E)
    x[1, 0] = 0.0                                  # the second cloud's seed dropped (if it was eligible)
    check_alone_and_in_149(x, m, oracle(x, m), "m > E")


@pytest.mark.parametrize("kind", ["few_distinct", "lattice", "paired"])
def test_ties_across_buckets(kind):
    """Clouds whose picks are decided by the tie key, in and across buckets, at the evaluation's size."""
    n, m = REG_CAP, EVAL_M
    if kind == "few_distinct":
        x = np.concatenate([few_distinct_clouds(2, n, 40, 61), few_distinct_clouds(1, n, ELIST + 100, 62)])
    elif kind == "lattice":
        x = lattice_clouds(3, n, 63)
    else:
        x = paired_clouds(3, n, 64)
    check_alone_and_in_149(x, m, oracle(x, m), kind)


@pytest.mark.parametrize("n", T_EDGES)
def test_tie_block_edges(n):
    """The tie key depends on T = min(2^floor(log2 n), 512); the clouds are made of ties and m > n."""
    m = n + 7
    x = np.concatenate([lattice_clouds(1, n, n), few_distinct_clouds(1, n, 40, n), paired_clouds(1, n, n),
                        dropped_seed_clouds(1, n, n)])
    want = oracle(x, m)
    check_alone_and_in_149(x, m, want, f"tie block T={min(1 << (n.bit_length() - 1), TIE_BLOCK)}")
    ks = np.flatnonzero((x[3] == COINCIDENT).all(-1))       # the eight coincident points of the last cloud
    assert want[3, 2] == min(ks, key=lambda k: tie_key(int(k), n))


# ---------------------------------------------------------------------------------------------------------------------
# 4. degenerate regimes on the multi kernel (b = 149) and on the pruned kernel (b = 148)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b", [NUM_SMS + 1, NUM_SMS])
def test_every_point_inside_the_radius(b):
    x = t1_clouds(b, 4096, 71)
    assert eligible(x).max() == 0
    got = fps(x, 64)
    label = case(0, 4096, 64, b, kernel_for(b, 4096), "trap T1")
    check(got, np.zeros_like(got), label, "expected index 0 throughout")
    check(got[-4:], oracle(x[-4:], 64), label)


@pytest.mark.parametrize("b", [NUM_SMS + 1, NUM_SMS])
def test_eligibility_threshold_in_double(b):
    n, m = 4096, 512
    x, above, below = threshold_clouds(b, n, 72)
    E = above.sum(1) + 100
    got = fps(x, m)
    labels = [case(E[c], n, m, b, kernel_for(b, n), "points on the eligibility threshold") for c in range(b)]
    check(got, oracle(x, m), labels)
    for c in range(b):                              # m > E: every eligible point is picked, no ineligible one but 0
        picked = np.zeros(n, bool)
        picked[got[c]] = True
        assert picked[above[c]].all() and not picked[below[c]].any(), labels[c]


@pytest.mark.parametrize("b", [NUM_SMS + 1, NUM_SMS])
def test_dropped_seed_pixel(b):
    n, m = 2048, 8
    x = dropped_seed_clouds(b, n, 73)
    got = fps(x, m)
    labels = [case(9, n, m, b, kernel_for(b, n), "dropped seed, eight coincident points") for c in range(b)]
    check(got, oracle(x, m), labels)
    for c in range(b):
        ks = np.flatnonzero((x[c] == COINCIDENT).all(-1))
        assert got[c, 0] == 0 and got[c, 2] == min(ks, key=lambda k: tie_key(int(k), n)), labels[c]


# ---------------------------------------------------------------------------------------------------------------------
# 5. every kernel, forced through DUSTY_FPS_ALGO (read once per process, so one process per variant)
# ---------------------------------------------------------------------------------------------------------------------
WORKER = r'''
import os, sys
import numpy as np, torch
sys.path.insert(0, os.environ["DUSTY_ROOT"])
from dusty_gan_b200.utils.sampling.fps import furthest_point_sampling
cases = np.load(sys.argv[1])
out = {}
for i in range(len(cases.files) // 2):
    x = torch.from_numpy(cases[f"x{i}"]).cuda()
    out[f"idx{i}"] = furthest_point_sampling(x, int(cases[f"m{i}"])).cpu().numpy()
np.savez(sys.argv[2], **out)
'''


@pytest.fixture(scope="module")
def variant_cases(tmp_path_factory):
    """(what, clouds, m, oracle indices) for a compact subset of the cases above, and the file the worker reads."""
    th, _, _ = threshold_clouds(3, 4096, 81)
    cases = [
        ("exact eligible counts", exact_eligible_clouds([0, 1, BUCKET + 1, MT_DCAP + 1, PR_CAP + 1, SMEM_CAP + 1],
                                                        REG_CAP, 82), EVAL_M),
        ("exact eligible counts", exact_eligible_clouds([BUCKET - 1, SMEM_CAP + 1], REG_CAP + 1, 83), 600),
        ("winner list edge", lidar_like_clouds(1, REG_CAP, 84), ELIST + 1),
        ("tie block edge", np.concatenate([lattice_clouds(1, 513, 85), paired_clouds(1, 513, 85)]), 520),
        ("tie block edge", np.concatenate([lattice_clouds(1, 1025, 86), few_distinct_clouds(1, 1025, 40, 86)]), 1032),
        ("ties across buckets", np.concatenate([lattice_clouds(1, REG_CAP, 87), few_distinct_clouds(1, 8192, 40, 87)
                                                .repeat(4, axis=1)]), EVAL_M),
        ("points on the eligibility threshold", th, 512),
        ("trap T1", t1_clouds(2, 4096, 88), 64),
        ("dropped seed", dropped_seed_clouds(3, 2048, 89), 8),
        ("more clouds than SMs", lidar_like_clouds(NUM_SMS + 2, 2049, 90), 256),
    ]
    path = tmp_path_factory.mktemp("fps_variants") / "cases.npz"
    np.savez(path, **{f"x{i}": x for i, (_, x, _) in enumerate(cases)}, **{f"m{i}": m for i, (_, _, m) in enumerate(cases)})
    return [(what, x, m, oracle(x, m)) for what, x, m in cases], path


@pytest.mark.parametrize("algo", ["flat", "single", "multi", "l2"])
def test_forced_variant(variant_cases, tmp_path, algo):
    cases, path = variant_cases
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out_path = tmp_path / "idx.npz"
    env = dict(os.environ, DUSTY_ROOT=ROOT, DUSTY_FPS_ALGO=algo)
    run = subprocess.run([sys.executable, str(script), str(path), str(out_path)], env=env, capture_output=True,
                         text=True, timeout=600)
    assert run.returncode == 0, run.stderr[-3000:]
    got = np.load(out_path)
    for i, (what, x, m, want) in enumerate(cases):
        b, n, _ = x.shape
        E = eligible(x)
        check(got[f"idx{i}"], want, [case(E[c], n, m, b, kernel_for(b, n, algo), f"{what}, DUSTY_FPS_ALGO={algo}")
                                     for c in range(b)])


# ---------------------------------------------------------------------------------------------------------------------
# 6. gather
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 3, 5])
def test_gather_with_repeated_indices(c):
    """Forward bit-equal; backward within m 2^-23 of a float64 scatter-add, relative to the sum of |gradient| that
    lands on each point. Repeated indices are the only case where the backward's atomics collide."""
    from dusty_gan_b200.utils.sampling.fps import gather_operation
    b, n, m = 3, 100, 300
    g = torch.Generator().manual_seed(c)
    feats = torch.randn(b, c, n, generator=g).cuda().requires_grad_(True)
    idx = torch.zeros(b, m, dtype=torch.int32)                         # T1's output: index 0 throughout
    idx[1] = torch.randint(0, n, (m,), generator=g, dtype=torch.int32)  # m > n: repeats
    idx[2] = torch.arange(m, dtype=torch.int32) % 7
    idx = idx.cuda()
    out = gather_operation(feats, idx)
    want = native.gather_points(feats.detach().cpu().numpy(), idx.cpu().numpy())
    assert np.array_equal(out.detach().cpu().numpy(), want)
    assert torch.equal(out, feats.detach().gather(2, idx.long()[:, None, :].expand(-1, c, -1)))
    grad = torch.randn(b, c, m, generator=g).cuda()
    out.backward(grad)
    ii = idx.long()[:, None, :].expand(-1, c, -1)
    ref = torch.zeros(b, c, n, dtype=torch.float64, device="cuda").scatter_add_(2, ii, grad.double())
    mass = torch.zeros(b, c, n, dtype=torch.float64, device="cuda").scatter_add_(2, ii, grad.double().abs())
    err = (feats.grad.double() - ref).abs()
    assert (err <= m * 2.0 ** -23 * mass).all(), (err.max().item(), c)
    assert (feats.grad[mass == 0] == 0).all()


@pytest.mark.parametrize("b", [3, NUM_SMS + 1])
def test_downsample_with_and_without_grad(b):
    """The fused gather (no grad) and fps + gather_operation (grad) give bit-identical points, T1 clouds included."""
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    x = np.concatenate([lidar_like_clouds(b - 1, 4096, 91), t1_clouds(1, 4096, 92)])
    t = torch.from_numpy(x).cuda()
    plain = downsample_point_clouds(t, 700)
    with_grad = downsample_point_clouds(t.clone().requires_grad_(True), 700)
    assert with_grad.requires_grad and not plain.requires_grad
    assert torch.equal(plain, with_grad.detach())
    assert torch.equal(plain[-1], t[-1, :1].expand(700, -1))
