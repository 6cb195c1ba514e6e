"""The JSD occupancy vote and divergence at the evaluation's shape, at every exact tie, on both sides of the search's
fallback threshold, at clamped cells, on non-finite input and at the grid-capacity edges of csrc/jsd.cu.

The vote must be bit-equal, counters and clouds_touching, to ``oracle.jsd.vote_torch``: the reference's brute force as
torch ops on the GPU, which ``test_vote_torch_equals_the_numpy_oracle`` pins to ``oracle.jsd.vote`` on every edge set
below. The divergence is checked against the f32 oracle chain and against a float64 restatement.
"""
import warnings

import numpy as np
import pytest
import torch

from helpers import lidar_like_clouds
from oracle import jsd as oj

pytestmark = pytest.mark.gpu

# Constants of csrc/jsd.cu, named so that a change there shows which edge moved.
RADIUS = 2             # vote_kernel searches the (2 RADIUS + 1)^3 cells around the point's rounded cell
SAFE = 2.4             # and trusts the best of them below (SAFE * spacing)^2; otherwise it scans the whole grid
HIST_CAP = 48 * 1024   # grid points one CTA's shared-memory histogram holds
TPB = 256              # threads per CTA: each thread of a cloud's CTA takes every TPB-th point

EVAL_B, EVAL_N, EVAL_RES = 1000, 2048, 28   # the evaluation: 1000 vs 1000 clouds of 2048 points, 28^3 grid
F32 = np.float32


def cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def axis_of(res):
    """The grid's coordinates along one axis, as the oracle's grid holds them."""
    return oj.grid_points(res, False)[0][:res, 2]


def spread(points, n):
    """n points spread evenly over an edge set."""
    return points[np.linspace(0, len(points) - 1, n).astype(np.int64)]


def safe_of(res):
    """(2.4 spacing)^2 with the kernel's f32 arithmetic."""
    s = F32(2.4) * F32(1.0 / float(res - 1))
    return s * s


def vote(x, res, in_sphere):
    """The library's vote of x (numpy or CUDA tensor, (B,N,3)) -> (counters, touching) as int64 numpy arrays."""
    from dusty_gan_b200.utils.metrics import jsd as J
    c, t = J._vote(x if torch.is_tensor(x) else cuda(x), res, in_sphere)
    return c.cpu().numpy().astype(np.int64), t.cpu().numpy().astype(np.int64)


def reference(x, res, in_sphere):
    """oracle.jsd.vote_torch on the GPU -> (counters, touching) as int64 numpy arrays."""
    c, t = oj.vote_torch(x if torch.is_tensor(x) else cuda(x), res, in_sphere)
    return c.cpu().numpy(), t.cpu().numpy()


def assert_votes_equal(x, res, in_sphere, what=""):
    got, want = vote(x, res, in_sphere), reference(x, res, in_sphere)
    for name, g, w in zip(("counters", "clouds_touching"), got, want):
        bad = np.flatnonzero(g != w)
        assert bad.size == 0, (f"{what} res={res} in_sphere={in_sphere}: {name} differ at {bad.size} grid points, "
                               f"first {bad[:5].tolist()}: got {g[bad[:5]].tolist()}, want {w[bad[:5]].tolist()}")


# ---------------------------------------------------------------------------------------------------------- edge sets
def tie_points(res, seed=0):
    """Exact and near ties: the origin and -0.0 coordinates, and the f32 midpoints (axis[i] + axis[i+1]) / 2 in one,
    two and three coordinates (2-, 4- and 8-way ties between grid points), the other coordinates on grid values
    inside the sphere."""
    ax = axis_of(res)
    mid = (ax[:-1] + ax[1:]) / F32(2.0)
    rng = np.random.default_rng(seed)
    inner_ax, inner_mid = ax[np.argsort(np.abs(ax))[:5]], mid[np.argsort(np.abs(mid))[:4]]
    pts = [[0.0, 0.0, 0.0], [-0.0, -0.0, -0.0], [-0.0, 0.0, 0.0], [0.0, -0.0, 0.0], [0.0, 0.0, -0.0]]
    for i in range(res - 1):
        for k in (1, 2, 3):                       # mid[i] and k - 1 midpoints near 0, in each rotation
            p = [mid[i], *(rng.choice(inner_mid) if c < k else rng.choice(inner_ax) for c in (1, 2))]
            pts += [np.roll(p, rot) for rot in range(3)]
    return np.asarray(pts, F32)


def near_midplane_points(res, seed=1):
    """Points near the mid-planes between grid points, the other two coordinates off the grid: 0, 1 and 3 ulp from
    the f32 midpoint, and 2^-16 to 2^-40 spacings from it. The two squared distances differ by about 2 spacing
    times the offset, so they tie only after rounding where that is below an ulp of the distance: near a mid-plane
    close to 0, such as x = 0 on the 28^3 grid, where the dropped points of a scan lie."""
    spacing = 1.0 / (res - 1)
    ax = axis_of(res)
    mid = (ax[:-1] + ax[1:]) / F32(2.0)
    rng = np.random.default_rng(seed)
    pts = []
    for m in mid:
        near = [ulps_from(m, k) for k in (-3, -1, 0, 1, 3)]
        near += [F32(m + s * 2.0 ** -e * spacing) for e in range(16, 41, 4) for s in (-1, 1)]
        for v in near:
            pts += [np.roll([v, *rng.uniform(-0.3, 0.3, 2)], rot) for rot in range(3)]
    return np.asarray(pts, F32)


def ulps_from(v, k):
    """The f32 k ulp above (k > 0) or below v."""
    for _ in range(abs(k)):
        v = np.nextafter(v, F32(np.copysign(np.inf, k)))
    return v


def ray_points(res, seed=2):
    """Points on rays from the origin (axes, face diagonals, space diagonals and 20 seeded directions) at radii from
    0.45 to 0.5 + 4 spacings in steps of spacing / 64: the neighbourhood's best distance crosses (2.4 spacing)^2
    along each in-sphere ray."""
    spacing = 1.0 / (res - 1)
    dirs = [d for d in np.ndindex(3, 3, 3) if d != (1, 1, 1)]
    dirs = np.asarray(dirs, np.float64) - 1.0
    rnd = np.random.default_rng(seed).normal(size=(20, 3))
    dirs = np.concatenate([dirs, rnd])
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    radii = 0.45 + np.arange(int(np.ceil((0.05 + 4 * spacing) / (spacing / 64))) + 1) * (spacing / 64)
    return (dirs[:, None, :] * radii[None, :, None]).astype(F32)          # (rays, radii, 3)


def cells_of(grid, res):
    """(ng,3) integer cell of each grid point: k for the coordinate k * spacing - 0.5."""
    return np.rint((grid.astype(np.float64) + 0.5) * (res - 1)).astype(np.int64)


def outward_points(res, seed=3, per=4):
    """Points 2.5 to 2.6 spacings straight out from each in-sphere grid point whose outward neighbour along that
    axis is not in the sphere, up to 0.3 spacings off the axis. Some of them have their nearest grid point three
    cells away, outside the searched neighbourhood, while a neighbourhood point lies within 2.6 spacings: only the
    full scan answers them, and a threshold a little above 2.4 spacings would not send them there."""
    spacing = 1.0 / (res - 1)
    grid = oj.grid_points(res, True)[0]
    cells = cells_of(grid, res)
    inside = np.zeros((res + 2,) * 3, bool)
    inside[tuple((cells + 1).T)] = True
    rng = np.random.default_rng(seed)
    pts = []
    for k in range(3):
        for s in (-1, 1):
            nb = cells + 1
            nb[:, k] += s
            g = grid[~inside[tuple(nb.T)]]
            for _ in range(per):
                off = rng.uniform(-0.3, 0.3, (len(g), 3))
                off[:, k] = s * rng.uniform(2.5, 2.6, len(g))
                pts.append(g.astype(np.float64) + off * spacing)
    return np.concatenate(pts).astype(F32)


def clamp_points(res):
    """Points outside the cube beyond each face, edge and corner, at 0.5 + spacing/3, 0.6, 1, 10 and 1e30, the other
    coordinates at 0 or inside the cube: their rounded cells are clamped to the cube."""
    spacing = 1.0 / (res - 1)
    pts = []
    for d in np.ndindex(3, 3, 3):
        d = np.asarray(d) - 1
        if not d.any():
            continue
        for t in (0.5 + spacing / 3, 0.6, 1.0, 10.0, 1e30):
            for rest in (0.0, 0.13, -0.29):
                pts.append(np.where(d != 0, d * t, rest))
    return np.asarray(pts, F32)


def nonfinite_points():
    """+inf, -inf and NaN in one coordinate and in all three: every distance is +inf or NaN, and the reference's
    argmin takes grid index 0."""
    pts = []
    for v in (np.inf, -np.inf, np.nan):
        for c in range(3):
            p = [0.1, -0.2, 0.05]
            p[c] = v
            pts.append(p)
        pts.append([v, v, v])
    return np.asarray(pts, F32)


def edge_sets(res):
    """Every constructed edge set at one resolution, each (n,3)."""
    return {"ties": tie_points(res), "near_midplanes": near_midplane_points(res), "rays": ray_points(res).reshape(-1, 3),
            "outward": outward_points(res), "clamped": clamp_points(res), "nonfinite": nonfinite_points()}


def nearest(points, res, in_sphere):
    """(best f32 distance, grid index) of each point, from the reference's brute force on the GPU."""
    d, i = oj.nearest_torch(cuda(points), torch.from_numpy(oj.grid_points(res, in_sphere, "cuda")[0]))
    return d.cpu().numpy(), i.cpu().numpy()


def rounded_cells(points, res):
    """The cell vote_kernel centres its search on: round-to-nearest-even of (p + 0.5) / spacing in f32, clamped."""
    inv = F32(1.0) / F32(1.0 / float(res - 1))
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.rint((points + F32(0.5)) * inv).astype(np.float64)
    return np.clip(np.nan_to_num(c, nan=0.0), 0, res - 1).astype(np.int64)


def tie_structure(points, res, in_sphere):
    """(multiplicity, by_rounding) per point: how many grid points share the reference's f32 minimum distance, and
    whether their float64 distances from the point differ, i.e. the f32 tie exists only after rounding."""
    grid = torch.from_numpy(oj.grid_points(res, in_sphere, "cuda")[0]).cuda()
    p = cuda(points)
    d = p[:, None, :] - grid[None]
    d = d * d
    d = (d[..., 0] + d[..., 1]) + d[..., 2]
    at_min = d == d.amin(1, keepdim=True)
    d64 = ((p.double()[:, None, :] - grid.double()[None]) ** 2).sum(-1)
    lo = torch.where(at_min, d64, torch.inf).amin(1)
    hi = torch.where(at_min, d64, -torch.inf).amax(1)
    return at_min.sum(1).cpu().numpy(), (hi > lo).cpu().numpy()


@pytest.fixture(scope="module")
def eval_sets():
    """The evaluation's two sets: 1000 lidar-like clouds of 2048 points each, 30 % of them dropped to the origin,
    halved as evaluate_synthesis.py does before compute_jsd."""
    return [cuda(lidar_like_clouds(EVAL_B, EVAL_N, seed, dropped=0.3) / F32(2.0)) for seed in (1201, 1202)]


@pytest.fixture(scope="module")
def eval_counts(eval_sets):
    """(kernel votes, reference votes) of each evaluation set, as (counters, touching) int64 numpy pairs."""
    return [(vote(x, EVAL_RES, True), reference(x, EVAL_RES, True)) for x in eval_sets]


# -------------------------------------------------------------------------------------- 1. the reference restatement
def test_library_grid_tables_equal_the_oracle_grid():
    """The grid, cell table and axis the library builds on the GPU are the reference's grid built on the GPU, at every
    resolution used here."""
    from dusty_gan_b200.utils.metrics import jsd as J
    for res in (3, 8, 28, 29, 36, 46, 47):
        for in_sphere in (True, False):
            grid, c2i, axis, spacing = J._grid_tables(res, in_sphere, "cuda")
            want = oj.grid_points(res, in_sphere, "cuda")[0]
            assert np.array_equal(grid.cpu().numpy(), want), (res, in_sphere)
            cells = cells_of(want, res)
            c2i = c2i.cpu().numpy()
            assert np.array_equal(c2i[(cells[:, 0] * res + cells[:, 1]) * res + cells[:, 2]], np.arange(len(want)))
            assert (c2i >= 0).sum() == len(want)
            assert np.array_equal(axis.cpu().numpy(), axis_of(res)) and spacing == 1.0 / (res - 1)
    assert len(oj.grid_points(28, True)[0]) == 10144          # the evaluation's grid: 10 144 in-sphere points of 28^3


@pytest.mark.parametrize("res", [3, 8, 28, 29, 33, 46, 47])
def test_grid_differs_between_devices_only_on_the_sphere(res):
    """The reference builds its grid on the points' device. An even resolution has no grid point on the sphere, so its
    grid is the same on the CPU and the GPU; at an odd one, torch.norm may round a point exactly on the sphere to
    either side of 0.5 depending on the device, and only such points may differ."""
    cpu, gpu = oj.grid_points(res, True, "cpu")[0], oj.grid_points(res, True, "cuda")[0]
    full = oj.grid_points(res, False)[0].astype(np.float64)
    on_sphere = np.abs(np.sqrt((full ** 2).sum(1)) - 0.5) < 1e-6
    if res % 2 == 0:
        assert not on_sphere.any() and np.array_equal(cpu, gpu)
    keys = lambda g: set(map(tuple, cells_of(g, res).tolist()))
    moved = keys(cpu) ^ keys(gpu)
    assert moved <= set(map(tuple, cells_of(full[on_sphere], res).tolist())), sorted(moved)[:5]


@pytest.mark.parametrize("in_sphere", [True, False])
@pytest.mark.parametrize("res", [3, 8, 28, 29])
def test_vote_torch_equals_the_numpy_oracle(res, in_sphere):
    """vote_torch (GPU, chunked) is vote (numpy, one core) exactly on every edge set, each set one cloud, plus a few
    lidar-like clouds, on the same grid: the one built on the CPU."""
    sets = list(edge_sets(res).values())
    sets += list(lidar_like_clouds(3, 700, 1100 + res) / F32(2.0))
    for pts in sets:
        c, t = oj.vote_torch(cuda(pts[None]), res, in_sphere, grid_device="cpu")
        with np.errstate(over="ignore"):                    # 1e30 squared
            oc, ot = oj.vote(pts[None], res, in_sphere)
        assert np.array_equal(c.cpu().numpy(), oc) and np.array_equal(t.cpu().numpy(), ot), (res, in_sphere, len(pts))
    # several clouds at once, and small chunks, give the same
    x = lidar_like_clouds(5, 300, 1150 + res) / F32(2.0)
    oc, ot = oj.vote(x, res, in_sphere)
    c, t = oj.vote_torch(cuda(x), res, in_sphere, grid_device="cpu")
    assert np.array_equal(c.cpu().numpy(), oc) and np.array_equal(t.cpu().numpy(), ot)
    d, i = oj.nearest_torch(cuda(x), torch.from_numpy(oj.grid_points(res, in_sphere)[0]), max_bytes=12 * 1000 * 7)
    assert np.array_equal(np.bincount(i.cpu().numpy(), minlength=len(oc)), oc)


# ----------------------------------------------------------------------------------------------------- 2. the vote
def test_evaluation_shape(eval_counts):
    for (got, want), name in zip(eval_counts, ("generated", "reference")):
        for what, g, w in zip(("counters", "clouds_touching"), got, want):
            bad = np.flatnonzero(g != w)
            assert bad.size == 0, f"{name} set: {what} differ at {bad.size} grid points, first {bad[:5].tolist()}"
        assert got[0].sum() == EVAL_B * EVAL_N
    # about 30 % of the points are dropped, sit at the origin and resolve the 8-way tie there to its lowest index
    grid = oj.grid_points(EVAL_RES, True)[0]
    origin_cell = int(np.flatnonzero((np.abs(grid) < 0.02).all(1))[0])
    assert 0.28 < eval_counts[0][1][0][origin_cell] / (EVAL_B * EVAL_N) < 0.40


@pytest.mark.parametrize("b,n", [(1, 1), (7, TPB - 1), (7, TPB), (7, TPB + 1), (7, 1000), (5000, 64)])
def test_point_counts_around_the_thread_stride(b, n):
    x = lidar_like_clouds(b, n, 1300 + n, dropped=0.3) / F32(2.0)
    for in_sphere in (True, False):
        assert_votes_equal(x, EVAL_RES, in_sphere, f"{b} clouds x {n} points")


@pytest.mark.parametrize("res", [28, 29])
def test_exact_and_rounding_ties(res):
    """The lowest compact index wins every tie: exact ones at the origin, at -0.0 and at f32 midpoints between grid
    points, and ones that exist only after the reference's f32 rounding, near the mid-planes."""
    ties, near = tie_points(res), near_midplane_points(res)
    mult, _ = tie_structure(ties, res, True)
    assert {2, 4, 8} <= set(mult.tolist()), sorted(set(mult.tolist()))
    if res == 28:
        assert mult[0] == 8                                  # the origin: axis[13] == -axis[14] in f32
    mult, by_rounding = tie_structure(near, res, True)
    if res % 2 == 0:                                         # x = 0 is a mid-plane of an even resolution's grid
        assert (by_rounding & (mult >= 2)).sum() >= 10, (by_rounding & (mult >= 2)).sum()
    for in_sphere in (True, False):
        assert_votes_equal(ties[None], res, in_sphere, "exact ties")
        assert_votes_equal(near[None], res, in_sphere, "near mid-planes")
        assert_votes_equal(ties[:, None], res, in_sphere, "exact ties, one point per cloud")


@pytest.mark.parametrize("res", [28, 29])
def test_both_sides_of_the_fallback_threshold(res):
    """Along every in-sphere ray the reference's best distance crosses (2.4 spacing)^2, so the neighbourhood answer
    and the full scan both run; the outward points reach grid points outside the neighbourhood."""
    safe = safe_of(res)
    rays = ray_points(res)
    best, _ = nearest(rays.reshape(-1, 3), res, True)
    beyond = ~(best < safe).reshape(rays.shape[:2])
    assert beyond.any(1).all() and (~beyond).any(1).all(), "a ray does not cross the threshold"
    out = outward_points(res)
    best, idx = nearest(out, res, True)
    far = np.abs(rounded_cells(out, res) - cells_of(oj.grid_points(res, True, "cuda")[0], res)[idx]).max(1) > RADIUS
    assert far.any(), "no point has its nearest grid point outside the searched neighbourhood"
    assert (best[far] >= safe).all(), "a point outside the neighbourhood's reach is below the threshold"
    wider = (F32(2.6) * F32(1.0 / (res - 1))) ** 2
    assert (best[far] < wider).any(), "no point would be misplaced by a threshold of 2.6 spacings"
    for in_sphere in (True, False):
        assert_votes_equal(rays, res, in_sphere, "rays, one per cloud")
        assert_votes_equal(out[None], res, in_sphere, "outward points")


@pytest.mark.parametrize("in_sphere", [True, False])
def test_clamped_cells(in_sphere):
    x = clamp_points(EVAL_RES)
    assert_votes_equal(x[None], EVAL_RES, in_sphere, "outside the cube")
    assert_votes_equal(x[:, None], EVAL_RES, in_sphere, "outside the cube, one point per cloud")


@pytest.mark.parametrize("in_sphere", [True, False])
def test_nonfinite_input_votes_for_grid_index_0(in_sphere):
    x = nonfinite_points()[:, None]
    c, t = reference(x, EVAL_RES, in_sphere)
    assert c[0] == len(x) and t[0] == len(x) and c.sum() == len(x)
    assert_votes_equal(x, EVAL_RES, in_sphere, "non-finite")


def test_resolutions_at_the_shared_memory_cap():
    """46 (47 600 in-sphere points) and 36 (46 656 points of the full cube) fit the 48 Ki histogram, 47 (50 883) and
    37 (50 653) do not; resolution 2 has no in-sphere point. 46, then 8, then 46 again runs the cached shared-memory
    opt-in both ways."""
    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.metrics import jsd as J
    x = np.concatenate([lidar_like_clouds(8, 2048, 1400) / F32(2.0), spread(outward_points(46), 2048)[None]])
    for res in (46, 8, 46):
        assert_votes_equal(x, res, True, "at the cap" if res == 46 else "below the cap")
    assert_votes_equal(x, 36, False, "at the cap")
    assert len(J._grid_tables(46, True, "cuda")[0]) == 47600 and len(J._grid_tables(36, False, "cuda")[0]) == 46656
    lib = _lib.load()
    for res, in_sphere in ((47, True), (37, False)):
        grid, c2i, axis, spacing = J._grid_tables(res, in_sphere, "cuda")
        ng = len(grid)
        assert ng > HIST_CAP
        with pytest.raises(RuntimeError, match=f"{ng} grid points exceed the 48k"):
            J._vote(cuda(x), res, in_sphere)
        out = torch.full((2, ng), 7, dtype=torch.int32, device="cuda")
        rc = lib.dusty_jsd_vote(_lib.ptr(cuda(x)), x.shape[0], x.shape[1], res, ng, _lib.ptr(grid), _lib.ptr(c2i),
                                _lib.ptr(axis), F32(spacing), _lib.ptr(out[0]), _lib.ptr(out[1]), None)
        assert rc == -1 and b"exceed the 48k" in lib.dusty_last_error_string()
        assert (out == 7).all()                              # refused before anything is written
    with pytest.raises(RuntimeError, match="bad sizes"):
        J._vote(cuda(x), 2, True)


def test_histogram_of_exactly_48ki_grid_points():
    """The cap itself: the 46^3 in-sphere grid padded with far-away points to 48 Ki entries runs; one more is
    refused. The padding is never nearest to a finite point and loses every tie to index 0."""
    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.metrics import jsd as J
    grid, c2i, axis, spacing = J._grid_tables(46, True, "cuda")
    padded = torch.cat([grid, torch.full((HIST_CAP + 1 - len(grid), 3), 1e6, device="cuda")]).contiguous()
    x = cuda(np.concatenate([lidar_like_clouds(4, 2048, 1500) / F32(2.0), spread(outward_points(46), 2048)[None],
                             np.resize(np.concatenate([clamp_points(46), nonfinite_points()]), (1, 2048, 3))]))
    want = reference(x, 46, True)
    lib = _lib.load()
    for ng in (HIST_CAP, HIST_CAP + 1):
        out = torch.full((2, ng), 7, dtype=torch.int32, device="cuda")
        rc = lib.dusty_jsd_vote(_lib.ptr(x), x.shape[0], x.shape[1], 46, ng, _lib.ptr(padded), _lib.ptr(c2i),
                                _lib.ptr(axis), F32(spacing), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.stream_of(x))
        if ng == HIST_CAP:
            assert rc == 0, lib.dusty_last_error_string()
            got = out.cpu().numpy().astype(np.int64)
            assert not got[:, len(grid):].any()
            assert np.array_equal(got[0, :len(grid)], want[0]) and np.array_equal(got[1, :len(grid)], want[1])
        else:
            assert rc == -1 and b"exceed the 48k" in lib.dusty_last_error_string()


def test_second_device():
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device")
    from dusty_gan_b200.utils.metrics import jsd as J
    x = lidar_like_clouds(8, 2048, 1600) / F32(2.0)
    x1 = torch.from_numpy(x).to("cuda:1")
    for res in (46, 28):
        c, t = J._vote(x1, res, True)
        assert c.device == x1.device
        want = oj.vote_torch(x1, res, True)
        assert torch.equal(c.long(), want[0]) and torch.equal(t.long(), want[1]), res


def test_deterministic_and_additive_over_batch_splits(eval_sets, eval_counts):
    x = eval_sets[0]
    counters, touching = eval_counts[0][0]
    again = vote(x, EVAL_RES, True)
    assert np.array_equal(again[0], counters) and np.array_equal(again[1], touching)
    for cut in (EVAL_B // 2, 1, 333):
        lo, hi = vote(x[:cut], EVAL_RES, True), vote(x[cut:], EVAL_RES, True)
        assert np.array_equal(lo[0] + hi[0], counters) and np.array_equal(lo[1] + hi[1], touching), cut


def test_runs_on_the_current_stream():
    """The inputs are written on a side stream behind a spin of about 50 ms; a launch on any other stream would read
    them before they exist."""
    from dusty_gan_b200.utils.metrics import jsd as J
    x = cuda(lidar_like_clouds(256, 2048, 1700) / F32(2.0))
    want = [t.cpu() for t in J._vote(x, EVAL_RES, True)]
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        xs = torch.full_like(x, 0.25)
        torch.cuda._sleep(100_000_000)
        xs.copy_(x)
        got = J._vote(xs, EVAL_RES, True)
        host = [torch.empty(g.shape, dtype=g.dtype, pin_memory=True) for g in got]
        for h, g in zip(host, got):
            h.copy_(g, non_blocking=True)
    side.synchronize()
    assert all(torch.equal(h, w) for h, w in zip(host, want))


def test_empty_input_gives_zeroed_outputs():
    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.metrics import jsd as J
    grid, c2i, axis, spacing = J._grid_tables(EVAL_RES, True, "cuda")
    lib = _lib.load()
    for b, n in ((0, 2048), (5, 0), (0, 0)):
        x = torch.zeros(b, n, 3, device="cuda")
        c, t = J._vote(x, EVAL_RES, True)
        assert c.shape == t.shape == (len(grid),) and not c.any() and not t.any()
        out = torch.full((2, len(grid)), 7, dtype=torch.int32, device="cuda")     # the call must clear them
        rc = lib.dusty_jsd_vote(_lib.ptr(x), b, n, EVAL_RES, len(grid), _lib.ptr(grid), _lib.ptr(c2i), _lib.ptr(axis),
                                F32(spacing), _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.stream_of(x))
        assert rc == 0 and not out.any(), (b, n)


# ------------------------------------------------------------------------------------------------ 3. the divergence
# |kernel - float64| is bounded in f32 ulp of the larger operand of the final subtraction plus 1/ln 2: each entropy
# term -p log2 p is computed from a p rounded to f32 (0.5 ulp), which moves the term by |log2 p + 1/ln 2| times that
# rounding; summed over the cells this is at most (H + 1/ln 2) half-ulp. The second part matters when one cell holds
# nearly all the mass: 1 + 1e-8 rounds to 1 in f32 and drops the eps the float64 restatement keeps.
ULPS_F64 = 8
REL_ORACLE = 2.0 ** -19   # |kernel - f32 oracle chain| relative to the same scale: the two f32 chains' errors added


def jsd_kernel(P, Q):
    from dusty_gan_b200 import _lib
    p = torch.from_numpy(np.asarray(P, np.uint32).view(np.int32)).cuda()
    q = torch.from_numpy(np.asarray(Q, np.uint32).view(np.int32)).cuda()
    out = torch.empty(1, device="cuda")
    lib = _lib.load()
    _lib.check(lib.dusty_jsd_from_counts(_lib.ptr(p), _lib.ptr(q), len(p), _lib.ptr(out), _lib.stream_of(out)),
               "dusty_jsd_from_counts")
    return float(out.item())


def histograms(eval_counts):
    ng = len(eval_counts[0][1][0])
    gen, ref = eval_counts[0][1][0], eval_counts[1][1][0]
    rng = np.random.default_rng(1800)
    even = np.where(np.arange(ng) % 2 == 0, rng.integers(1, 1000, ng), 0)
    odd = np.where(np.arange(ng) % 2 == 1, rng.integers(1, 1000, ng), 0)
    one = np.zeros(ng, np.int64)
    one[ng // 3] = 2048
    big = rng.integers(0, 2 ** 31, ng)
    big[rng.uniform(size=ng) < 0.2] = 0
    mid = rng.integers(0, 2 ** 12, ng)                        # total about 2^25
    return {"identical": (gen, gen), "disjoint supports": (even, odd), "one cell vs evaluation": (one, ref),
            "one cell on both sides": (one, one), "uniform": (np.full(ng, 7), np.full(ng, 7)),
            "uniform vs evaluation": (np.full(ng, 7), gen), "evaluation": (gen, ref),
            "totals above 2^24": (big, mid), "totals above 2^24 vs evaluation": (big, ref)}


def test_divergence_against_the_f32_oracle_and_float64(eval_counts):
    for name, (P, Q) in histograms(eval_counts).items():
        got = jsd_kernel(P, Q)
        want32 = oj.jsd_from_counts(P, Q)
        want64, e_sum, e1, e2 = oj.jsd_from_counts_f64(P, Q)
        scale = max(e_sum, (e1 + e2) / 2) + 1 / np.log(2)
        ulp = float(np.spacing(F32(scale)))
        tol = ULPS_F64 * ulp
        assert abs(got - want64) <= tol, (name, got, want64, (got - want64) / ulp)
        assert abs(got - want32) <= REL_ORACLE * scale, (name, got, want32)
        if name.startswith("identical") or name == "uniform" or name == "one cell on both sides":
            assert want64 > 10 * tol                 # the eps leak: identical histograms do not give 0 ...
            assert abs(want32 - want64) <= REL_ORACLE * scale   # ... in the reference's chain either


def test_divergence_of_an_all_zero_histogram_is_nan(eval_counts):
    gen = eval_counts[0][1][0]
    zero = np.zeros_like(gen)
    for P, Q in ((zero, gen), (gen, zero), (zero, zero)):
        with np.errstate(invalid="ignore"):
            assert np.isnan(oj.jsd_from_counts(P, Q))
        assert np.isnan(jsd_kernel(P, Q))


@pytest.mark.parametrize("in_sphere", [True, False])
def test_occupancy_entropy_against_float64(eval_sets, in_sphere):
    from dusty_gan_b200.utils.metrics import jsd as J
    x = eval_sets[1]
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        acc, counters = J.entropy_of_occupancy_grid(x, EVAL_RES, in_sphere)
    assert not [w for w in caught if "Point-clouds" in str(w.message)]     # the halved clouds fit the unit sphere
    c, t = reference(x, EVAL_RES, in_sphere)
    assert counters.dtype == torch.float32 and np.array_equal(counters.cpu().numpy(), c.astype(np.float32))
    want = oj.acc_entropy_f64(t, len(x), len(c))
    assert abs(float(acc) - want) <= 4e-6 * want, (float(acc), want)

