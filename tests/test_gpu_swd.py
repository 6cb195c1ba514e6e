"""Sliced Wasserstein distance on the B200: stage A (descriptors and statistics) and stage B (projection, segmented
sort, |a - b| sums) against float64 numpy, compute_swd against the float64 oracle and the published op chain
(oracle/swd.py), its properties and its sharding over gloo ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import swd as oswd

pytestmark = pytest.mark.gpu


def _swd():
    from dusty_gan_b200.utils.metrics import swd
    return swd


def _draws(h, w, c, seed, n_pyramids=None, **kw):
    torch.manual_seed(seed)
    return _swd().draw(h, w, c, oswd.default_pyramids(h) if n_pyramids is None else n_pyramids, **kw)


@pytest.mark.parametrize("n,c,h,w", [(3, 1, 64, 512), (4, 3, 32, 64)])
def test_descriptors_and_statistics_match_float64(n, c, h, w):
    swd = _swd()
    x = oswd.range_images(n, c, h, w, 3)
    draws = _draws(h, w, c, 1)
    positions, _ = swd.upload_draws(draws, "cuda")
    levels = len(draws)
    desc, stats = swd.descriptors(x.cuda(), positions, levels, 128)
    pyr = oswd.pyramid_numpy(x.numpy(), levels - 1)
    for level in range(levels):
        want = oswd.descriptors_numpy(pyr[level], draws[level][0].numpy())
        got = desc[level].double().cpu().numpy()
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max(), level
        rows = want.reshape(-1, c, 49)
        mean, std = rows.mean(axis=(0, 2)), rows.std(axis=(0, 2), ddof=1)
        s = stats[level].cpu().numpy()
        assert (np.abs(s[:, 0] - mean) <= 1e-5 * std).all() and (np.abs(s[:, 1] - std) <= 1e-5 * std).all(), level
    desc2, stats2 = swd.descriptors(x.cuda(), positions, levels, 128)
    assert torch.equal(desc, desc2) and torch.equal(stats, stats2)


def _identity_stats(c):
    """mean 0, std 1: (x - 0) / f32(1 + 1e-8) = x exactly."""
    s = torch.zeros(1, c, 2, dtype=torch.float64, device="cuda")
    s[..., 1] = 1.0
    return s


def _sums(a, b, dirs, begin=0, stride=1):
    """Stage B on hand-built (rows, K) descriptor sets with identity statistics; dirs (K, D)."""
    c = a.shape[1] // 49
    st = _identity_stats(c)
    return _swd().sliced_sums(a[None].contiguous(), st, b[None].contiguous(), st, dirs[None].contiguous(), begin,
                              stride)[0]


def _one_hot(k, d):
    dirs = torch.zeros(k, d, device="cuda")
    dirs[torch.arange(d) % k, torch.arange(d)] = 1.0
    return dirs


def _f64_sums(a, b, dirs):
    pa = a.double().cpu().numpy() @ dirs.double().cpu().numpy()
    pb = b.double().cpu().numpy() @ dirs.double().cpu().numpy()
    return np.abs(np.sort(pa, axis=0) - np.sort(pb, axis=0)).sum(axis=0)


def test_integer_shift_gives_exactly_delta_times_rows():
    g = torch.Generator().manual_seed(0)
    rows = 3001
    a = torch.randint(-50, 50, (rows, 49), generator=g).float().cuda()
    for delta in (1, 7, -3):
        s = _sums(a, a + delta, _one_hot(49, 64))
        assert (s == abs(delta) * rows).all(), (delta, s)


def test_special_keys():
    rows, k = 4099, 49
    g = torch.Generator().manual_seed(1)
    mags = 10.0 ** torch.empty(rows, k).uniform_(-30, 30, generator=g)
    signs = torch.where(torch.rand(rows, k, generator=g) < 0.5, -1.0, 1.0)
    cases = {
        "equal": (torch.full((rows, k), 0.25), torch.full((rows, k), -0.5)),
        # whole rows of -0 and of +0: the projection of an all -0 row is -0, so both zero keys go through the sort
        "zeros": (torch.where(torch.rand(rows, 1, generator=g) < 0.5, -0.0, 0.0).expand(rows, k).contiguous(),
                  torch.rand(rows, k, generator=g) - 0.5),
        "subnormal": (torch.randint(-2 ** 20, 2 ** 20, (rows, k), generator=g).float() * 2.0 ** -149,
                      torch.randint(-2 ** 20, 2 ** 20, (rows, k), generator=g).float() * 2.0 ** -149),
        "extreme": (mags * signs, (mags * signs).flip(0) * 3.0),
    }
    dirs = _one_hot(k, 49)
    for name, (a, b) in cases.items():
        a, b = a.float().cuda(), b.float().cuda()
        got = _sums(a, b, dirs).cpu().numpy()
        want = _f64_sums(a, b, dirs)
        assert (np.abs(got - want) <= 1e-12 * np.abs(want)).all(), name
    a = torch.full((rows, k), 0.25, device="cuda")
    assert (_sums(a, a, dirs) == 0).all()
    b = a.clone()
    b[17, 3] = float("nan")
    assert torch.isnan(_sums(a, b, dirs)).all()        # 0 * NaN is NaN: the row is NaN on every direction


# 32 (warp), 128 (projection tile) and 512 (sort tile) each +-1
ROWS = [1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513, 128000, 640000]


@pytest.mark.parametrize("rows", ROWS)
def test_segment_lengths(rows):
    g = torch.Generator().manual_seed(rows)
    a = torch.randn(rows, 49, generator=g).cuda()
    b = torch.randn(rows, 49, generator=g).cuda() * 1.5 + 0.7
    one_hot = _one_hot(49, 8)
    got = _sums(a, b, one_hot).cpu().numpy()                   # the projection is exact: this checks the sort
    want = _f64_sums(a, b, one_hot)
    assert (np.abs(got - want) <= 1e-12 * want).all(), (got, want)
    dirs = torch.randn(49, 40, generator=g).cuda()
    got = _sums(a, b, dirs).cpu().numpy()
    want = _f64_sums(a, b, dirs)
    # an f32 dot product of 49 terms is within 49 * 2^-24 * sum_k |w_k x_k| of the exact one; over many rows the
    # errors average out and 1e-6 of the sum itself holds
    wabs = np.abs(dirs.double().cpu().numpy())
    scale = (np.abs(a.double().cpu().numpy()) @ wabs).sum(0) + (np.abs(b.double().cpu().numpy()) @ wabs).sum(0)
    assert (np.abs(got - want) <= 49 * 2.0 ** -24 * scale).all()
    if rows >= 128000:
        assert (np.abs(got - want) <= 1e-6 * want).all(), np.abs(got / want - 1).max()


@pytest.mark.parametrize("rows,n_dirs,begin,stride", [(640000, 420, 1, 1), (12265 * 128, 512, 2, 3)])
def test_calls_stay_inside_the_queried_workspace(rows, n_dirs, begin, stride):
    """Direction ranges whose own balanced batch is larger than the one the workspace query sized for n_dirs (the
    second is rank 2 of 3 at N = 12265): the call must cap its batch, touch nothing past the workspace, and give the
    sums a full-range call gives."""
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    g = torch.Generator().manual_seed(rows)
    a = torch.randn(rows, 49, generator=g).cuda()
    b = (torch.randn(rows, 49, generator=g) * 0.8).cuda()
    dirs = torch.randn(49, n_dirs, generator=g).cuda()
    st = _identity_stats(1)
    need = lib.dusty_swd_sliced_workspace_bytes(rows, 1, n_dirs)
    guard = 1 << 20
    ws = torch.full((need + guard,), 0x5A, dtype=torch.uint8, device="cuda")
    sums = torch.zeros(n_dirs, dtype=torch.float64, device="cuda")
    _lib.check(lib.dusty_swd_sliced(_lib.ptr(a), _lib.ptr(b), _lib.ptr(st), _lib.ptr(st), rows, 1, _lib.ptr(dirs),
                                    n_dirs, begin, n_dirs, stride, _lib.ptr(sums), _lib.ptr(ws), need,
                                    _lib.stream_of(a)), "dusty_swd_sliced")
    assert (ws[need:] == 0x5A).all()
    del ws
    full = _sums(a, b, dirs)
    assert torch.equal(sums[begin::stride], full[begin::stride])


def test_sums_do_not_depend_on_the_direction_deal():
    g = torch.Generator().manual_seed(5)
    rows = 640000
    a = torch.randn(rows, 49, generator=g).cuda()
    b = (torch.randn(rows, 49, generator=g) * 0.8).cuda()
    dirs = torch.randn(49, 512, generator=g).cuda()
    full = _sums(a, b, dirs)                      # two batches of 256 directions
    assert torch.equal(_sums(a, b, dirs), full)
    for begin, stride in ((1, 3), (0, 2), (7, 8)):
        part = _sums(a, b, dirs, begin, stride)
        assert torch.equal(part[begin::stride], full[begin::stride])
        mask = torch.ones(512, dtype=torch.bool)
        mask[begin::stride] = False
        assert (part[mask.cuda()] == 0).all()


@pytest.mark.parametrize("n,c,h,w", [(4, 1, 64, 512), (3, 3, 32, 64), (2, 2, 64, 128)])
def test_compute_swd_matches_the_float64_oracle_and_the_published_chain(n, c, h, w):
    swd = _swd()
    x1, x2 = oswd.range_images(n, c, h, w, 10), oswd.range_images(n, c, h, w, 11)
    torch.manual_seed(4)
    got = swd.compute_swd(x1.cuda(), x2.cuda(), return_by_resolution=True).double().numpy()
    draws = _draws(h, w, c, 4)
    want = oswd.swd_numpy(x1.numpy(), x2.numpy(), [p.numpy() for p, _ in draws], [d.numpy() for _, d in draws],
                          len(draws) - 1)
    assert (np.abs(got - want) <= 1e-5 * want).all(), (got, want)
    torch.manual_seed(4)
    ref = oswd.swd_torch(x1.cuda(), x2.cuda(), return_by_resolution=True).double().numpy()
    assert (np.abs(got - ref) <= 1e-4 * ref).all(), (got, ref)


def test_dusty_like_images_at_n_1000_match_the_published_chain():
    swd = _swd()
    x1 = oswd.range_images(1000, 1, 64, 512, 20).cuda()
    x2 = oswd.range_images(1000, 1, 64, 512, 21, dropped=0.4).cuda()
    torch.manual_seed(9)
    got = swd.compute_swd(x1, x2, return_by_resolution=True).double().numpy()
    torch.manual_seed(9)
    ref = oswd.swd_torch(x1, x2, return_by_resolution=True).double().numpy()
    assert (np.abs(got - ref) <= 1e-4 * ref).all(), (got, ref)


def test_properties():
    swd = _swd()
    x1 = oswd.range_images(6, 1, 64, 512, 30).cuda()
    x2 = oswd.range_images(6, 1, 64, 512, 31).cuda()

    def run(a, b, **kw):
        torch.manual_seed(2)
        return swd.compute_swd(a, b, **kw)
    score = run(x1, x2)
    assert score.dtype == torch.float32 and score.dim() == 0 and score.device.type == "cpu"
    assert run(x1, x1).item() == 0.0
    assert torch.equal(run(x2, x1), score)
    assert torch.equal(run(x1, x2), score)
    per_level = run(x1, x2, return_by_resolution=True)
    assert per_level.shape == (3,) and torch.equal(torch.mean(per_level), score)
    positions = _draws(64, 512, 1, 2)[0][0]
    py, px = divmod(int(positions[0]), 512 - 6)
    bad = x1.clone()
    bad[4, 0, py + 3, px + 3] = float("nan")
    assert torch.isnan(run(bad, x2))


def test_refusals():
    swd = _swd()
    from dusty_gan_b200 import _lib
    x = oswd.range_images(2, 1, 64, 512, 1).cuda()
    with pytest.raises(TypeError):
        swd.compute_swd(x.double(), x.double())
    for a, b, kw in [(x, x[:1], {}), (x[0], x[0], {}), (x, x, {"slice_size": 9}), (x[..., :510], x[..., :510], {}),
                     (x, x, {"n_descriptors": 1221}), (x[:, :, :32, :32], x[:, :, :32, :32], {})]:
        with pytest.raises(ValueError):
            swd.compute_swd(a, b, **kw)
    with pytest.raises(RuntimeError, match="no CPU path"):
        swd.compute_swd(x.cpu(), x.cpu())
    with pytest.raises(ValueError, match="different devices"):
        swd.compute_swd(x, x.cpu())
    positions = torch.zeros(3, 4, dtype=torch.int32, device="cuda")
    positions[2, 1] = 10 * 122                     # one past the last position of the 16x128 level
    desc = torch.empty(3 * 2 * 4 * 49, device="cuda")
    stats = torch.empty(3, 1, 2, dtype=torch.float64, device="cuda")
    ws = _lib.workspace(_lib.load().dusty_swd_descriptors_workspace_bytes(2, 1, 64, 512, 3, 4), "cuda")
    rc = _lib.load().dusty_swd_descriptors(_lib.ptr(x), 2, 1, 64, 512, 3, _lib.ptr(positions), 4, _lib.ptr(desc),
                                           _lib.ptr(stats), _lib.ptr(ws), ws.numel(), _lib.stream_of(x))
    assert rc == -1 and b"outside" in _lib.load().dusty_last_error_string()
    positions[2, 1] = -1
    rc = _lib.load().dusty_swd_descriptors(_lib.ptr(x), 2, 1, 64, 512, 3, _lib.ptr(positions), 4, _lib.ptr(desc),
                                           _lib.ptr(stats), _lib.ptr(ws), 0, _lib.stream_of(x))
    assert rc == -3                                # DUSTY_ENOSPACE comes before the positions are read


WORKER = r'''
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["DUSTY_ROOT"])
torch.cuda.set_device(0)
from dusty_gan_b200.utils.metrics.swd import compute_swd
from oracle.swd import range_images
cases = [(range_images(5, 1, 64, 512, 1), range_images(5, 1, 64, 512, 2)),
         (range_images(3, 3, 32, 64, 3), range_images(3, 3, 32, 64, 4))]
cases = [(a.cuda(), b.cuda()) for a, b in cases]
def run(a, b):
    torch.manual_seed(7)
    return compute_swd(a, b, return_by_resolution=True)
single = [run(a, b) for a, b in cases]
dist.init_process_group("gloo")
ok = all(torch.equal(run(a, b), s) for (a, b), s in zip(cases, single))
flags = [None] * dist.get_world_size(); dist.all_gather_object(flags, bool(ok))
if int(os.environ["RANK"]) == 0: print("RESULT", json.dumps({"ok": all(flags), "world": dist.get_world_size()}))
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_scores_equal_one_rank_sharing_one_gpu(tmp_path, world):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, DUSTY_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", str(29590 + world), str(script)],
                         env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][-1]
    assert '"ok": true' in line and f'"world": {world}' in line, line
