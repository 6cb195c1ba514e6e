"""Reconstruction metrics on the B200: the metre images bit-equal to the reference's torch chain on the same device,
the per-scan sums against the float64 oracle, empty and degenerate scans, determinism and batch independence, the
caller's stream, pipeline.reconstruction_scores and the example script."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import depth as od

pytestmark = pytest.mark.gpu

EXACT = [0, 1, 2, 7, 8, 9]          # |S|, |pred valid|, |target valid|, #a1, #a2, #a3


def bits(t):
    return t.contiguous().view(torch.int32)


def assert_bit_equal(a, b, what):
    assert a.shape == b.shape, what
    same = (bits(a) == bits(b)) | (torch.isnan(a) & torch.isnan(b))
    assert bool(same.all()), f"{what}: {(~same).sum().item()} of {same.numel()} differ"


def lidar_of(h, w, min_depth=0.9, max_depth=120.0):
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    return LiDAR(h, w, min_depth, max_depth, angle=synthetic_hdl64e_angles()).cuda()


def images(b, h, w, seed, dropped=0.3):
    """DUSty-like tanh-space range images with dropped pixels at exactly -1, made on the GPU."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.tanh(torch.randn(b, 1, h, w, generator=g, device="cuda") * 0.8 - 0.2)
    return torch.where(torch.rand(b, 1, h, w, generator=g, device="cuda") < dropped, torch.full_like(x, -1.0), x)


def oracle(x, y, lidar, tol=0.0):
    mx, vx = od.metres_torch(x.clone(), lidar.min_depth, lidar.max_depth, tol)
    my, vy = od.metres_torch(y.clone(), lidar.min_depth, lidar.max_depth, tol)
    return mx, my, od.sums_numpy(mx.cpu().numpy(), vx.cpu().numpy(), my.cpu().numpy(), vy.cpu().numpy())


def assert_sums_close(got, want):
    got = got.cpu().numpy() if isinstance(got, torch.Tensor) else got
    assert np.array_equal(got[:, EXACT], want[:, EXACT]), "counts differ"
    for k in (3, 4, 5):
        assert np.allclose(got[:, k], want[:, k], rtol=1e-11, atol=0, equal_nan=True), k
    assert np.allclose(got[:, 6], want[:, 6], rtol=1e-9, atol=1e-12, equal_nan=True), 6


@pytest.mark.parametrize("limits", [(0.9, 120.0), (2.95, 144.9)])
@pytest.mark.parametrize("h,w", [(64, 512), (64, 2048)])
@pytest.mark.parametrize("b", [1, 3, 32, 257])
def test_metre_images_bit_exact_and_sums_against_the_oracle(b, h, w, limits):
    """f32(1/min - 1/max) and f32(1/max) are formed in double and rounded once, as ATen's kernels receive them; for both
    limit pairs that differs from the f32 arithmetic on the rounded limits."""
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics, depth_sums
    lidar = lidar_of(h, w, *limits)
    x, y = images(b, h, w, 10 + b), images(b, h, w, 20 + b, dropped=0.45)
    sums, pm, tm = depth_sums(x, y, lidar, return_depth=True)
    want_p, want_t, want = oracle(x, y, lidar)
    assert_bit_equal(pm, want_p, "pred metres")
    assert_bit_equal(tm, want_t, "target metres")
    assert_sums_close(sums, want)
    mean = compute_depth_metrics(x, y, lidar)
    ref = od.mean_numpy(want)
    assert mean["#scans"] == b and mean["#empty"] == ref["#empty"] == 0
    for k in od.KEYS:
        assert math.isclose(mean[k], ref[k], rel_tol=1e-9, abs_tol=1e-12), (k, mean[k], ref[k])


@pytest.mark.parametrize("tol", [0.0, 0.25])
def test_empty_and_degenerate_scans(tol):
    """Scan 0: prediction dropped; scan 1: target dropped; scan 2: disjoint masks; scan 3: inputs exactly -1, above 1,
    +-inf, NaN and at tol (x = -0.5 gives inv = 0.25 exactly); scans 4, 5: ordinary."""
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics
    h, w = 64, 512
    lidar = lidar_of(h, w)
    x, y = images(6, h, w, 1), images(6, h, w, 2)
    x[0] = -1.0
    y[1] = -1.0
    even = (torch.arange(h * w, device="cuda").view(1, h, w) % 2) == 0
    x[2] = torch.where(even, x[2].clamp(min=-0.9), torch.full_like(x[2], -1.0))
    y[2] = torch.where(even, torch.full_like(y[2], -1.0), y[2].clamp(min=-0.9))
    special = torch.tensor([-1.0, 1.0, 1.5, 7.0, float("inf"), float("-inf"), float("nan"), -0.5, -2.0, 0.0],
                           device="cuda")
    flat_x, flat_y = x[3].view(-1), y[3].view(-1)
    flat_x[: 40 * len(special)] = special.repeat(40)
    flat_y[: 40 * len(special)] = special.roll(3).repeat(40)
    scores, pm, tm = compute_depth_metrics(x, y, lidar, tol=tol, reduction="none", return_depth=True)
    want_p, want_t, want = oracle(x, y, lidar, tol)
    assert_bit_equal(pm, want_p, "pred metres")
    assert_bit_equal(tm, want_t, "target metres")
    from dusty_gan_b200.utils.metrics.depth import depth_sums
    assert_sums_close(depth_sums(x, y, lidar, tol), want)
    assert want[:3, 0].tolist() == [0, 0, 0] and (want[3:, 0] > 0).all()
    per = od.finalise_numpy(want)
    for k in od.KEYS:
        got = scores[k].numpy()
        assert scores[k].dtype == torch.float64 and got.shape == (6,)
        assert np.allclose(got, per[k], rtol=1e-9, atol=1e-12, equal_nan=True), k
        if k.startswith("mask_"):
            continue
        assert np.isnan(got[:3]).all() and np.isfinite(got[3:]).all(), k
    mean = compute_depth_metrics(x, y, lidar, tol=tol)
    assert mean["#scans"] == 6 and mean["#empty"] == 3
    assert math.isclose(mean["rmse"], float(np.mean(per["rmse"][3:])), rel_tol=1e-9)


def test_every_scan_empty_gives_nan_means():
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics
    lidar = lidar_of(64, 512)
    x = torch.full((2, 1, 64, 512), -1.0, device="cuda")
    mean = compute_depth_metrics(x, images(2, 64, 512, 3), lidar)
    assert mean["#empty"] == 2 and all(math.isnan(mean[k]) for k in od.KEYS)


def test_deterministic_and_independent_of_the_batch():
    from dusty_gan_b200.utils.metrics.depth import depth_sums
    lidar = lidar_of(64, 512)
    x, y = images(257, 64, 512, 5), images(257, 64, 512, 6, dropped=0.5)
    first, second = depth_sums(x, y, lidar), depth_sums(x, y, lidar)
    assert torch.equal(first.view(torch.int64), second.view(torch.int64))
    for i in (0, 1, 128, 256):
        alone = depth_sums(x[i:i + 1], y[i:i + 1], lidar)
        assert torch.equal(alone.view(torch.int64), first[i:i + 1].view(torch.int64)), i
    mid = depth_sums(x[100:140], y[100:140], lidar)
    assert torch.equal(mid.view(torch.int64), first[100:140].view(torch.int64))


def test_runs_on_the_current_stream():
    """The inputs are written on a side stream behind a spin of about 50 ms; a launch on any other stream would read
    them before they exist."""
    from dusty_gan_b200.utils.metrics.depth import depth_sums
    lidar = lidar_of(64, 512)
    x, y = images(32, 64, 512, 7), images(32, 64, 512, 8)
    want = depth_sums(x, y, lidar)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        xs, ys = torch.full_like(x, -1.0), torch.full_like(y, -1.0)
        torch.cuda._sleep(100_000_000)
        xs.copy_(x)
        ys.copy_(y)
        got = depth_sums(xs, ys, lidar)
        host = torch.empty(got.shape, dtype=got.dtype, pin_memory=True)
        host.copy_(got, non_blocking=True)
    side.synchronize()
    assert torch.equal(host.view(torch.int64), want.cpu().view(torch.int64))


def _head_and_batch(b, seed):
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.models.dusty import DUSty1
    from oracle import head_projection as hp, real_data as rd
    h, w = 64, 512
    lidar = lidar_of(h, w)
    head = DUSty1(torch.nn.Identity(), tau=1.0).cuda().eval()
    g = torch.Generator().manual_seed(seed)
    head.gumbel.fixed_noise = hp.logistic_noise(torch.rand(1, 1, h, w, generator=g).cuda(),
                                                torch.rand(1, 1, h, w, generator=g).cuda())
    output = {"depth": torch.tanh(torch.randn(b, 1, h, w, generator=g) * 0.8 - 0.3).cuda(),
              "confidence": (torch.randn(b, 1, h, w, generator=g) * 2 + 1).cuda()}
    scans = torch.from_numpy(rd.synthetic_scans(b, seed=seed, hs=h, ws=4 * w)).cuda()
    real_inv, _, real_points = pipeline.preprocess_reals(scans, lidar)
    return head, output, real_inv, real_points, lidar


def test_reconstruction_scores_are_the_library_calls_they_combine():
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_cd
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics
    head, output, real_inv, real_points, lidar = _head_and_batch(4, 3)
    scores = pipeline.reconstruction_scores(head, {k: v.clone() for k, v in output.items()}, real_inv, real_points,
                                            lidar)
    out = pipeline.maskout_and_project(head, {k: v.clone() for k, v in output.items()}, lidar)
    assert out["points"].shape == (4, 64 * 512, 3)
    cd = compute_cd(real_points, out["points"]).mean()
    assert np.float32(scores["cd"]) == cd.cpu().numpy() and scores["cd"] == float(cd)
    depth = compute_depth_metrics(out["depth"], real_inv, lidar)
    assert set(scores) == set(depth) | {"cd"}
    for k, v in depth.items():
        assert scores[k] == v or (math.isnan(scores[k]) and math.isnan(v)), k
    assert depth["#empty"] == 0 and all(math.isfinite(depth[k]) for k in od.KEYS)


def test_example_script_prints_every_score():
    env = dict(os.environ, PYTHONNOUSERSITE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "evaluate_reconstruction.py"), "--num-test",
                          "64", "--steps", "3"], capture_output=True, text=True, env=env, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    scores = json.loads(out.stdout)
    for k in od.KEYS + ("cd", "inversion_loss"):
        assert k in scores and math.isfinite(scores[k]), (k, scores.get(k))
    assert scores["#scans"] == 64
