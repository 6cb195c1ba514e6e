"""Reconstruction metrics without a GPU: the oracle on hand-computed images, its properties, the torch chain against
the float64 restatement, the finaliser against the oracle, and every argument refusal of compute_depth_metrics and the
C ABI before any launch."""
import math
import re
import subprocess

import numpy as np
import pytest
import torch

from oracle import depth as od


def test_metres_of_the_postprocess_chain_by_hand():
    # min 1 m, max 4 m: disp = inv * 0.75 + 0.25, every constant exact in f32
    x = torch.tensor([[[[1.0, 3.0, -1.0, -2.0], [0.0, -0.5, float("nan"), 0.5]]]])
    m, valid = od.metres_torch(x, 1.0, 4.0)
    want = [[1.0, 1.0, 0.0, 0.0], [np.float32(1 / 0.625), np.float32(1 / 0.4375), np.nan, np.float32(1 / 0.8125)]]
    assert np.array_equal(m.numpy()[0, 0], np.float32(want), equal_nan=True)
    assert valid[0, 0].tolist() == [[True, True, False, False], [True, True, False, True]]
    # tol: a pixel exactly at tol is not valid (|inv| > tol)
    _, v = od.metres_torch(torch.tensor([[[[-0.5, -0.4999, 1.0, -1.0]]]]), 1.0, 4.0, tol=0.25)
    assert v[0, 0, 0].tolist() == [False, True, True, False]


def test_sums_and_metrics_by_hand():
    p = np.float32([[[[1, 2, 4, 0], [5, 0, 2, 3]]]])
    t = np.float32([[[[1, 1, 5, 2], [0, 0, 2.25, 2]]]])
    s = od.sums_numpy(p, p > 0, t, t > 0)[0]
    # S = pairs (1,1), (2,1), (4,5), (2,2.25), (3,2); six valid on each side
    assert s[:3].tolist() == [5, 6, 6]
    assert math.isclose(s[3], 0 + 1 + 0.2 + 0.25 / 2.25 + 0.5, rel_tol=1e-15)
    assert math.isclose(s[4], 0 + 1 + 0.2 + 0.0625 / 2.25 + 0.5, rel_tol=1e-15)
    assert math.isclose(s[5], 0 + 1 + 1 + 0.0625 + 1, rel_tol=1e-15)
    lg = [0.0, math.log(2), math.log(4) - math.log(5), math.log(2) - math.log(2.25), math.log(3) - math.log(2)]
    assert math.isclose(s[6], sum(v * v for v in lg), rel_tol=1e-14)
    # ratios 1, 2, 1.25 (not < 1.25), 1.125, 1.5 (2 is not < 1.953125)
    assert s[7:].tolist() == [2, 4, 4]
    m = od.finalise_numpy(s[None])
    assert math.isclose(m["abs_rel"][0], s[3] / 5) and math.isclose(m["rmse"][0], math.sqrt(s[5] / 5))
    assert math.isclose(m["rmse_log"][0], math.sqrt(s[6] / 5))
    assert (m["a1"][0], m["a2"][0], m["a3"][0]) == (0.4, 0.8, 0.8)
    assert math.isclose(m["mask_precision"][0], 5 / 6) and math.isclose(m["mask_recall"][0], 5 / 6)
    assert math.isclose(m["mask_iou"][0], 5 / 7)


def _images(b, h, w, seed, dropped=0.3):
    g = torch.Generator().manual_seed(seed)
    x = torch.tanh(torch.randn(b, 1, h, w, generator=g) * 0.8 - 0.2)
    return torch.where(torch.rand(b, 1, h, w, generator=g) < dropped, torch.full_like(x, -1.0), x)


def test_identical_images_give_zero_errors_and_full_accuracy():
    x = _images(3, 8, 32, 1)
    m, v = od.metres_torch(x, 0.9, 120.0)
    s = od.sums_numpy(m.numpy(), v.numpy(), m.numpy(), v.numpy())
    r = od.finalise_numpy(s)
    for k in ("abs_rel", "sq_rel", "rmse", "rmse_log"):
        assert (r[k] == 0).all(), k
    for k in ("a1", "a2", "a3", "mask_precision", "mask_recall", "mask_iou"):
        assert (r[k] == 1).all(), k


def test_empty_scans_are_nan_and_left_out_of_the_mean():
    x, y = _images(3, 8, 32, 2), _images(3, 8, 32, 3)
    x[1] = -1.0                                                   # scan 1: prediction dropped entirely
    mx, vx = od.metres_torch(x, 0.9, 120.0)
    my, vy = od.metres_torch(y, 0.9, 120.0)
    s = od.sums_numpy(mx.numpy(), vx.numpy(), my.numpy(), vy.numpy())
    per = od.finalise_numpy(s)
    assert np.isnan(per["rmse"][1]) and np.isnan(per["mask_precision"][1]) and per["mask_recall"][1] == 0
    mean = od.mean_numpy(s)
    assert mean["#scans"] == 3 and mean["#empty"] == 1
    assert math.isclose(mean["rmse"], (per["rmse"][0] + per["rmse"][2]) / 2)


def test_torch_chain_agrees_with_the_float64_restatement():
    x, y = _images(4, 16, 64, 4), _images(4, 16, 64, 5, dropped=0.5)
    mx, vx = od.metres_torch(x, 0.9, 120.0)
    my, vy = od.metres_torch(y, 0.9, 120.0)
    want = od.sums_numpy(mx.numpy(), vx.numpy(), my.numpy(), vy.numpy())
    got = od.sums_torch(mx, vx, my, vy).numpy()
    assert np.array_equal(got[:, [0, 1, 2, 7, 8, 9]], want[:, [0, 1, 2, 7, 8, 9]])
    assert np.allclose(got, want, rtol=1e-12, atol=0)


def test_finaliser_matches_the_oracle():
    from dusty_gan_b200.utils.metrics.depth import KEYS, finalise
    assert KEYS == od.KEYS
    x, y = _images(5, 8, 32, 6), _images(5, 8, 32, 7)
    x[2] = -1.0
    y[3] = -1.0
    mx, vx = od.metres_torch(x, 0.9, 120.0)
    my, vy = od.metres_torch(y, 0.9, 120.0)
    s = od.sums_numpy(mx.numpy(), vx.numpy(), my.numpy(), vy.numpy())
    got, want = finalise(s), od.finalise_numpy(s)
    for k in KEYS:
        assert np.array_equal(got[k], want[k], equal_nan=True), k


def test_compute_depth_metrics_refuses_bad_arguments_before_any_launch():
    from dusty_gan_b200 import _lib
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    from dusty_gan_b200.utils.metrics.depth import compute_depth_metrics
    lidar = LiDAR(8, 32, 0.9, 120.0, angle=synthetic_hdl64e_angles())
    x = torch.zeros(2, 1, 8, 32)
    before = _lib.launch_count()
    with pytest.raises(RuntimeError, match="no CPU path"):
        compute_depth_metrics(x, x, lidar)
    odd = LiDAR(8, 30, 0.9, 120.0, angle=synthetic_hdl64e_angles())
    for a, b, lid, kw, msg in [(x, x[:1], lidar, {}, "differ in shape"),
                               (x, torch.zeros(2, 1, 8, 28), lidar, {}, "differ in shape"),
                               (x[:, 0], x[:, 0], lidar, {}, r"\(B,1,H,W\)"),
                               (x.expand(2, 2, 8, 32), x.expand(2, 2, 8, 32), lidar, {}, r"\(B,1,H,W\)"),
                               (x[..., :16], x[..., :16], lidar, {}, "LiDAR's range image"),
                               (torch.zeros(2, 1, 8, 30), torch.zeros(2, 1, 8, 30), odd, {}, "multiple of 4"),
                               (x, x, lidar, {"reduction": "sum"}, "reduction")]:
        with pytest.raises(ValueError, match=msg):
            compute_depth_metrics(a, b, lid, **kw)
    assert _lib.launch_count() == before


def test_c_abi_workspace_and_refusals_without_a_gpu():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    # 32 chunks of 1024 pixels per 64x512 scan, ten doubles each
    assert lib.dusty_depth_metrics_workspace_bytes(5000, 64, 512) == 5000 * 32 * 10 * 8
    assert lib.dusty_depth_metrics_workspace_bytes(3, 64, 2048) == 3 * 128 * 10 * 8
    assert lib.dusty_depth_metrics_workspace_bytes(1, 2, 4) == 10 * 8
    assert lib.dusty_depth_metrics_workspace_bytes(0, 64, 512) == 0
    assert lib.dusty_depth_metrics_workspace_bytes(1, 64, 510) == 0
    assert lib.dusty_depth_metrics(None, None, None, None, None, None, None, 0, None) == -1
    assert b"null params" in lib.dusty_last_error_string()
    p = _lib.HeadParams()
    for (b, h, w), msg in [((-1, 64, 512), b"bad shape"), ((1, 0, 512), b"bad shape"), ((1, 64, 510), b"multiple of 4"),
                           ((1, 65536, 65536), b"too large"), ((0x7FFFFFFF, 64, 2048), b"overflow the grid")]:
        p.b, p.h, p.w = b, h, w
        assert lib.dusty_depth_metrics(p, None, None, None, None, None, None, 0, None) == -1, (b, h, w)
        assert msg in lib.dusty_last_error_string(), (b, h, w)
    p.b, p.h, p.w = 0, 64, 512
    assert lib.dusty_depth_metrics(p, None, None, None, None, None, None, 0, None) == 0      # nothing to do


def test_depth_kernels_use_no_local_memory():
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-res-usage", _lib.LIB_PATH], text=True)
    usage = re.findall(r"Function (\S+):\s+REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    for frag in ("depth_chunk_kernel", "depth_combine_kernel"):
        rows = [u for u in usage if frag in u[0]]
        assert len(rows) == 1, (frag, rows)
        _, reg, stack, local = rows[0]
        assert int(stack) == 0 and int(local) == 0, (frag, reg, stack, local)
