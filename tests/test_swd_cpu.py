"""Sliced Wasserstein distance without a GPU: the float64 oracle against the published op chain (oracle/swd.py), the
wrapper's draws against the published draws, the C ABI's workspace queries and refusals, the wrapper's argument
checks and the register budget of the SWD kernels."""
import re
import subprocess

import numpy as np
import pytest
import torch

from oracle import swd as oswd


def _torch_and_draws(x1, x2, seed, **kw):
    draws = []
    torch.manual_seed(seed)
    per_level = oswd.swd_torch(x1, x2, return_by_resolution=True, draws=draws, **kw)
    return per_level.numpy().astype(np.float64), draws


@pytest.mark.parametrize("n,c,h,w", [(4, 1, 64, 512), (3, 3, 32, 64)])
def test_float64_oracle_agrees_with_the_published_op_chain(n, c, h, w):
    x1, x2 = oswd.range_images(n, c, h, w, 1), oswd.range_images(n, c, h, w, 2)
    want, draws = _torch_and_draws(x1, x2, 5)
    got = oswd.swd_numpy(x1.numpy(), x2.numpy(), [p.numpy() for p, _ in draws], [d.numpy() for _, d in draws],
                         oswd.default_pyramids(h))
    assert len(got) == oswd.default_pyramids(h) + 1
    assert (np.abs(got - want) <= 1e-5 * np.abs(want)).all(), (got, want)


def _oracle(x1, x2, seed=3):
    from dusty_gan_b200.utils.metrics.swd import draw
    n, c, h, w = x1.shape
    torch.manual_seed(seed)
    dr = draw(h, w, c, oswd.default_pyramids(h))
    return oswd.swd_numpy(x1, x2, [p.numpy() for p, _ in dr], [d.numpy() for _, d in dr], oswd.default_pyramids(h))


def test_oracle_properties():
    x1 = oswd.range_images(3, 1, 64, 256, 7).numpy()
    x2 = oswd.range_images(3, 1, 64, 256, 8).numpy()
    base = _oracle(x1, x2)
    assert (base > 0).all()
    assert (_oracle(x1, x1) == 0).all()                                     # self distance
    assert np.array_equal(_oracle(x2, x1), base)                            # symmetric
    assert (np.abs(_oracle(3 * x1, x2) - base) <= 1e-5 * base).all()        # per-set normalisation
    const1, const2 = np.full_like(x1, 0.3), np.full_like(x1, 0.7)
    # two constant sets of one sign normalise to the same rows up to the 1e-8 of (std + 1e-8)
    assert (_oracle(const1, const2) <= 1e-5 * base).all()
    assert (_oracle(const1, const1) == 0).all() and (_oracle(0 * x1, 0 * x2) == 0).all()
    shifted = _oracle(x1 + 0.5, x2)                                         # zero padding: not shift invariant
    assert (np.abs(shifted - base) > 1e-3 * base).any()


@pytest.mark.parametrize("kw", [{}, {"n_pyramids": 1, "n_descriptors": 37, "proj_per_repeat": 3,
                                     "n_repeat_projection": 5}])
def test_wrapper_draws_equal_the_published_draws(kw):
    from dusty_gan_b200.utils.metrics.swd import draw
    x1, x2 = oswd.range_images(1, 1, 64, 128, 1), oswd.range_images(1, 1, 64, 128, 2)
    _, want = _torch_and_draws(x1, x2, 11, **kw)
    torch.manual_seed(11)
    got = draw(64, 128, 1, kw.get("n_pyramids", 2), kw.get("n_descriptors", 128), kw.get("n_repeat_projection", 128),
               kw.get("proj_per_repeat", 4))
    assert len(got) == len(want)
    for (p, d), (wp, wd) in zip(got, want):
        assert torch.equal(p, wp) and torch.equal(d, wd)
    assert got[0][1].shape == (49, kw.get("n_repeat_projection", 128) * kw.get("proj_per_repeat", 4))


def test_workspace_queries_and_argument_errors_without_a_gpu():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    # Gaussian levels 1 and 2 of 5000 64x512 images, then (mean, M2) per (level, channel, image)
    assert lib.dusty_swd_descriptors_workspace_bytes(5000, 1, 64, 512, 3, 128) == \
        5000 * (32 * 256 + 16 * 128) * 4 + 3 * 5000 * 2 * 8
    assert lib.dusty_swd_descriptors_workspace_bytes(0, 1, 64, 512, 3, 128) == 0
    # keys of both sets in two sort buffers: 512 directions in two balanced batches of 256 at 640 000 rows
    assert lib.dusty_swd_sliced_workspace_bytes(640000, 1, 512) == 16 * 640000 * 256
    assert lib.dusty_swd_sliced_workspace_bytes(512, 1, 512) == 16 * 512 * 512
    assert lib.dusty_swd_sliced_workspace_bytes(0, 1, 512) == 0

    def desc(n=2, c=1, h=64, w=512, levels=3, n_desc=128):
        return lib.dusty_swd_descriptors(None, n, c, h, w, levels, None, n_desc, None, None, None, 0, None)
    for kwargs, msg in [({"c": 0}, b"channels"), ({"c": 5}, b"channels"),
                        ({"h": 62}, b"not divisible"), ({"w": 510}, b"not divisible"),
                        ({"h": 16, "levels": 3}, b"smaller than the 7x7 patch"),
                        ({"h": 24, "w": 24, "levels": 3, "n_desc": 1}, b"smaller than the 7x7 patch"),
                        ({"h": 32, "w": 64, "levels": 3}, b"fewer than n_desc"),
                        ({"n": 1 << 24, "n_desc": 128}, b"overflow"),
                        ({"h": 65536, "w": 65536, "levels": 1}, b"overflow"),
                        ({"n": 1, "n_desc": 43827150}, b"overflow"),           # n_desc * 49 > 2^31 - 1
                        ({"n": 1, "c": 4, "n_desc": 10956788}, b"overflow"),   # n_desc * 4 * 49 > 2^31 - 1
                        ({"levels": 0}, b"levels"), ({"n_desc": 0}, b"n_desc")]:
        assert desc(**kwargs) == -1, kwargs
        assert msg in lib.dusty_last_error_string(), (kwargs, lib.dusty_last_error_string())

    def sliced(rows=100, c=1, n_dirs=8, begin=0, end=8, stride=1):
        return lib.dusty_swd_sliced(None, None, None, None, rows, c, None, n_dirs, begin, end, stride, None, None, 0,
                                    None)
    for kwargs, msg in [({"c": 5}, b"channels"), ({"rows": 0}, b"rows"), ({"rows": (1 << 30) + 1}, b"rows"),
                        ({"end": 9}, b"direction range"), ({"stride": 0}, b"direction range"),
                        ({"begin": -1}, b"direction range")]:
        assert sliced(**kwargs) == -1, kwargs
        assert msg in lib.dusty_last_error_string(), kwargs


def test_compute_swd_refuses_bad_arguments_before_any_launch():
    from dusty_gan_b200.utils.metrics.swd import compute_swd
    x = torch.zeros(2, 1, 64, 512)
    with pytest.raises(RuntimeError, match="no CPU path"):
        compute_swd(x, x)
    for a, b, kw, msg in [(x, x[:1], {}, "differ in shape"), (x[0], x[0], {}, r"\(N,C,H,W\)"),
                          (x, x, {"slice_size": 5}, "7x7"), (x.expand(2, 5, 64, 512),) * 2 + ({}, "channels"),
                          (x[..., :510], x[..., :510], {}, "not divisible"),
                          (x[:, :, :32], x[:, :, :32], {"n_pyramids": 3}, "smaller than the 7x7"),
                          (x[:, :, :32, :32], x[:, :, :32, :32], {}, "fewer than"),
                          (x[:, :, :8], x[:, :, :8], {}, "no default")]:
        with pytest.raises(ValueError, match=msg):
            compute_swd(a, b, **kw)


def test_swd_kernels_use_no_local_memory():
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-res-usage", _lib.LIB_PATH], text=True)
    usage = re.findall(r"Function (\S+):\s+REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    for frag in ("swd_down_kernel", "swd_patch_kernel", "swd_stats_kernel", "swd_project_kernel", "swd_radix_kernel",
                 "swd_absdiff_kernel"):
        rows = [u for u in usage if frag in u[0]]
        assert len(rows) == 1, (frag, rows)
        _, reg, stack, local = rows[0]
        assert int(stack) == 0 and int(local) == 0, (frag, reg, stack, local)
