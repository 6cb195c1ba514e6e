"""Backward of the fused head (dusty_head_project_backward) without a GPU: the workspace query, argument errors
reported with a message before any device is touched, and the register budget of its kernels."""
import re
import subprocess

import pytest

DUSTY_EINVAL, DUSTY_EALIGN, DUSTY_ENOSPACE = -1, -2, -3


def params(b=2, h=8, w=16, channels=1, layout=1):
    from dusty_gan_b200 import _lib
    p = _lib.HeadParams()
    p.b, p.h, p.w, p.conf_channels, p.points_layout = b, h, w, channels, layout
    p.gate_pixel.mode = _lib.NOISE_LOGISTIC
    p.gate_pixel.noise_a = 0x10000
    p.gate_pixel.pixel_stride = 1
    p.gate_image.mode = _lib.NOISE_NONE
    return p


def backward(p, depth=0x20000, conf=0x30000, trig=None, grad_mask=None, grad_depth=0x40000, grad_points=None,
             grad_depth_in=0x50000, grad_conf=0x60000, grad_tau=None, ws=None, ws_bytes=0):
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    return lib.dusty_head_project_backward(p, depth, conf, trig, grad_mask, grad_depth, grad_points, grad_depth_in,
                                           grad_conf, grad_tau, ws, ws_bytes, None)


def error():
    from dusty_gan_b200 import _lib
    return _lib.load().dusty_last_error_string().decode()


def test_workspace_query_without_a_gpu():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    assert lib.dusty_head_project_backward_workspace_bytes(256, 64, 512) == 2 * 256 * 32 * 4  # one float per gate and CTA
    assert lib.dusty_head_project_backward_workspace_bytes(3, 8, 20) == 256                    # rounded up to 256 B
    assert lib.dusty_head_project_backward_workspace_bytes(0, 64, 512) == 0
    assert lib.dusty_head_project_backward_workspace_bytes(2, 0, 512) == 0


@pytest.mark.parametrize("case,code,message", [
    ("null params", DUSTY_EINVAL, "null params"),
    ("w not a multiple of 4", DUSTY_EINVAL, "multiple of 4"),
    ("bad layout", DUSTY_EINVAL, "points_layout"),
    ("bad channels", DUSTY_EINVAL, "conf_channels"),
    ("null depth", DUSTY_EINVAL, "null pointer"),
    ("null grad_confidence", DUSTY_EINVAL, "null pointer"),
    ("grad_points without trig", DUSTY_EINVAL, "null pointer"),
    ("misaligned depth", DUSTY_EALIGN, "16-byte aligned"),
    ("misaligned grad_mask", DUSTY_EALIGN, "16-byte aligned"),
    ("misaligned grad_points", DUSTY_EALIGN, "16-byte aligned"),
    ("gate without noise pointer", DUSTY_EINVAL, "needs noise_a"),
    ("gate hard flag not 0 or 1", DUSTY_EINVAL, "hard must be 0 or 1"),
    ("grad_inv_tau without workspace", DUSTY_ENOSPACE, "workspace bytes"),
])
def test_argument_errors_are_reported_without_a_gpu(case, code, message):
    p = params()
    kw = {}
    if case == "null params":
        p = None
    elif case == "w not a multiple of 4":
        p.w = 18
    elif case == "bad layout":
        p.points_layout = 2
    elif case == "bad channels":
        p.conf_channels = 3
    elif case == "null depth":
        kw["depth"] = None
    elif case == "null grad_confidence":
        kw["grad_conf"] = None
    elif case == "grad_points without trig":
        kw["grad_points"] = 0x70000
    elif case == "misaligned depth":
        kw["depth"] = 0x20004
    elif case == "misaligned grad_mask":
        kw["grad_mask"] = 0x80008
    elif case == "misaligned grad_points":
        kw.update(grad_points=0x7000c, trig=0x90000)
    elif case == "gate without noise pointer":
        p.gate_pixel.noise_a = None
    elif case == "gate hard flag not 0 or 1":
        p.gate_pixel.hard = 2
    elif case == "grad_inv_tau without workspace":
        kw["grad_tau"] = 0xa0000
    assert backward(p, **kw) == code, case
    assert message in error(), (case, error())


def test_backward_kernels_keep_their_register_budget():
    """One instantiation per (channels, projection): no spills, no local memory, and the registers ptxas gave them
    when they were written (DUSty-I / DUSty-II: 42 / 64 without the projection, 70 / 80 with it; at 256 threads per
    CTA that is 5, 4, 3 and 3 CTAs per SM)."""
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-res-usage", _lib.LIB_PATH], text=True)
    usage = re.findall(r"Function (\S+):\s+REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    bounds = {"head_backward_kernelILi1ELb0E": 42, "head_backward_kernelILi2ELb0E": 64,
              "head_backward_kernelILi1ELb1E": 70, "head_backward_kernelILi2ELb1E": 80}
    for frag, bound in bounds.items():
        rows = [u for u in usage if frag in u[0]]
        assert len(rows) == 1, (frag, rows)
        _, reg, stack, local = rows[0]
        assert int(reg) <= bound and int(stack) == 0 and int(local) == 0, (frag, reg, stack, local)
    assert len([u for u in usage if "head_backward_kernel" in u[0]]) == 4
