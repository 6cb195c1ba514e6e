"""Speed of dusty_head_project_backward (not a test): batch 256 of 64x512 range images, DUSty-I / DUSty-II, fixed
and fresh noise, maskout alone and with the fused projection, without and with the gradients of the gates'
temperatures (``grad_inv_tau``: one per-CTA partial per gate, then one reduction pass), against autograd through the
reference's op chain (oracle.head_projection) on the same GPU.

    python tests/perf_head_backward.py

Algorithmic bytes per pixel: read depth 4, confidence 4C, the upstream gradients (depth 4, mask 4C, points 12 with
the projection) and fresh noise 8 (U1, U2 of the per-pixel gate; the image gate draws one pair per image); write
4 + 4C. The fixed noise map and the trig table are L2 resident and not counted. Two input/output sets alternate so
that no launch finds the previous launch's data in the 126 MB L2. Bandwidth is reported as a share of the HBM copy
bandwidth bench_micro/hbm_probe.py measures in the same run.
"""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from dusty_gan_b200 import _lib  # noqa: E402
from dusty_gan_b200.models.dusty import _projection_fields  # noqa: E402
from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles  # noqa: E402
from oracle import head_projection as hp  # noqa: E402

B, H, W = 256, 64, 512
SETS = 2


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        power = "unknown"
    return name, power


def hbm_copy_gbs():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench_micro", "hbm_probe.py")], text=True)
    return json.loads(out.strip().splitlines()[-1])["copy_1r_1w"]


def time_per_call(fns, reps=5, calls=20):
    """Best mean time per call (s) over ``reps`` windows of ``calls`` launches, alternating the buffer sets."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(calls):
            fns[i % len(fns)]()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) * 1e-3 / calls)
    return best


def gate(mode_fixed, per_pixel, noise):
    g = _lib.Gate()
    g.hard, g.inv_tau, g.eps = 1, np.float32(1.0), np.float32(1e-10)
    if mode_fixed:
        g.mode, g.noise_a, g.noise_b, g.batch_stride = _lib.NOISE_LOGISTIC, noise[0].data_ptr(), None, 0
    else:
        g.mode, g.noise_a, g.noise_b = _lib.NOISE_UNIFORM, noise[0].data_ptr(), noise[1].data_ptr()
        g.batch_stride = noise[0][0].numel()
    g.pixel_stride = 1 if per_pixel else 0
    return g


def main():
    lib = _lib.load()
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    peak = hbm_copy_gbs()
    lidar = LiDAR(H, W, 0.9, 120.0, angle=synthetic_hdl64e_angles()).cuda()
    trig = lidar.trig_table(dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    print(f"GPU: {name}, power limit {power}; HBM copy bandwidth (bench_micro/hbm_probe.py, same run): {peak:.0f} GB/s")
    print(f"batch {B} x {H}x{W}; time per backward call; algorithmic bytes per pixel; share of the copy bandwidth")
    rows = []
    for kind in (1, 2):
        for noise in ("fixed", "fresh"):
            fixed_p = [hp.logistic_noise(torch.rand(1, 1, H, W, device=dev, generator=gen),
                                         torch.rand(1, 1, H, W, device=dev, generator=gen))]
            fixed_i = [hp.logistic_noise(torch.rand(1, 1, 1, 1, device=dev, generator=gen),
                                         torch.rand(1, 1, 1, 1, device=dev, generator=gen))]
            sets = []
            for _ in range(SETS):
                s = {"depth": torch.tanh(torch.randn(B, 1, H, W, device=dev, generator=gen)),
                     "conf": torch.randn(B, kind, H, W, device=dev, generator=gen) * 2,
                     "gd": torch.randn(B, 1, H, W, device=dev, generator=gen),
                     "gm": torch.randn(B, kind, H, W, device=dev, generator=gen),
                     "gp": torch.randn(B, H * W, 3, device=dev, generator=gen)}
                s["out_d"], s["out_c"] = torch.empty_like(s["depth"]), torch.empty_like(s["conf"])
                s["out_tau"] = torch.empty(kind, device=dev)
                s["ws"] = _lib.workspace(lib.dusty_head_project_backward_workspace_bytes(B, H, W), dev)
                if noise == "fresh":
                    s["np"] = [torch.rand(B, 1, H, W, device=dev, generator=gen) for _ in range(2)]
                    s["ni"] = [torch.rand(B, 1, 1, 1, device=dev, generator=gen) for _ in range(2)]
                else:
                    s["np"], s["ni"] = fixed_p, fixed_i
                p = _lib.HeadParams()
                p.b, p.h, p.w, p.conf_channels, p.points_layout = B, H, W, kind, 1
                p.gate_pixel = gate(noise == "fixed", True, s["np"])
                p.gate_image = gate(noise == "fixed", False, s["ni"])
                p.threshold, p.drop_const = np.float32(0.5), np.float32(-1.0)
                _projection_fields(p, lidar, 0.0)
                s["p"] = p
                sets.append(s)
            for proj in (False, True):
                def launch(s=None, proj=proj, tau=False):
                    _lib.check(lib.dusty_head_project_backward(
                        C.byref(s["p"]), _lib.ptr(s["depth"]), _lib.ptr(s["conf"]), _lib.ptr(trig), _lib.ptr(s["gm"]),
                        _lib.ptr(s["gd"]), _lib.ptr(s["gp"] if proj else None), _lib.ptr(s["out_d"]),
                        _lib.ptr(s["out_c"]), _lib.ptr(s["out_tau"] if tau else None), _lib.ptr(s["ws"] if tau else None),
                        s["ws"].numel() if tau else 0, _lib.stream_of(s["depth"])), "dusty_head_project_backward")
                t = time_per_call([lambda s=s: launch(s) for s in sets])
                t_tau = time_per_call([lambda s=s: launch(s, tau=True) for s in sets])
                nbytes = 4 + 4 * kind + 4 + 4 * kind + (12 if proj else 0) + (8 if noise == "fresh" else 0) + 4 + 4 * kind
                gbs = nbytes * B * H * W / t / 1e9
                # the same backward through autograd of the reference's op chain
                s = sets[0]
                d = s["depth"].clone().requires_grad_(True)
                c = s["conf"].clone().requires_grad_(True)
                lp = s["np"][0] if noise == "fixed" else hp.logistic_noise(*s["np"])
                li = s["ni"][0] if noise == "fixed" else hp.logistic_noise(*s["ni"])
                if kind == 1:
                    mask, dout = hp.maskout_dusty1(d, c, lp)
                else:
                    mask, dout = hp.maskout_dusty2(d, c, lp, noise_image=li)
                outs, grads = [mask, dout], [s["gm"], s["gd"]]
                if proj:
                    outs.append(hp.project_2d_to_3d_dense(dout, lidar.angle, 0.9, 120.0, 0.0))
                    grads.append(s["gp"])
                t_ref = time_per_call([lambda: torch.autograd.backward(outs, grads, retain_graph=True)], reps=3, calls=5)
                del outs, grads, mask, dout, d, c
                row = {"dusty": kind, "noise": noise, "projection": proj, "us": round(t * 1e6, 1),
                       "us_with_grad_inv_tau": round(t_tau * 1e6, 1), "bytes_per_px": nbytes,
                       "GB_s": round(gbs), "frac_hbm_copy": round(gbs / peak, 3), "oracle_autograd_us": round(t_ref * 1e6, 1),
                       "speedup": round(t_ref / t, 1)}
                rows.append(row)
                print(json.dumps(row))
            del sets
            torch.cuda.empty_cache()
    print(json.dumps({"gpu": name, "power_limit": power, "hbm_copy_gbs": peak, "rows": rows}))


if __name__ == "__main__":
    main()
