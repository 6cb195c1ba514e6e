"""Seeded synthetic inputs shared by the tests (and mirrored by bench.py)."""
import numpy as np
import torch


def lidar_like_clouds(n_clouds, n_points, seed, dropped=0.3, near=0.15):
    """(n,P,3) f32 clouds shaped like projected range images: points on rings around the sensor at
    normalised range in (0,1], a fraction exactly at the origin (dropped pixels) and a fraction
    inside the FPS exclusion radius (|p|^2 <= 1e-3)."""
    rng = np.random.default_rng(seed)
    az = rng.uniform(-np.pi, np.pi, (n_clouds, n_points))
    el = np.deg2rad(rng.uniform(-24.8, 2.0, (n_clouds, n_points)))
    r = np.exp(rng.uniform(np.log(0.035), np.log(0.7), (n_clouds, n_points)))
    r = np.where(rng.uniform(size=r.shape) < near, rng.uniform(0.008, 0.03, r.shape), r)
    r = np.where(rng.uniform(size=r.shape) < dropped, 0.0, r)
    xyz = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], -1)
    return xyz.astype(np.float32)


def sampled_clouds(n_clouds, n_points, seed):
    """FPS-like clouds: no dropped points, ranges spread over the scene."""
    return lidar_like_clouds(n_clouds, n_points, seed, dropped=0.0, near=0.0)


def head_inputs(B, C, H, W, seed, device="cpu", calibrated=True):
    """Backbone-like outputs: depth in tanh space, confidence logits, U1/U2 for the fixed noise."""
    g = torch.Generator().manual_seed(seed)
    depth = torch.tanh(torch.randn(B, 1, H, W, generator=g) * (1.2 if calibrated else 0.115) - (0.3 if calibrated else 0.04))
    conf = torch.randn(B, C, H, W, generator=g) * 2.0
    u1 = torch.rand(1, 1, H, W, generator=g)
    u2 = torch.rand(1, 1, H, W, generator=g)
    return depth.to(device), conf.to(device), u1.to(device), u2.to(device)


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-30)


def oracle_gate_settings(gate):
    """(tau, hard, leaf) of a GumbelSigmoid module as oracle.head_projection.gumbel_sigmoid takes them: its scalar
    temperature, or for tau=None the inverse temperature softplus(w) + 1/tau_max of a detached copy w of its weight
    (reference models/dusty.py:39-41), returned as ``leaf`` so that a test can read ``w.grad``; None otherwise."""
    if gate.tau is not None:
        return gate.tau, gate.hard, None
    w = gate.weight.detach().clone().requires_grad_(True)
    return torch.nn.functional.softplus(w) + 1.0 / gate.tau_max, gate.hard, w


def oracle_head_noise(head, B, H, W, seed=None):
    """The logistic noise each gate of ``head`` (DUSty1 or DUSty2, in its current mode) read: its ``fixed_noise`` or
    the reference's two RNG draws (models/dusty.py:33-34) with the gate's own eps, replayed after
    ``torch.manual_seed(seed)`` in the head's order (pixel gate, then the image gate, which only training mode calls).
    Returns (noise_pixel, noise_image); noise_image is None when the image gate is not called."""
    from oracle import head_projection as hp
    if seed is not None:
        torch.manual_seed(seed)
    gates = [head.gumbel] if hasattr(head, "gumbel") else [head.gumbel_pixel] + ([head.gumbel_image] if head.training else [])
    noise = []
    for g in gates:
        if g.fixed_noise is not None:
            noise.append(g.fixed_noise)
            continue
        u1 = torch.rand(*((B, 1, H, W) if g.pixelwise else (B, 1, 1, 1)), device="cuda")
        u2 = torch.rand_like(u1)
        noise.append(hp.logistic_noise(u1, u2, g.eps))
    return noise[0], (noise[1] if len(noise) > 1 else None)


def oracle_head_maskout(head, depth, confidence, noise_pixel, noise_image, threshold=0.5):
    """``head.maskout`` through the reference's op chain (oracle.head_projection), each gate with its own temperature
    and ``hard`` flag. Returns (mask, depth_out, (w_pixel, w_image)): the weight copies of the tau=None gates whose
    ``.grad`` autograd fills (None for a gate with a fixed temperature or one that is not called)."""
    from oracle import head_projection as hp
    drop = float(head.drop_const)
    if hasattr(head, "gumbel"):
        tau, hard, w = oracle_gate_settings(head.gumbel)
        mask, dout = hp.maskout_dusty1(depth, confidence, noise_pixel, tau, threshold, drop, hard)
        return mask, dout, (w, None)
    tau_p, hard_p, wp = oracle_gate_settings(head.gumbel_pixel)
    tau_i, hard_i, wi = oracle_gate_settings(head.gumbel_image) if noise_image is not None else (None, None, None)
    mask, dout = hp.maskout_dusty2(depth, confidence, noise_pixel, tau_p, threshold, drop, noise_image, hard_p, tau_i,
                                   hard_i)
    return mask, dout, (wp, wi)
