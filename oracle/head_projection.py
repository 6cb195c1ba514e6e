"""Restatement of the point-drop head and the inverse projection as the element-wise ATen chains
the reference executes -- TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The arithmetic on this part of the path lives in PyTorch itself (module ``pytorch``, pinned 1.8.1 by
the reference's environment.yaml:5; the installed 2.11 is what runs here): sigmoid, log, reciprocal,
scalar mul/div, cos, sin. Every function below therefore issues the same torch ops in the same
order as the cited reference lines, on whatever device its inputs live on; run on the GPU it IS the
reference's rounding on that GPU (ATen's CUDA kernels multiply by a reciprocal where its CPU kernels
divide -- SURVEY.md trap T2 -- which is why the same-device run is the bit-exactness oracle).
"""
import torch
import torch.nn.functional as F


def logistic_noise(u1, u2, eps=1e-10):
    """reference models/dusty.py:35 given its two uniform draws (:33-34)."""
    return -torch.log(torch.log(u1 + eps) / torch.log(u2 + eps) + eps)


def gumbel_sigmoid(logits, noise, tau=1.0, threshold=0.5, hard=True):
    """reference models/dusty.py:38-59: noise is the logistic sample, fixed or fresh. ``tau`` is a Python scalar
    temperature (``x / tau``), or a 0-dim tensor holding the learnable inverse temperature
    ``softplus(weight) + 1/tau_max`` (tau=None, :39-41: ``x * inverse_tau``). ``hard=False`` returns the soft mask."""
    x = logits + (noise.expand(logits.shape[0], -1, -1, -1) if noise.shape[0] == 1 else noise)
    soft = torch.sigmoid(x * tau if isinstance(tau, torch.Tensor) else x / tau)
    if not hard:
        return soft
    mask_hard = (soft > threshold).float()
    return mask_hard - soft.detach() + soft


def maskout_dusty1(depth, confidence, noise, tau=1.0, threshold=0.5, drop_const=-1.0, hard=True):
    """reference models/dusty.py:77-91 -> (mask, depth_out)."""
    dc = torch.tensor(drop_const).float().to(depth.device)
    mask = gumbel_sigmoid(confidence, noise, tau, threshold, hard)
    return mask, mask * depth + (1 - mask) * dc


def maskout_dusty2(depth, confidence, noise_pixel, tau=1.0, threshold=0.5, drop_const=-1.0, noise_image=None,
                   hard=True, tau_image=None, hard_image=None):
    """reference models/dusty.py:107-127 -> (mask (B,2,H,W), depth_out); eval mode when noise_image is None.
    ``tau``/``hard`` are the pixel gate's; the image gate has its own ``tau_image``/``hard_image`` (None: the pixel
    gate's). Both gates see the same threshold, as in the reference."""
    dc = torch.tensor(drop_const).float().to(depth.device)
    mask_pixel = gumbel_sigmoid(confidence[:, [0]], noise_pixel, tau, threshold, hard)
    if noise_image is None:
        mask_image = (confidence[:, [1]] > 0.0).float()
    else:
        mask_image = gumbel_sigmoid(confidence[:, [1]], noise_image, tau if tau_image is None else tau_image, threshold,
                                    hard if hard_image is None else hard_image)
    mask = mask_pixel * mask_image
    return torch.cat([mask_pixel, mask_image], dim=1), mask * depth + (1 - mask) * dc


def tanh_to_sigmoid_clamped(x):
    """reference utils/__init__.py:76-79 followed by .clamp_(0, 1) (evaluate_synthesis.py:60)."""
    return ((x + 1.0) / 2.0).clamp_(0, 1)


def angle_grid(angles_2x64x2048, H, W):
    """reference utils/lidar.py:127-130."""
    return F.interpolate(angles_2x64x2048[None], size=(H, W), mode="bilinear")


def inv_to_xyz(inv_depth, angle, min_depth, max_depth, tol=1e-8, drop_const=0):
    """reference utils/lidar.py:61-68 with revert_depth (:38-47), normalize/denormalize_minmax
    (:23-29) and pol_to_xyz (:49-56) inlined in call order."""
    valid = torch.abs(inv_depth - drop_const) > tol
    disp = inv_depth * (1 / min_depth - 1 / max_depth) + 1 / max_depth      # denormalize_minmax
    depth = 1 / disp
    depth = (depth - min_depth) / (max_depth - min_depth)                    # normalize_minmax
    depth = depth * (max_depth - min_depth) + min_depth
    depth /= max_depth
    depth *= valid
    grid_cos = torch.cos(angle)
    grid_sin = torch.sin(angle)
    grid_x = depth * grid_cos[:, [0]] * grid_cos[:, [1]]
    grid_y = depth * grid_cos[:, [0]] * grid_sin[:, [1]]
    grid_z = depth * grid_sin[:, [0]]
    return torch.cat((grid_x, grid_y, grid_z), dim=1)


def project_2d_to_3d_dense(inv_tanh, angle, min_depth, max_depth, tol=0.0):
    """reference evaluate_synthesis.py:59-62 up to (and excluding) FPS -> points (B,N,3) contiguous."""
    xyz = inv_to_xyz(tanh_to_sigmoid_clamped(inv_tanh), angle, min_depth, max_depth, tol)
    return xyz.flatten(2).transpose(1, 2).contiguous()
