"""Approximate Earth Mover's Distance on libdustyb200.

Public names and call signatures are those of the reference module (utils/metrics/distance/emd/, the PyTorchEMD
interface): ``EarthMoverDistanceFunction`` and ``earth_mover_distance(xyz1, xyz2, transpose=True) -> cost (B,)``
with a backward pass. The match is the approxmatch plan of Fan et al. 2017; it counts as a constant in the
gradient, as in the reference. Instead of the reference's dense (B, M, N) match the forward saves ten per-level
factor vectors per pair, (B, 10, N + M) floats, from which the backward rebuilds the match.
"""
import torch

from ..... import _lib

__all__ = ["earth_mover_distance"]

LEVELS = 10


def _check_pair(xyz1, xyz2):
    for t, name in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        _lib.require_cuda(t, name)
    ok = xyz1.dim() == 3 and xyz2.dim() == 3 and xyz1.size(2) == 3 and xyz2.size(2) == 3 and xyz1.size(0) == xyz2.size(0)
    if not ok:
        raise ValueError(f"expected (B,N,3) and (B,M,3), got {tuple(xyz1.shape)} and {tuple(xyz2.shape)}")
    if xyz1.size(1) == 0 or xyz2.size(1) == 0:
        raise ValueError("clouds must hold at least one point (the approximate match divides by the point counts)")


def emd_forward(a, b, keep_factors=True):
    """a (B,N,3), b (B,M,3) contiguous CUDA f32 -> (cost (B,), factors (B,10,N+M) or None)."""
    B, N, M = a.size(0), a.size(1), b.size(1)
    cost = torch.empty(B, device=a.device, dtype=torch.float32)
    factors = torch.empty(B, LEVELS, N + M, device=a.device, dtype=torch.float32) if keep_factors else None
    lib = _lib.load()
    nbytes = lib.dusty_emd_forward_workspace_bytes(B, N, M)
    ws = _lib.workspace(nbytes, a.device)
    with torch.cuda.device(a.device):
        rc = lib.dusty_emd_forward(_lib.ptr(a), _lib.ptr(b), B, N, M, _lib.ptr(cost), _lib.ptr(factors), _lib.ptr(ws), nbytes,
                                   _lib.stream_of(a))
    _lib.check(rc, "dusty_emd_forward")
    return cost, factors


def emd_backward(a, b, factors, grad_cost):
    ga, gb = torch.empty_like(a), torch.empty_like(b)
    lib = _lib.load()
    with torch.cuda.device(a.device):
        rc = lib.dusty_emd_backward(_lib.ptr(a), _lib.ptr(b), a.size(0), a.size(1), b.size(1), _lib.ptr(grad_cost),
                                    _lib.ptr(factors), _lib.ptr(ga), _lib.ptr(gb), None, 0, _lib.stream_of(a))
    _lib.check(rc, "dusty_emd_backward")
    return ga, gb


class EarthMoverDistanceFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2):
        _check_pair(xyz1, xyz2)
        a, b = xyz1.contiguous(), xyz2.contiguous()
        grad = any(ctx.needs_input_grad)
        cost, factors = emd_forward(a, b, keep_factors=grad)
        if grad:
            ctx.save_for_backward(a, b, factors)
        return cost

    @staticmethod
    def backward(ctx, grad_cost):
        a, b, factors = ctx.saved_tensors
        return emd_backward(a, b, factors, grad_cost.contiguous().float())


def earth_mover_distance(xyz1, xyz2, transpose=True):
    """Approximate EMD of each cloud pair. ``transpose=True`` takes (B,3,N) and (B,3,M); ``transpose=False`` takes
    (B,N,3) and (B,M,3). 2-D inputs are one cloud each. Returns the match cost (B,), not divided by the point
    count. CUDA tensors only."""
    if xyz1.dim() == 2:
        xyz1 = xyz1.unsqueeze(0)
    if xyz2.dim() == 2:
        xyz2 = xyz2.unsqueeze(0)
    if transpose:
        xyz1 = xyz1.transpose(1, 2)
        xyz2 = xyz2.transpose(1, 2)
    return EarthMoverDistanceFunction.apply(xyz1, xyz2)
