"""Point-drop heads of DUSty-GAN on libdustyb200 (mirror of reference models/dusty.py).

Same class names, constructor arguments, attribute names (``fixed_noise``, ``drop_const``,
``gumbel``, ``gumbel_pixel``, ``gumbel_image``) and output-dict keys as the reference.
``utils.setup``'s fixed-noise forward pre-hook (reference utils/__init__.py:141-149) is registered on the
GumbelSigmoid modules; the fused heads do not call those modules, so ``_head_call`` runs their pre-hooks
itself before reading ``fixed_noise`` (``tests/test_gpu_head.py::test_setup_fixed_noise_hook_*``). The
element-wise chains run as single CUDA kernels through the C ABI, and so does their backward: ``maskout``,
``forward`` and ``pipeline.maskout_and_project(..., differentiable=True)`` carry gradients to the backbone's
``depth`` and ``confidence`` (and to each gate's learnable temperature) through ``dusty_head_project_backward``.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn
from torch.autograd.function import once_differentiable

from .. import _lib


def _run_forward_pre_hooks(module, logits):
    """The fused heads read a gate's state without going through ``Module.__call__``, so the gate's forward
    pre-hooks are run here, with the arguments ``__call__`` would pass. ``utils.setup(fix_noise=True)`` relies on
    one: its ``set_gumbel_noise`` hook freezes ``fixed_noise`` on the first call (reference
    utils/__init__.py:141-149). A hook that returns replacement inputs is not supported on the fused path."""
    for hook_id, hook in list(module._forward_pre_hooks.items()):
        if hook_id in getattr(module, "_forward_pre_hooks_with_kwargs", {}):
            result = hook(module, (logits,), {})
        else:
            result = hook(module, (logits,))
        if result is not None:
            raise NotImplementedError("a forward pre-hook that replaces the gate's input is not supported by the fused "
                                      "head; call GumbelSigmoid directly")


def _gate_struct(module, logits):
    """Describe ``module`` (a GumbelSigmoid) for ``logits`` (B,1,H,W): its own temperature, eps and ``hard`` flag,
    and how it supplies its noise.

    Returns (Gate, keepalive tensors). With ``fixed_noise`` set the same (1,1,H,W) map is shared by
    the whole batch (reference models/dusty.py:48-50); otherwise fresh U1, U2 are drawn with the
    same two RNG calls as the reference (models/dusty.py:33-34) and l is formed inside the kernel.
    """
    B, _, H, W = logits.shape
    g = _lib.Gate()
    g.hard = 1 if module.hard else 0
    g.inv_tau = module._inv_tau()
    g.eps = np.float32(module.eps)
    if module.fixed_noise is not None:
        noise = module.fixed_noise
        _lib.require_cuda(noise, "fixed_noise")
        noise = noise.contiguous()
        per_pixel = noise.shape[-2:] == (H, W)
        if not per_pixel and noise.shape[-2:] != (1, 1):
            raise ValueError(f"fixed_noise shape {tuple(noise.shape)} does not broadcast over {(H, W)}")
        if noise.shape[0] not in (1, B):
            raise ValueError(f"fixed_noise batch {noise.shape[0]} does not broadcast over {B}")
        g.mode = _lib.NOISE_LOGISTIC
        g.noise_a = noise.data_ptr()
        g.noise_b = None
        g.batch_stride = 0 if noise.shape[0] == 1 else noise[0].numel()
        g.pixel_stride = 1 if per_pixel else 0
        return g, (noise,)
    shape = (B, 1, H, W) if module.pixelwise else (B, 1, 1, 1)
    u1 = torch.rand(*shape, device=logits.device)
    u2 = torch.rand_like(u1)
    g.mode = _lib.NOISE_UNIFORM
    g.noise_a = u1.data_ptr()
    g.noise_b = u2.data_ptr()
    g.batch_stride = u1[0].numel()
    g.pixel_stride = 1 if module.pixelwise else 0
    return g, (u1, u2)


class _GumbelSigmoidFn(torch.autograd.Function):
    """Forward on the CUDA kernel; backward is the straight-through soft-sigmoid gradient
    (reference models/dusty.py:54-57: ``mask_hard - mask_soft.detach() + mask_soft``)."""

    @staticmethod
    def forward(ctx, logits, module, threshold, weight=None):
        _lib.require_cuda(logits, "logits")
        if logits.dim() != 4 or logits.shape[1] != 1:
            raise ValueError(f"expected (B,1,H,W) logits, got {tuple(logits.shape)}")
        x = logits.contiguous()
        B, _, H, W = x.shape
        gate, keep = _gate_struct(module, x)
        out = torch.empty_like(x)
        lib = _lib.load()
        with torch.cuda.device(x.device):
            _lib.check(lib.dusty_gumbel_sigmoid(_lib.ptr(x), C.byref(gate), np.float32(threshold), B, H * W,
                                                _lib.ptr(out), _lib.stream_of(x)), "dusty_gumbel_sigmoid")
        ctx.module = module
        # the soft mask is re-derived in backward from (logits, noise); keep the noise alive
        if gate.mode == _lib.NOISE_UNIFORM:
            noise = module._logistic_from_uniform(*keep)
        else:
            noise = keep[0]
        ctx.save_for_backward(x, noise)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        """Gradient of the soft mask (the straight-through estimator for hard=True; the value itself for
        hard=False), also with respect to the learnable temperature's weight. Off the evaluate path: torch ops."""
        x, noise = ctx.saved_tensors
        m = ctx.module
        if m.tau is not None:
            it = float(m._inv_tau())
            soft = torch.sigmoid((x + noise) * it)
            return grad_out * soft * (1 - soft) * it, None, None, None
        with torch.enable_grad():
            xin = x.detach().requires_grad_(True)
            soft = torch.sigmoid((xin + noise) * m._inverse_tau_tensor())
            gx, gw = torch.autograd.grad(soft, (xin, m.weight), grad_out)
        return gx, None, None, gw


class GumbelSigmoid(nn.Module):
    """Binary Gumbel-softmax gate with a hard straight-through output (reference models/dusty.py:6-62)."""

    def __init__(self, tau: float = 1.0, tau_max: float = 1.0, hard: bool = True, eps: float = 1e-10,
                 pixelwise: bool = True):
        super().__init__()
        self.tau = tau
        self.tau_max = tau_max
        self.hard = hard
        self.eps = eps
        if self.tau is None:
            self.weight = nn.Parameter(torch.tensor(0.0))
        self.pixelwise = pixelwise
        self.fixed_noise = None

    def _inverse_tau_tensor(self):
        """Learnable temperature (reference models/dusty.py:39-41): softplus(weight) + 1/tau_max, a 0-dim tensor."""
        return torch.nn.functional.softplus(self.weight) + 1.0 / self.tau_max

    def _inv_tau(self):
        if self.tau is None:
            # the reference multiplies the logits by this f32 tensor; its value is read back once per weight version
            key = (self.weight._version, self.weight.data_ptr())
            cached = getattr(self, "_inv_tau_cache", None)
            if cached is None or cached[0] != key:
                with torch.no_grad():
                    cached = (key, np.float32(self._inverse_tau_tensor().item()))
                object.__setattr__(self, "_inv_tau_cache", cached)
            return cached[1]
        # ATen's CUDA division by a Python scalar multiplies by the reciprocal, formed in double and
        # rounded to f32 once (SURVEY appendix, trap T2; torch 2.11 div_true_kernel_cuda)
        return np.float32(1.0 / self.tau)

    def _logistic_from_uniform(self, u1, u2):
        out = torch.empty_like(u1)
        lib = _lib.load()
        with torch.cuda.device(u1.device):
            _lib.check(lib.dusty_logistic_noise(_lib.ptr(u1), _lib.ptr(u2), np.float32(self.eps), u1.numel(),
                                                _lib.ptr(out), _lib.stream_of(u1)), "dusty_logistic_noise")
        return out

    def logistic_noise(self, logits):
        """l = -log(log(U1+eps)/log(U2+eps)+eps) with the reference's two RNG draws (models/dusty.py:30-36)."""
        _lib.require_cuda(logits, "logits")
        B, _, H, W = logits.shape
        shape = (B, 1, H, W) if self.pixelwise else (B, 1, 1, 1)
        u1 = torch.rand(*shape, device=logits.device)
        u2 = torch.rand_like(u1)
        return self._logistic_from_uniform(u1, u2)

    def forward(self, logits, threshold: float = 0.5):
        return _GumbelSigmoidFn.apply(logits, self, threshold, self.weight if self.tau is None else None)

    def extra_repr(self):
        return f"hard={self.hard}, eps={self.eps}"


def _projection_fields(params, lidar, tol):
    """Fill the projection scalars exactly as the reference's element-wise kernels receive them
    (reference utils/lidar.py:23-29,38-47,61-68): Python-double arithmetic on the config values,
    then one cast to f32; a division by a Python scalar is a multiply by f32(1/scalar), the reciprocal
    taken in double (torch 2.11 div_true_kernel_cuda)."""
    f32 = np.float32
    params.tol = f32(tol)
    params.disp_scale = f32(1 / lidar.min_depth - 1 / lidar.max_depth)
    params.disp_shift = f32(1 / lidar.max_depth)
    params.min_depth = f32(lidar.min_depth)
    params.range = f32(lidar.max_depth - lidar.min_depth)
    params.inv_range = f32(1.0 / (lidar.max_depth - lidar.min_depth))
    params.inv_max_depth = f32(1.0 / lidar.max_depth)


def _drop_value(module):
    """The drop_const buffer as a host float, read back once per buffer version (a per-call
    ``float(tensor)`` would put a device synchronisation on the hot path)."""
    key = (module.drop_const._version, module.drop_const.data_ptr())
    cached = getattr(module, "_drop_cache", None)
    if cached is None or cached[0] != key:
        cached = (key, float(module.drop_const))
        object.__setattr__(module, "_drop_cache", cached)
    return cached[1]


class _HeadFn(torch.autograd.Function):
    """``dusty_head_project`` as an autograd op: (depth, confidence, pixel gate's temperature weight, image gate's
    temperature weight) -> (mask, depth, points). ``launch`` runs the forward kernel into ``outputs``. The backward
    kernel rebuilds every forward value from the same inputs and noise, so the forward keeps only its inputs, its
    parameters (``params``, whose noise pointers stay valid because ``keep`` holds the noise tensors), the trig table
    and the gate modules (``gates``: pixel gate, image gate or None)."""

    @staticmethod
    def forward(ctx, depth, conf, weight_pixel, weight_image, launch, outputs, params, trig, keep, gates):
        ctx.set_materialize_grads(False)
        launch()
        ctx.params, ctx.trig, ctx.keep, ctx.gates = params, trig, keep, gates
        ctx.save_for_backward(depth, conf)
        return outputs

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mask, g_depth, g_points):
        depth, conf = ctx.saved_tensors
        lib = _lib.load()
        grads = [None if g is None else g.contiguous() for g in (g_mask, g_depth, g_points)]
        grad_depth = torch.empty_like(depth)
        grad_conf = torch.empty_like(conf)
        want_tau = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        p = ctx.params
        # d loss / d inv_tau of each gate: pixel, then (DUSty-II) image
        grad_tau = torch.empty(p.conf_channels, device=depth.device, dtype=torch.float32) if want_tau else None
        ws_bytes = lib.dusty_head_project_backward_workspace_bytes(p.b, p.h, p.w) if want_tau else 0
        ws = _lib.workspace(ws_bytes, depth.device) if want_tau else None
        with torch.cuda.device(depth.device):
            _lib.check(lib.dusty_head_project_backward(
                C.byref(p), _lib.ptr(depth), _lib.ptr(conf), _lib.ptr(ctx.trig if grads[2] is not None else None),
                *(_lib.ptr(g) for g in grads), _lib.ptr(grad_depth), _lib.ptr(grad_conf), _lib.ptr(grad_tau),
                _lib.ptr(ws), ws_bytes, _lib.stream_of(depth)), "dusty_head_project_backward")
        grad_weights = [None, None]
        for i, gate in enumerate(ctx.gates):
            if ctx.needs_input_grad[2 + i]:     # inv_tau = softplus(weight) + 1/tau_max (reference models/dusty.py:39-41)
                with torch.enable_grad():
                    (grad_weights[i],) = torch.autograd.grad(gate._inverse_tau_tensor(), gate.weight, grad_tau[i])
        return (grad_depth if ctx.needs_input_grad[0] else None, grad_conf if ctx.needs_input_grad[1] else None,
                *grad_weights, None, None, None, None, None, None)


def _head_call(module, output, threshold, lidar=None, tol=1e-8, points_layout=1, compact=False, buffers=None):
    """Shared body of maskout (lidar=None) and the fused generate->points path (lidar given).
    ``buffers`` may hold preallocated ``mask``, ``depth``, ``points`` (and, for ``compact``, ``valid_count``,
    ``valid_index``, ``valid_points``, ``workspace``) tensors to write into (steady-state callers reuse them; the
    evaluate loop of the reference reallocates every batch).

    When grad mode is on and ``depth`` or ``confidence`` requires grad, the launch runs inside ``_HeadFn``: the
    returned mask, depth and points then carry gradients (compaction outputs excepted)."""
    buffers = buffers or {}
    assert isinstance(output, dict)
    assert "confidence" in output
    assert "depth" in output
    depth, conf = output["depth"], output["confidence"]
    _lib.require_cuda(depth, "depth")
    _lib.require_cuda(conf, "confidence")
    channels = 2 if isinstance(module, DUSty2) else 1
    if depth.dim() != 4 or depth.shape[1] != 1 or conf.shape != (depth.shape[0], channels, *depth.shape[2:]):
        raise ValueError(f"expected depth (B,1,H,W) and confidence (B,{channels},H,W), got "
                         f"{tuple(depth.shape)} and {tuple(conf.shape)}")
    differentiable = torch.is_grad_enabled() and (depth.requires_grad or conf.requires_grad)
    d, c = depth.contiguous(), conf.contiguous()
    B, _, H, W = d.shape
    p = _lib.HeadParams()
    p.b, p.h, p.w, p.conf_channels = B, H, W, channels
    keep = []
    if channels == 1:
        _run_forward_pre_hooks(module.gumbel, c)
        p.gate_pixel, k = _gate_struct(module.gumbel, c)
        keep.append(k)
        gates = (module.gumbel, None)
    else:
        _run_forward_pre_hooks(module.gumbel_pixel, c[:, :1])
        p.gate_pixel, k = _gate_struct(module.gumbel_pixel, c[:, :1])
        keep.append(k)
        if module.training:     # the reference calls the image gate in training mode only (models/dusty.py:117-120)
            _run_forward_pre_hooks(module.gumbel_image, c[:, 1:])
            p.gate_image, k = _gate_struct(module.gumbel_image, c[:, 1:])
            keep.append(k)
            gates = (module.gumbel_pixel, module.gumbel_image)
        else:
            p.gate_image.mode = _lib.NOISE_NONE     # (logit > 0), reference models/dusty.py:120
            gates = (module.gumbel_pixel, None)
    p.threshold = np.float32(threshold)
    p.drop_const = np.float32(_drop_value(module))
    p.points_layout = points_layout
    mask = buffers["mask"] if "mask" in buffers else torch.empty_like(c)
    dout = buffers["depth"] if "depth" in buffers else torch.empty_like(d)
    for t, like in ((mask, c), (dout, d)):
        if t.shape != like.shape or t.dtype != torch.float32 or t.device != d.device or not t.is_contiguous():
            raise ValueError("preallocated buffer does not match the expected shape/dtype/device")
    points = count = index = compacted = trig = ws = None
    if lidar is not None:
        _projection_fields(p, lidar, tol)
        trig = lidar.trig_table(d.device)
        pshape = (B, H * W, 3) if points_layout == 1 else (B, 3, H, W)
        points = buffers["points"] if "points" in buffers else torch.empty(pshape, device=d.device, dtype=torch.float32)
        if tuple(points.shape) != pshape or points.dtype != torch.float32 or not points.is_contiguous():
            raise ValueError("preallocated points buffer does not match the expected shape/dtype")
        if compact:
            def scratch(name, shape, dtype):
                t = buffers.get(name)
                if t is None:
                    return torch.empty(shape, device=d.device, dtype=dtype)
                if tuple(t.shape) != shape or t.dtype != dtype or t.device != d.device or not t.is_contiguous():
                    raise ValueError(f"preallocated {name} buffer does not match {shape} {dtype}")
                return t
            count = scratch("valid_count", (B,), torch.int32)
            index = scratch("valid_index", (B, H * W), torch.int32)
            compacted = scratch("valid_points", (B, H * W, 3), torch.float32)
    lib = _lib.load()
    ws_bytes = lib.dusty_head_project_workspace_bytes(B, H, W) if compact else 0
    ws = (buffers.get("workspace") if buffers.get("workspace") is not None else _lib.workspace(ws_bytes, d.device)) if compact else None
    if ws is not None and ws.numel() < ws_bytes:
        raise ValueError("preallocated workspace is too small")
    def launch():
        with torch.cuda.device(d.device):
            _lib.check(lib.dusty_head_project(C.byref(p), _lib.ptr(d), _lib.ptr(c), _lib.ptr(trig), _lib.ptr(mask),
                                              _lib.ptr(dout), _lib.ptr(points), _lib.ptr(count), _lib.ptr(index),
                                              _lib.ptr(compacted), _lib.ptr(ws), ws_bytes, _lib.stream_of(d)),
                       "dusty_head_project")
    if differentiable:
        weights = [g.weight if g is not None and g.tau is None else None for g in gates]
        mask, dout, points = _HeadFn.apply(d, c, *weights, launch, (mask, dout, points), p, trig, keep, gates)
    else:
        launch()
    output["depth_orig"] = depth
    output["mask"] = mask
    output["depth"] = dout
    return output, points, count, index, compacted


class DUSty1(nn.Module):
    """Pixel-wise measurability head (reference models/dusty.py:65-91)."""

    def __init__(self, backbone, tau, drop_const=-1):
        super().__init__()
        self.backbone = backbone
        self.gumbel = GumbelSigmoid(hard=True, tau=tau, pixelwise=True)
        self.register_buffer("drop_const", torch.tensor(drop_const).float())

    def forward(self, latent, **kwargs):
        output = self.backbone(latent, **kwargs)
        output = self.maskout(output)
        return output

    def maskout(self, output, threshold=0.5):
        return _head_call(self, output, threshold)[0]


class DUSty2(nn.Module):
    """Pixel-wise x image-wise measurability head (reference models/dusty.py:94-127)."""

    def __init__(self, backbone, tau, drop_const=-1):
        super().__init__()
        self.backbone = backbone
        self.gumbel_pixel = GumbelSigmoid(hard=True, tau=tau, pixelwise=True)
        self.gumbel_image = GumbelSigmoid(hard=True, tau=tau, pixelwise=False)
        self.register_buffer("drop_const", torch.tensor(drop_const).float())

    def forward(self, latent, **kwargs):
        output = self.backbone(latent, **kwargs)
        output = self.maskout(output)
        return output

    def maskout(self, output, threshold=0.5):
        return _head_call(self, output, threshold)[0]
