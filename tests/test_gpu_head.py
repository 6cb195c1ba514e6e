"""Fused head + projection: bit-exact against the reference's op chain (oracle.head_projection) run
on the same GPU, and against the golden CPU vectors up to ATen's CPU/CUDA last-ulp differences."""
import math

import numpy as np
import pytest
import torch

from helpers import head_inputs, oracle_head_maskout, oracle_head_noise
from oracle import head_projection as hp

pytestmark = pytest.mark.gpu


def make_lidar(H, W):
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    return LiDAR(H, W, 0.9, 120.0, angle=synthetic_hdl64e_angles()).cuda()


def bits(t):
    return t.contiguous().view(torch.int32)


def assert_bit_equal(a, b, what):
    assert a.shape == b.shape, what
    same = (bits(a) == bits(b)) | (torch.isnan(a) & torch.isnan(b))
    assert bool(same.all()), f"{what}: {(~same).sum().item()} of {same.numel()} differ"


@pytest.mark.parametrize("kind", [1, 2])
@pytest.mark.parametrize("shape,compaction", [((5, 64, 512), "segment"), ((3, 16, 64), "segment"), ((2, 8, 20), "segment"),
                                              ((5, 64, 512), "image"), ((2, 8, 20), "image"), ((3, 40, 100), "image"),
                                              ((130, 64, 512), None)])
def test_fixed_noise_bit_exact_on_device(kind, shape, compaction, monkeypatch):
    """``compaction`` forces one of the two ordered-compaction kernels (None: the library's own choice, which is
    one CTA per image from 128 images on)."""
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2
    from dusty_gan_b200 import pipeline
    if compaction:
        monkeypatch.setenv("DUSTY_HEAD_COMPACT", compaction)
    B, H, W = shape
    depth, conf, u1, u2 = head_inputs(B, kind, H, W, 42 + kind, "cuda")
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=1.0).cuda().eval()
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    gate.fixed_noise = gate._logistic_from_uniform(u1, u2)
    noise = hp.logistic_noise(u1, u2)
    assert_bit_equal(gate.fixed_noise, noise, "logistic noise")
    lidar = make_lidar(H, W)
    out = head.maskout({"depth": depth.clone(), "confidence": conf.clone()})
    if kind == 1:
        mask, dout = hp.maskout_dusty1(depth, conf, noise)
    else:
        mask, dout = hp.maskout_dusty2(depth, conf, noise)
    assert_bit_equal(out["mask"], mask, "mask")
    assert_bit_equal(out["depth"], dout, "depth")
    assert out["depth_orig"] is depth or torch.equal(out["depth_orig"], depth)
    # fused path: mask + projection + (B,N,3) layout + compaction in one launch
    fused = pipeline.maskout_and_project(head, {"depth": depth.clone(), "confidence": conf.clone()}, lidar, tol=0.0, compact=True)
    pts = hp.project_2d_to_3d_dense(dout, lidar.angle, 0.9, 120.0, 0.0)
    assert_bit_equal(fused["mask"], mask, "fused mask")
    assert_bit_equal(fused["depth"], dout, "fused depth")
    assert_bit_equal(fused["points"], pts, "fused points")
    valid = hp.tanh_to_sigmoid_clamped(dout).flatten(1) != 0
    assert torch.equal(fused["valid_count"].long(), valid.sum(1))
    for b in range(B):
        k = int(valid[b].sum())
        assert torch.equal(fused["valid_index"][b, :k].long(), torch.nonzero(valid[b]).flatten())
        assert_bit_equal(fused["valid_points"][b, :k], pts[b][valid[b]], "compacted points")


def _diverged_weights(head):
    with torch.no_grad():
        head.gumbel_pixel.weight.fill_(0.37)
        head.gumbel_image.weight.fill_(-1.2)


# name -> (kind, training, tau of the constructor, per-gate setup): each gate's own temperature, eps and hard flag
GATE_CASES = {
    "dusty1_learnable": (1, False, None, lambda h: h.gumbel.weight.data.fill_(0.37)),
    "dusty1_soft": (1, False, 1.0, lambda h: setattr(h.gumbel, "hard", False)),
    "dusty2_diverged_learnable": (2, True, None, _diverged_weights),
    "dusty2_image_tau": (2, True, 0.7, lambda h: setattr(h.gumbel_image, "tau", 1.9)),
    "dusty2_soft_pixel": (2, True, 1.0, lambda h: setattr(h.gumbel_pixel, "hard", False)),
    "dusty2_soft_image": (2, True, 1.0, lambda h: setattr(h.gumbel_image, "hard", False)),
    "dusty2_image_eps": (2, True, 1.0, lambda h: setattr(h.gumbel_image, "eps", 0.05)),
}


@pytest.mark.parametrize("noise", ["fixed", "fresh"])
@pytest.mark.parametrize("threshold", [0.3, 0.5, 0.7, float("nan")])
@pytest.mark.parametrize("case", list(GATE_CASES))
def test_each_gate_keeps_its_own_settings_bit_exact_on_device(case, threshold, noise, monkeypatch):
    """Every gate is computed with its own temperature (fixed or learnable), eps and ``hard`` flag, as the reference's
    GumbelSigmoid modules are, and one threshold serves both gates. A NaN threshold is no sentinel: a hard gate then
    gives the reference's exact zeros. Checked through maskout, the fused projection in both point layouts and both
    compaction kernels (each has its own gate code). At threshold 0.5 the hard mask does not depend on the
    temperature; 0.3 and 0.7 are where a wrong temperature flips mask values."""
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2, _head_call
    kind, training, tau, setup = GATE_CASES[case]
    B, H, W = 3, 40, 100                          # 4000 pixels: a partial last segment and a partial last image step
    depth, conf, _, _ = head_inputs(B, kind, H, W, 60 + kind, "cuda")
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=tau).cuda().train(training)
    setup(head)
    if noise == "fixed":
        g = torch.Generator().manual_seed(61)
        for gate, shape in ([(head.gumbel, (1, 1, H, W))] if kind == 1 else
                            [(head.gumbel_pixel, (1, 1, H, W)), (head.gumbel_image, (1, 1, 1, 1))]):
            gate.fixed_noise = hp.logistic_noise(torch.rand(shape, generator=g).cuda(), torch.rand(shape, generator=g).cuda(),
                                                 gate.eps)
    seed = 62
    mask, dout, _ = oracle_head_maskout(head, depth, conf, *oracle_head_noise(head, B, H, W, seed), threshold)
    lidar = make_lidar(H, W)
    pts = hp.project_2d_to_3d_dense(dout, lidar.angle, 0.9, 120.0, 0.0)
    planar = hp.inv_to_xyz(hp.tanh_to_sigmoid_clamped(dout), lidar.angle, 0.9, 120.0, 0.0)
    valid = hp.tanh_to_sigmoid_clamped(dout).flatten(1) != 0
    pixel_gate = head.gumbel if kind == 1 else head.gumbel_pixel
    if math.isnan(threshold) and pixel_gate.hard:
        assert bool((mask[:, 0] == 0).all())      # soft > nan is false: every hard pixel mask is 0
    for path in ("maskout", "points", "planar", "segment", "image"):
        inputs = {"depth": depth.clone(), "confidence": conf.clone()}
        torch.manual_seed(seed)                   # fresh noise: the draws the oracle replayed
        if path == "maskout":
            out = head.maskout(inputs, threshold=threshold)
        elif path == "points":
            out = pipeline.maskout_and_project(head, inputs, lidar, tol=0.0, threshold=threshold)
            assert_bit_equal(out["points"], pts, f"{path}: points")
        elif path == "planar":
            out, points, _, _, _ = _head_call(head, inputs, threshold, lidar=lidar, tol=0.0, points_layout=0)
            assert_bit_equal(points, planar, f"{path}: points")
        else:
            monkeypatch.setenv("DUSTY_HEAD_COMPACT", path)
            out = pipeline.maskout_and_project(head, inputs, lidar, tol=0.0, threshold=threshold, compact=True)
            assert_bit_equal(out["points"], pts, f"{path}: points")
            assert torch.equal(out["valid_count"].long(), valid.sum(1)), path
            for b in range(B):
                k = int(valid[b].sum())
                assert torch.equal(out["valid_index"][b, :k].long(), torch.nonzero(valid[b]).flatten()), path
                assert_bit_equal(out["valid_points"][b, :k], pts[b][valid[b]], f"{path}: compacted points")
        assert_bit_equal(out["mask"], mask, f"{path}: mask")
        assert_bit_equal(out["depth"], dout, f"{path}: depth")


def test_fresh_noise_uses_the_reference_rng_draws():
    from dusty_gan_b200.models.dusty import DUSty2
    depth, conf, _, _ = head_inputs(4, 2, 16, 64, 5, "cuda")
    head = DUSty2(torch.nn.Identity(), tau=1.0).cuda().train()
    torch.manual_seed(123)
    out = head.maskout({"depth": depth.clone(), "confidence": conf.clone()})
    torch.manual_seed(123)
    u1p = torch.rand(4, 1, 16, 64, device="cuda"); u2p = torch.rand_like(u1p)
    u1i = torch.rand(4, 1, 1, 1, device="cuda"); u2i = torch.rand_like(u1i)
    mask, dout = hp.maskout_dusty2(depth, conf, hp.logistic_noise(u1p, u2p), noise_image=hp.logistic_noise(u1i, u2i))
    assert_bit_equal(out["mask"], mask, "mask")
    assert_bit_equal(out["depth"], dout, "depth")


def test_gumbel_sigmoid_module_thresholds_and_grad():
    from dusty_gan_b200.models.dusty import GumbelSigmoid
    g = GumbelSigmoid(tau=0.7).cuda()
    logits = torch.randn(3, 1, 16, 64, device="cuda", requires_grad=True)
    noise = g.logistic_noise(logits)[[0]]
    g.fixed_noise = noise
    for thr in (0.5, 0.3, 0.9, float("nan")):        # NaN: soft > nan is false, so the hard gate gives exact zeros
        out = g(logits, thr)
        assert_bit_equal(out.detach(), hp.gumbel_sigmoid(logits.detach(), noise, 0.7, thr), f"thr={thr}")
    assert bool((out == 0).all())
    out = g(logits)
    out.sum().backward()
    ref_logits = logits.detach().clone().requires_grad_(True)
    hp.gumbel_sigmoid(ref_logits, noise, 0.7).sum().backward()
    assert torch.allclose(logits.grad, ref_logits.grad, rtol=1e-5, atol=1e-7)


def test_inv_to_xyz_bit_exact_and_tolerances(golden):
    g = golden("lidar_projection.npz")
    lidar = make_lidar(16, 64)
    assert np.array_equal(lidar.angle.cpu().numpy(), g["angle"])
    inv = torch.from_numpy(g["inv"]).cuda()
    for tol, key in ((1e-8, "xyz_tol1e8"), (0, "xyz_tol0"), (0.008, "xyz_tol8e3")):
        xyz = lidar.inv_to_xyz(inv, tol)
        assert_bit_equal(xyz, hp.inv_to_xyz(inv.clone(), lidar.angle, 0.9, 120.0, tol), f"tol={tol}")
        # the reference on CPU divides where CUDA multiplies by a reciprocal (trap T2): a few ulp
        assert np.allclose(xyz.cpu().numpy(), g[key], rtol=1e-6, atol=1e-9)
        assert np.array_equal(xyz.cpu().numpy() == 0, g[key] == 0)


@pytest.mark.parametrize("min_depth,max_depth,tau", [(1.72, 67.2, 1.19), (2.95, 144.9, 0.7), (0.53, 129.9, 1.0)])
def test_other_depth_limits_and_temperatures_bit_exact(min_depth, max_depth, tau):
    """Limits/temperatures for which f32(1/double(s)) != 1.0f/f32(s): ATen's CUDA kernels divide by a
    Python scalar by multiplying with the former (torch 2.11 div_true_kernel_cuda)."""
    from dusty_gan_b200.models.dusty import DUSty1
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    from dusty_gan_b200 import pipeline
    B, H, W = 3, 16, 64
    depth, conf, u1, u2 = head_inputs(B, 1, H, W, 77, "cuda")
    head = DUSty1(torch.nn.Identity(), tau=tau).cuda().eval()
    head.gumbel.fixed_noise = head.gumbel._logistic_from_uniform(u1, u2)
    lidar = LiDAR(H, W, min_depth, max_depth, angle=synthetic_hdl64e_angles()).cuda()
    mask, dout = hp.maskout_dusty1(depth, conf, hp.logistic_noise(u1, u2), tau=tau)
    fused = pipeline.maskout_and_project(head, {"depth": depth.clone(), "confidence": conf.clone()}, lidar, tol=0.0)
    assert_bit_equal(fused["mask"], mask, "mask")
    assert_bit_equal(fused["depth"], dout, "depth")
    assert_bit_equal(fused["points"], hp.project_2d_to_3d_dense(dout, lidar.angle, min_depth, max_depth, 0.0), "points")
    inv = torch.rand(B, 1, H, W, device="cuda")
    assert_bit_equal(lidar.inv_to_xyz(inv, 0.0), hp.inv_to_xyz(inv.clone(), lidar.angle, min_depth, max_depth, 0.0), "xyz")


@pytest.mark.parametrize("name,kind", [("head_dusty1_eval.npz", 1), ("head_dusty2_eval.npz", 2)])
def test_against_reference_module_golden(golden, name, kind):
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2
    g = golden(name)
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=1.0).cuda().eval()
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    gate.fixed_noise = torch.from_numpy(g["fixed_noise_pixel"]).cuda()
    out = head.maskout({"depth": torch.from_numpy(g["depth"]).cuda(), "confidence": torch.from_numpy(g["confidence"]).cuda()})
    mask = out["mask"].cpu().numpy()
    # CPU and CUDA exp differ in the last ulp, which can flip a mask only where sigmoid == 0.5 +- 1ulp
    x = g["confidence"][:, :1] + g["fixed_noise_pixel"]
    decided = np.abs(x) > 1e-6
    assert np.array_equal(mask[:, :1][decided], g["fixed_mask"][:, :1][decided])
    if kind == 2:
        assert np.array_equal(mask[:, 1], g["fixed_mask"][:, 1])
    same_mask = np.all(mask == g["fixed_mask"], axis=1, keepdims=True)
    assert np.array_equal(out["depth"].cpu().numpy()[same_mask], g["fixed_depth"][same_mask])


def test_rejects_cpu_and_grad_inputs():
    from dusty_gan_b200.models.dusty import DUSty1
    head = DUSty1(torch.nn.Identity(), tau=1.0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        head.maskout({"depth": torch.zeros(1, 1, 8, 8), "confidence": torch.zeros(1, 1, 8, 8)})


@pytest.mark.parametrize("kind", [1, 2])
def test_setup_fixed_noise_hook_freezes_the_noise_on_the_fused_heads(kind):
    """utils.setup(fix_noise=True) registers a forward pre-hook on every GumbelSigmoid that freezes
    ``fixed_noise`` on the first call (reference utils/__init__.py:141-149). The fused heads never call the
    gate modules, so they must run those hooks themselves: one noise map for every batch, masks bit-equal to
    the op chain fed that map."""
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2, GumbelSigmoid
    from dusty_gan_b200 import pipeline
    B, H, W = 4, 64, 512
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=1.0).cuda().eval()

    def set_gumbel_noise(m, i):                    # verbatim from the reference's setup()
        if m.fixed_noise is None:
            m.fixed_noise = m.logistic_noise(i[0])[[0]]

    for m in head.modules():
        if isinstance(m, GumbelSigmoid):
            m.register_forward_pre_hook(set_gumbel_noise)
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    assert gate.fixed_noise is None
    lidar = make_lidar(H, W)
    torch.manual_seed(123)
    outs = []
    for seed in (1, 2, 3):
        depth, conf, _, _ = head_inputs(B, kind, H, W, seed, "cuda")
        if seed == 2:
            out = pipeline.maskout_and_project(head, {"depth": depth, "confidence": conf}, lidar, tol=0.0)
        else:
            out = head.maskout({"depth": depth, "confidence": conf})
        noise = gate.fixed_noise
        assert noise is not None and noise.shape == (1, 1, H, W)
        outs.append(noise.clone())
        if kind == 1:
            mask, dout = hp.maskout_dusty1(depth, conf, noise)
        else:
            mask, dout = hp.maskout_dusty2(depth, conf, noise)
        assert_bit_equal(out["mask"], mask, "mask under the frozen noise")
        assert_bit_equal(out["depth"], dout, "depth under the frozen noise")
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])      # drawn once, reused forever
    if kind == 2:
        assert head.gumbel_image.fixed_noise is None       # eval mode never calls the image gate (models/dusty.py:120)


def test_inv_to_xyz_and_downsample_are_differentiable_like_the_reference():
    """demo.py back-propagates a Chamfer loss through lidar.inv_to_xyz and downsample_point_clouds
    (GatherOperation): the gradients must flow, and match autograd through the reference's op chain."""
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    H, W = 16, 64
    lidar = make_lidar(H, W)
    g = torch.Generator().manual_seed(9)
    inv = torch.rand(2, 1, H, W, generator=g).cuda()
    inv[:, :, ::3, ::5] = 0.0                                   # dropped pixels
    x = inv.clone().requires_grad_(True)
    xyz = lidar.inv_to_xyz(x, tol=0.0)
    w = torch.randn(xyz.shape, generator=g).cuda()
    (xyz * w).sum().backward()
    y = inv.clone().requires_grad_(True)
    ref = hp.inv_to_xyz(y, lidar.angle, 0.9, 120.0, 0.0)
    (ref * w).sum().backward()
    assert torch.allclose(x.grad, y.grad, rtol=1e-4, atol=1e-6)
    assert bool((x.grad[:, :, ::3, ::5] == 0).all())
    pts = xyz.detach().flatten(2).transpose(1, 2).contiguous().requires_grad_(True)
    sub = downsample_point_clouds(pts, 32)
    assert sub.requires_grad
    sub.sum().backward()
    assert pts.grad.sum().item() == pytest.approx(2 * 32 * 3)
    with torch.no_grad():
        assert torch.equal(downsample_point_clouds(pts, 32), sub)


def test_learnable_temperature_and_soft_output_match_the_reference_op_chain():
    """GumbelSigmoid(tau=None) multiplies by softplus(weight) + 1/tau_max (reference models/dusty.py:39-41) and
    GumbelSigmoid(hard=False) returns the soft mask (:58-59); forward bit-equal to the op chain on this device,
    gradients (logits and the temperature weight) equal to autograd through it."""
    from dusty_gan_b200.models.dusty import GumbelSigmoid
    B, H, W = 3, 16, 64
    _, conf, u1, u2 = head_inputs(B, 1, H, W, 77, "cuda")
    for hard in (True, False):
        gate = GumbelSigmoid(tau=None, tau_max=2.0, hard=hard).cuda()
        with torch.no_grad():
            gate.weight.fill_(0.37)
        gate.fixed_noise = gate._logistic_from_uniform(u1, u2)
        x = conf.clone().requires_grad_(True)
        out = gate(x, threshold=0.4)
        w = torch.randn_like(out)
        (out * w).sum().backward()
        # the reference's op chain
        y = conf.clone().requires_grad_(True)
        wt = gate.weight.detach().clone().requires_grad_(True)
        it = torch.nn.functional.softplus(wt) + 1.0 / 2.0
        soft = torch.sigmoid((y + gate.fixed_noise.expand(B, -1, -1, -1)) * it)
        ref = ((soft > 0.4).float() - soft.detach() + soft) if hard else soft
        (ref * w).sum().backward()
        assert_bit_equal(out.detach(), ref.detach(), f"learnable-tau forward, hard={hard}")
        assert torch.allclose(x.grad, y.grad, rtol=1e-5, atol=1e-7)
        assert torch.allclose(gate.weight.grad, wt.grad, rtol=1e-4, atol=1e-6)
    soft_gate = GumbelSigmoid(tau=0.7, hard=False).cuda()
    soft_gate.fixed_noise = gate.fixed_noise
    got = soft_gate(conf)
    want = torch.sigmoid((conf + gate.fixed_noise.expand(B, -1, -1, -1)) / 0.7)
    assert_bit_equal(got, want, "soft mask, fixed temperature")
