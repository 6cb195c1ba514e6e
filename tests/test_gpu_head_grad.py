"""Backward of the fused head (dusty_head_project_backward) against autograd through the reference's op chain
(oracle.head_projection) on the same GPU: DUSty-I / DUSty-II, fixed and fresh noise, soft gates, each gate's own
learnable temperature, the fused projection in both point layouts, exact zeros, the inversion loss end to end, a
DUSty-II generator step on its two temperatures, determinism and the refused cases."""
import pytest
import torch

from helpers import head_inputs, oracle_head_maskout, oracle_head_noise, sampled_clouds
from oracle import head_projection as hp

pytestmark = pytest.mark.gpu

MIN_DEPTH, MAX_DEPTH = 0.9, 120.0
SHAPES = [(5, 64, 512), (3, 16, 64), (2, 8, 20), (130, 64, 512)]
# (channels, training, noise, variant): variant "soft" makes the pixel gate (DUSty-I's only gate) GumbelSigmoid(hard=False)
# and "soft_image" DUSty-II's image gate; "learnable" is tau=None with the pixel gate's weight at 0.37, "diverged" is
# tau=None with the pixel gate's weight at 0.37 and the image gate's at -1.2 (what training makes of them), run at
# threshold 0.3, where the temperatures also decide mask values
CASES = [(1, False, "fixed", None), (1, False, "fresh", None), (2, False, "fixed", None), (2, False, "fresh", None),
         (2, True, "fixed", None), (2, True, "fresh", None), (1, False, "fixed", "soft"),
         (1, False, "fixed", "learnable"), (1, True, "fresh", "learnable"), (2, False, "fixed", "learnable"),
         (2, True, "fixed", "diverged"), (2, True, "fresh", "diverged"), (2, True, "fixed", "soft"),
         (2, True, "fresh", "soft_image")]
PROJ_CASES = [CASES[0], CASES[3], CASES[5], CASES[6], CASES[7], CASES[10], CASES[11], CASES[13]]


def make_lidar(H, W):
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    return LiDAR(H, W, MIN_DEPTH, MAX_DEPTH, angle=synthetic_hdl64e_angles()).cuda()


def bits(t):
    return t.contiguous().view(torch.int32)


def assert_bit_equal(a, b, what):
    assert a.shape == b.shape, what
    same = (bits(a) == bits(b)) | (torch.isnan(a) & torch.isnan(b))
    assert bool(same.all()), f"{what}: {(~same).sum().item()} of {same.numel()} differ"


def assert_close(a, b, rtol, atol, what):
    ok = torch.isclose(a, b, rtol=rtol, atol=atol)
    if not bool(ok.all()):
        i = int((~ok).flatten().nonzero()[0])
        raise AssertionError(f"{what}: {(~ok).sum().item()} of {ok.numel()} differ, e.g. {a.flatten()[i].item()!r} "
                             f"vs {b.flatten()[i].item()!r}")


def make_head(kind, training, noise, variant, H, W, seed):
    """The head under test and, for fixed noise, its noise maps."""
    from dusty_gan_b200.models.dusty import DUSty1, DUSty2
    learnable = variant in ("learnable", "diverged")
    head = (DUSty1 if kind == 1 else DUSty2)(torch.nn.Identity(), tau=None if learnable else 1.0).cuda()
    head.train(training)
    gate = head.gumbel if kind == 1 else head.gumbel_pixel
    with torch.no_grad():
        if learnable:
            gate.weight.fill_(0.37)
        if variant == "diverged":
            head.gumbel_image.weight.fill_(-1.2)
    if variant == "soft":
        gate.hard = False
    if variant == "soft_image":
        head.gumbel_image.hard = False
    if noise == "fixed":
        g = torch.Generator().manual_seed(seed)
        u = [torch.rand(1, 1, H, W, generator=g).cuda() for _ in range(2)]
        gate.fixed_noise = hp.logistic_noise(*u)
        if kind == 2:
            v = [torch.rand(1, 1, 1, 1, generator=g).cuda() for _ in range(2)]
            head.gumbel_image.fixed_noise = hp.logistic_noise(*v)
    return head, gate


def run_both(kind, training, noise, variant, shape, seed, lib_fn, oracle_fn, loss_fn):
    """Run the library arm (``lib_fn(head, depth, conf) -> outputs``) and the oracle arm (``oracle_fn(mask, dout)``
    on the oracle's maskout), back-propagate ``loss_fn(outputs)`` through both and return the pairs of results: the
    outputs, then (depth, confidence, (pixel weight grad, image weight grad)) of each arm, a weight grad being None
    where the oracle has no learnable temperature for that gate."""
    B, H, W = shape
    depth, conf, _, _ = head_inputs(B, kind, H, W, seed, "cuda")
    head, gate = make_head(kind, training, noise, variant, H, W, seed + 1)
    threshold = 0.3 if variant == "diverged" else 0.5
    d = depth.clone().requires_grad_(True)
    c = conf.clone().requires_grad_(True)
    torch.manual_seed(seed + 2)
    out = lib_fn(head, d, c, threshold)
    loss_fn(out).backward()
    noise_pixel, noise_image = oracle_head_noise(head, B, H, W, None if noise == "fixed" else seed + 2)
    dr = depth.clone().requires_grad_(True)
    cr = conf.clone().requires_grad_(True)
    mask, dout, leaves = oracle_head_maskout(head, dr, cr, noise_pixel, noise_image, threshold)
    ref = oracle_fn(mask, dout)
    loss_fn(ref).backward()
    gates = (gate, head.gumbel_image if kind == 2 else None)
    lib_w = tuple(None if w is None else g.weight.grad for g, w in zip(gates, leaves))
    return out, ref, (d, c, lib_w), (dr, cr, tuple(None if w is None else w.grad for w in leaves))


def assert_weight_grads(gw, gwr):
    """Each learnable temperature's weight.grad, pixel gate and image gate separately."""
    for what, a, b in zip(("pixel", "image"), gw, gwr):
        if b is not None:
            assert a is not None, what
            assert_close(a, b, 1e-4, 1e-6, f"{what} gate temperature weight.grad")


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind,training,noise,variant", CASES)
def test_maskout_gradients_match_autograd_through_the_reference(kind, training, noise, variant, shape):
    """Loss = sum w1 * depth_out + sum w2 * mask. d depth is one product (grad_depth * mask): bit-equal."""
    B, H, W = shape
    w1, w2 = [torch.randn(s, generator=torch.Generator().manual_seed(7 + i)).cuda()
              for i, s in enumerate([(B, 1, H, W), (B, kind, H, W)])]

    def lib(head, d, c, threshold):
        out = head.maskout({"depth": d, "confidence": c}, threshold=threshold)
        return out["depth"], out["mask"]

    out, ref, (d, c, gw), (dr, cr, gwr) = run_both(
        kind, training, noise, variant, shape, 11 * kind + B, lib, lambda mask, dout: (dout, mask),
        lambda o: (w1 * o[0]).sum() + (w2 * o[1]).sum())
    assert_bit_equal(out[0].detach(), ref[0].detach(), "depth_out")
    assert_bit_equal(out[1].detach(), ref[1].detach(), "mask")
    assert_bit_equal(d.grad, dr.grad, "depth.grad")
    assert_close(c.grad, cr.grad, 1e-5, 1e-7, "confidence.grad")
    if kind == 2 and not training:
        assert bool((c.grad[:, 1] == 0).all())                  # the eval-mode image gate is (logit > 0)
    if variant in ("learnable", "diverged"):
        assert gw[0] is not None and gwr[0] is not None
    if variant == "diverged":
        assert gw[1] is not None and gwr[1] is not None
    assert_weight_grads(gw, gwr)


@pytest.mark.parametrize("shape", SHAPES[:3])
@pytest.mark.parametrize("kind,training,noise,variant", PROJ_CASES)
@pytest.mark.parametrize("with_depth", [False, True])
def test_fused_projection_gradients_match_autograd_through_the_reference(kind, training, noise, variant, shape,
                                                                         with_depth):
    """maskout_and_project(..., differentiable=True) -> (B,N,3) points; loss on the points, or points + depth."""
    from dusty_gan_b200 import pipeline
    B, H, W = shape
    lidar = make_lidar(H, W)
    w1, w3 = [torch.randn(s, generator=torch.Generator().manual_seed(5 + i)).cuda()
              for i, s in enumerate([(B, 1, H, W), (B, H * W, 3)])]

    def lib(head, d, c, threshold):
        out = pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar, threshold=threshold,
                                           differentiable=True)
        return out["depth"], out["points"]

    def oracle(mask, dout):
        return dout, hp.project_2d_to_3d_dense(dout, lidar.angle, MIN_DEPTH, MAX_DEPTH, 0.0)

    def loss(o):
        return (w3 * o[1]).sum() + ((w1 * o[0]).sum() if with_depth else 0.0)

    out, ref, (d, c, gw), (dr, cr, gwr) = run_both(kind, training, noise, variant, shape, 3 * kind + B, lib, oracle, loss)
    assert_bit_equal(out[1].detach(), ref[1].detach(), "points")
    assert_close(d.grad, dr.grad, 1e-4, 1e-6, "depth.grad")
    assert_close(c.grad, cr.grad, 1e-4, 1e-6, "confidence.grad")
    assert_weight_grads(gw, gwr)


@pytest.mark.parametrize("kind", [1, 2])
def test_planar_points_layout_through_the_abi(kind):
    """points_layout 0, (B,3,H,W) like inv_to_xyz, is the other layout the forward writes; its backward reads the
    gradient in that layout."""
    from dusty_gan_b200.models.dusty import _head_call
    B, H, W = 3, 16, 64
    lidar = make_lidar(H, W)
    w3 = torch.randn((B, 3, H, W), generator=torch.Generator().manual_seed(3)).cuda()

    def lib(head, d, c, threshold):
        return _head_call(head, {"depth": d, "confidence": c}, threshold, lidar=lidar, tol=0.0, points_layout=0)[1]

    def oracle(mask, dout):
        return hp.inv_to_xyz(hp.tanh_to_sigmoid_clamped(dout), lidar.angle, MIN_DEPTH, MAX_DEPTH, 0.0)

    out, ref, (d, c, _), (dr, cr, _) = run_both(kind, kind == 2, "fixed", None, (B, H, W), 21, lib, oracle,
                                                lambda o: (w3 * o).sum())
    assert_bit_equal(out.detach(), ref.detach(), "planar points")
    assert_close(d.grad, dr.grad, 1e-4, 1e-6, "depth.grad")
    assert_close(c.grad, cr.grad, 1e-4, 1e-6, "confidence.grad")


def test_gradients_are_exactly_zero_where_the_references_are():
    """A loss on the points only: nothing flows back from dropped pixels (m = 0), from pixels at or under tol, nor
    from pixels the clamp cuts (depth outside [-1, 1])."""
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.models.dusty import DUSty1
    B, H, W = 4, 16, 64
    tol = 0.05
    depth, conf, u1, u2 = head_inputs(B, 1, H, W, 31, "cuda")
    depth[:, :, ::4, ::8] = -1.5                                  # (x + 1) / 2 < 0: cut by the clamp
    depth[:, :, 1::4, ::8] = 1.5                                  # > 1: cut too (clamp_backward keeps only [0, 1])
    depth[:, :, 2::4, ::8] = -0.95                                # inv = 0.025 <= tol
    conf[:, :, :3, ::8] = 30.0                                    # kept, whatever the noise
    conf[:, :, 3, :] = -30.0                                      # dropped
    head = DUSty1(torch.nn.Identity(), tau=1.0).cuda().eval()
    head.gumbel.fixed_noise = hp.logistic_noise(u1, u2)
    lidar = make_lidar(H, W)
    w3 = torch.randn((B, H * W, 3), generator=torch.Generator().manual_seed(4)).cuda()
    d, c = depth.clone().requires_grad_(True), conf.clone().requires_grad_(True)
    out = pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar, tol=tol, differentiable=True)
    (w3 * out["points"]).sum().backward()
    dr, cr = depth.clone().requires_grad_(True), conf.clone().requires_grad_(True)
    mask, dout = hp.maskout_dusty1(dr, cr, head.gumbel.fixed_noise)
    (w3 * hp.project_2d_to_3d_dense(dout, lidar.angle, MIN_DEPTH, MAX_DEPTH, tol)).sum().backward()
    assert bool((out["mask"][:, :, :3, ::8] == 1).all()) and bool((out["mask"][:, :, 3] == 0).all())
    special = torch.zeros(B, 1, H, W, dtype=torch.bool, device="cuda")
    for r in range(H):
        if r % 4 < 3:
            special[:, :, r, ::8] = True                          # kept or not: cut, or at or under tol
    special[:, :, 3, :] = True                                    # dropped
    for name, g, gr in (("depth", d.grad, dr.grad), ("confidence", c.grad, cr.grad)):
        assert bool((gr[special] == 0).all()), name
        assert bool((g[special] == 0).all()), name
        assert bool((g[gr == 0] == 0).all()), name
        assert bool((g != 0).any()), name
    assert_close(d.grad, dr.grad, 1e-4, 1e-6, "depth.grad")
    assert_close(c.grad, cr.grad, 1e-4, 1e-6, "confidence.grad")


class _Backbone(torch.nn.Module):
    """A small generator: latent (B,16) -> {"depth" tanh, "confidence"} (B,1,H,W)."""

    def __init__(self, H, W):
        super().__init__()
        self.H, self.W = H, W
        self.fc = torch.nn.Linear(16, 2 * H * W)

    def forward(self, z):
        y = self.fc(z).view(-1, 2, self.H, self.W)
        return {"depth": torch.tanh(y[:, :1] * 2.0), "confidence": y[:, 1:] * 4.0}


def test_inversion_loss_end_to_end():
    """demo.py:510-515: latent -> G -> maskout -> tanh_to_sigmoid -> inv_to_xyz -> FPS gather -> Chamfer, backward to
    the latent; once with the library head, once with the oracle head, FPS and Chamfer from the library in both."""
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.models.dusty import DUSty1
    from dusty_gan_b200.utils.metrics.distance import chamfer_distance
    from dusty_gan_b200.utils.sampling.fps import downsample_point_clouds
    B, H, W, P = 2, 32, 256, 512
    torch.manual_seed(0)
    head = DUSty1(_Backbone(H, W), tau=1.0).cuda().eval()
    g = torch.Generator().manual_seed(1)
    head.gumbel.fixed_noise = hp.logistic_noise(torch.rand(1, 1, H, W, generator=g).cuda(),
                                                torch.rand(1, 1, H, W, generator=g).cuda())
    lidar = make_lidar(H, W)
    target = torch.from_numpy(sampled_clouds(B, P, 2)).cuda()
    latent0 = torch.randn(B, 16, generator=g).cuda()

    def chamfer_loss(points):
        d1, d2 = chamfer_distance(downsample_point_clouds(points, P), target)
        return d1.mean() + d2.mean()

    z = latent0.clone().requires_grad_(True)
    out = pipeline.maskout_and_project(head, head.backbone(z), lidar, differentiable=True)
    chamfer_loss(out["points"]).backward()
    zr = latent0.clone().requires_grad_(True)
    o = head.backbone(zr)
    _, dout = hp.maskout_dusty1(o["depth"], o["confidence"], head.gumbel.fixed_noise)
    points_ref = hp.project_2d_to_3d_dense(dout, lidar.angle, MIN_DEPTH, MAX_DEPTH, 0.0)
    chamfer_loss(points_ref).backward()
    assert_bit_equal(out["points"].detach(), points_ref.detach(), "points")     # hence the same FPS indices
    assert z.grad is not None and bool(torch.isfinite(z.grad).all()) and bool((z.grad != 0).any())
    # rtol 1e-4, with an absolute floor of 1e-4 of the largest entry for entries the Linear backward cancels
    assert_close(z.grad, zr.grad, 1e-4, 1e-4 * zr.grad.abs().max().item(), "latent.grad")


def test_backward_is_deterministic():
    """Each temperature's gradient is a fixed-order reduction (per-CTA partials per gate, one final pass): two
    backward passes on the same inputs give bit-identical gradients, DUSty-I and DUSty-II in training with both
    temperatures learnable."""
    from dusty_gan_b200 import pipeline
    B, H, W = 8, 64, 512
    lidar = make_lidar(H, W)
    for kind, training, variant in ((1, False, "learnable"), (2, True, "diverged")):
        head, _ = make_head(kind, training, "fixed", variant, H, W, 5)
        weights = [p for p in head.parameters()]
        assert len(weights) == kind
        depth, conf, _, _ = head_inputs(B, kind, H, W, 6, "cuda")
        w1, w3 = [torch.randn(s, generator=torch.Generator().manual_seed(8 + i)).cuda()
                  for i, s in enumerate([(B, 1, H, W), (B, H * W, 3)])]
        grads = []
        for _ in range(2):
            for w in weights:
                w.grad = None
            d, c = depth.clone().requires_grad_(True), conf.clone().requires_grad_(True)
            out = pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar, threshold=0.3,
                                               differentiable=True)
            ((w3 * out["points"]).sum() + (w1 * out["depth"]).sum()).backward()
            grads.append((d.grad, c.grad, *(w.grad.clone() for w in weights)))
        for a, b, what in zip(*grads, ("depth", "confidence", "weight", "image weight")):
            assert_bit_equal(a, b, f"DUSty-{'I' * kind}: {what}")


def test_dusty2_generator_step_trains_each_temperature():
    """A generator step of DUSty-II in training mode with tau=None: three SGD steps on the two gates' temperature
    weights, with the same seeded noise in the library arm and in the oracle arm. Both start at 0; their gradients
    differ, so they part after the first step, and the two arms move them alike."""
    from dusty_gan_b200.models.dusty import DUSty2
    B, H, W = 4, 32, 256
    depth, conf, _, _ = head_inputs(B, 2, H, W, 71, "cuda")
    w1, w2 = [torch.randn(s, generator=torch.Generator().manual_seed(72 + i)).cuda()
              for i, s in enumerate([(B, 1, H, W), (B, 2, H, W)])]

    def loss(mask, dout):
        return (w1 * dout).mean() + (w2 * mask).mean()

    head = DUSty2(torch.nn.Identity(), tau=None).cuda().train()
    weights = [head.gumbel_pixel.weight, head.gumbel_image.weight]
    ref = [w.detach().clone().requires_grad_(True) for w in weights]
    opt, opt_ref = torch.optim.SGD(weights, lr=1.0), torch.optim.SGD(ref, lr=1.0)
    for step in range(3):
        seed = 73 + step
        torch.manual_seed(seed)
        out = head.maskout({"depth": depth.clone().requires_grad_(True), "confidence": conf.clone().requires_grad_(True)})
        opt.zero_grad()
        loss(out["mask"], out["depth"]).backward()
        opt.step()
        noise_pixel, noise_image = oracle_head_noise(head, B, H, W, seed)
        it = [torch.nn.functional.softplus(w) + 1.0 / head.gumbel_pixel.tau_max for w in ref]
        mask, dout = hp.maskout_dusty2(depth.clone().requires_grad_(True), conf.clone().requires_grad_(True), noise_pixel,
                                       it[0], noise_image=noise_image, tau_image=it[1])
        opt_ref.zero_grad()
        loss(mask, dout).backward()
        opt_ref.step()
        for what, w, r in zip(("pixel", "image"), weights, ref):
            assert_close(w.detach(), r.detach(), 1e-5, 1e-7, f"step {step}: {what} gate temperature weight")
        if step == 0:
            assert weights[0].item() != weights[1].item()


@pytest.mark.parametrize("kind", [1, 2])
def test_forward_under_grad_is_the_no_grad_forward(kind):
    from dusty_gan_b200 import pipeline
    B, H, W = 3, 16, 64
    lidar = make_lidar(H, W)
    head, _ = make_head(kind, kind == 2, "fixed", None, H, W, 9)
    depth, conf, _, _ = head_inputs(B, kind, H, W, 10, "cuda")
    with torch.no_grad():
        plain = pipeline.maskout_and_project(head, {"depth": depth.clone(), "confidence": conf.clone()}, lidar)
        plain_mask = head.maskout({"depth": depth.clone(), "confidence": conf.clone()})
    d, c = depth.clone().requires_grad_(True), conf.clone().requires_grad_(True)
    graded = pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar, differentiable=True)
    graded_mask = head.maskout({"depth": d, "confidence": c})
    assert graded["points"].requires_grad and graded_mask["mask"].requires_grad
    for key in ("mask", "depth", "points"):
        assert_bit_equal(graded[key].detach(), plain[key], key)
    for key in ("mask", "depth"):
        assert_bit_equal(graded_mask[key].detach(), plain_mask[key], key)
    # the default stays under no_grad
    assert not pipeline.maskout_and_project(head, {"depth": d, "confidence": c}, lidar)["points"].requires_grad


def test_refused_cases():
    from dusty_gan_b200 import pipeline
    from dusty_gan_b200.models.dusty import DUSty1
    B, H, W = 2, 8, 20
    lidar = make_lidar(H, W)
    depth, conf, _, _ = head_inputs(B, 2, H, W, 12, "cuda")
    head1, _ = make_head(1, False, "fixed", None, H, W, 13)
    d, c = depth.clone().requires_grad_(True), conf[:, :1].clone().requires_grad_(True)
    with pytest.raises(ValueError, match="compact"):
        pipeline.maskout_and_project(head1, {"depth": d, "confidence": c}, lidar, compact=True, differentiable=True)
    cpu = DUSty1(torch.nn.Identity(), tau=1.0)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        cpu.maskout({"depth": torch.zeros(1, 1, 8, 8, requires_grad=True),
                     "confidence": torch.zeros(1, 1, 8, 8, requires_grad=True)})
