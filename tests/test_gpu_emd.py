"""Approximate EMD on the B200: the op, the matrix and the MMD/COV/1-NNA-EMD scores against the reference's kernels
restated in oracle/emd_reference.cu (bit for bit where the reference's order of operations is kept) and against
the float64 oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from helpers import lidar_like_clouds, rel_err, sampled_clouds
from oracle import emd as oemd
from oracle import emd_ref

pytestmark = pytest.mark.gpu

CASES = [(4, 2048, 2048), (3, 1024, 2048), (5, 2048, 1024), (2, 1, 7), (2, 33, 33), (8, 300, 300), (1, 5000, 5000)]


def _clouds(kind, b, n, m, seed):
    make = sampled_clouds if kind == "sampled" else lidar_like_clouds
    return (torch.from_numpy(make(b, n, seed)).cuda(), torch.from_numpy(make(b, m, seed + 1)).cuda())


@pytest.mark.parametrize("kind", ["sampled", "lidar"])
@pytest.mark.parametrize("b,n,m", CASES)
def test_forward_is_bit_equal_to_the_reference_kernels(kind, b, n, m):
    from dusty_gan_b200.utils.metrics.distance import earth_mover_distance
    x1, x2 = _clouds(kind, b, n, m, 7 * n + m)
    cost = earth_mover_distance(x1, x2, transpose=False)
    ref = emd_ref.earth_mover_distance(x1, x2)
    assert torch.equal(cost, ref), (cost, ref)
    f64 = oemd.cost(x1[0].cpu().numpy(), x2[0].cpu().numpy())
    assert rel_err(cost[0].item(), f64) < 1e-4, (cost[0].item(), f64)
    assert torch.equal(earth_mover_distance(x1, x2, transpose=False), cost)        # two runs: bit-equal


@pytest.mark.parametrize("kind,b,n,m", [("sampled", 3, 512, 384), ("lidar", 2, 300, 300), ("sampled", 1, 2500, 1200)])
def test_gradients_match_the_reference_kernels(kind, b, n, m):
    from dusty_gan_b200.utils.metrics.distance import earth_mover_distance
    x1, x2 = _clouds(kind, b, n, m, 11)
    x1.requires_grad_(True)
    x2.requires_grad_(True)
    g = torch.rand(b, device="cuda") + 0.5
    (earth_mover_distance(x1, x2, transpose=False) * g).sum().backward()
    with torch.no_grad():
        match = emd_ref.approxmatch(x1, x2)
        r1, r2 = emd_ref.matchcost_grad(x1, x2, match, g)
    for got, want in ((x1.grad, r1), (x2.grad, r2)):
        scale = want.abs().amax(dim=(1, 2), keepdim=True)
        assert ((got - want).abs() <= 1e-5 * scale).all(), ((got - want).abs().max(), scale.min())


def test_layouts_and_refusals():
    from dusty_gan_b200.utils.metrics.distance import earth_mover_distance
    x1, x2 = _clouds("sampled", 3, 200, 150, 3)
    want = earth_mover_distance(x1, x2, transpose=False)
    assert torch.equal(earth_mover_distance(x1.transpose(1, 2), x2.transpose(1, 2)), want)             # (B,3,N)
    assert torch.equal(earth_mover_distance(x1.transpose(1, 2).contiguous(), x2.transpose(1, 2).contiguous()), want)
    assert torch.equal(earth_mover_distance(x1[1], x2[1], transpose=False), want[1:2])                  # 2-D
    wide = torch.cat([x1, x1], dim=2)[:, :, 1:4]                                                         # non-contiguous
    assert not wide.is_contiguous()
    assert torch.equal(earth_mover_distance(wide, x2, transpose=False),
                       earth_mover_distance(wide.contiguous(), x2, transpose=False))
    with pytest.raises(RuntimeError, match="no CPU path"):
        earth_mover_distance(x1.cpu(), x2.cpu(), transpose=False)
    with pytest.raises(ValueError, match="at least one point"):
        earth_mover_distance(x1[:, :0], x2, transpose=False)


@pytest.mark.parametrize("kind", ["sampled", "lidar"])
def test_matrix_entries_equal_compute_emd_bit_for_bit(kind):
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_emd, emd_matrix
    A, _ = _clouds(kind, 5, 300, 300, 21)
    B, _ = _clouds(kind, 6, 257, 257, 22)
    M = emd_matrix(A, B)
    want = torch.stack([torch.cat([compute_emd(A[i:i + 1], B[j:j + 1]) for j in range(6)]) for i in range(5)])
    assert torch.equal(M, want)
    assert torch.equal(M, emd_ref.emd_matrix(A, B))
    assert (rel_err(M.cpu().numpy(), oemd.emd_matrix(A.cpu().numpy(), B.cpu().numpy())) < 1e-4).all()
    shard = torch.full_like(M, -1.0)
    emd_matrix(A, B, rows=(1, 5, 2), out=shard)
    assert torch.equal(shard[1::2], M[1::2]) and (shard[0::2] == -1).all()


def _reference_scores(M_rr, M_rg, M_gg):
    """The reference's _compute_cov_mmd and _compute_nna(k=1) (cov_mmd_1nna.py:54-106) on full matrices."""
    N_ref, N_gen = M_rg.shape
    mmd_gen, min_idx_gen = M_rg.min(dim=0)
    mmd_ref, _ = M_rg.min(dim=1)
    out = {"mmd": mmd_ref.mean().item(), "mmd-sample": mmd_gen.mean().item(),
           "cov": float(len(torch.unique(min_idx_gen))) / float(N_ref)}
    label = torch.cat((torch.ones(N_ref), torch.zeros(N_gen))).to(M_rr)
    M = torch.cat((torch.cat((M_rr, M_rg), 1), torch.cat((M_rg.t(), M_gg), 1)), 0)
    M = M + torch.diag(torch.full((N_ref + N_gen,), float("inf"), device=M.device))
    _, idx = M.topk(1, 0, False)
    pred = (label.index_select(0, idx[0]) >= 0.5).float()
    s = {"tp": (pred * label).sum().item(), "fp": (pred * (1 - label)).sum().item(),
         "fn": ((1 - pred) * label).sum().item(), "tn": ((1 - pred) * (1 - label)).sum().item()}
    s["accuracy"] = torch.eq(label, pred).float().mean().item()
    out.update({f"1-nn-{k}": v for k, v in s.items()})
    return out


@pytest.mark.parametrize("nr,ng,pr,pg", [(12, 12, 512, 512), (9, 14, 300, 300), (8, 7, 256, 384)])
def test_scores_equal_the_reference_formulation(nr, ng, pr, pg):
    from dusty_gan_b200.utils.metrics import cov_mmd_1nna as C
    ref = torch.from_numpy(sampled_clouds(nr, pr, nr + pr)).cuda()
    gen = torch.from_numpy(lidar_like_clouds(ng, pg, ng + pg)).cuda()
    both = C.compute_cov_mmd_1nna(gen, ref, 512, ("cd", "emd"), verbose=False)
    cd = C.compute_cov_mmd_1nna(gen, ref, 512, ("cd",), verbose=False)
    assert {k: v for k, v in both.items() if k.endswith("-cd")} == cd
    emd = {k[:-4]: v for k, v in both.items() if k.endswith("-emd")}
    want = _reference_scores(emd_ref.emd_matrix(ref, ref), emd_ref.emd_matrix(ref, gen), emd_ref.emd_matrix(gen, gen))
    for k, v in want.items():
        if k in ("mmd", "mmd-sample"):
            assert emd[k] == pytest.approx(v, rel=1e-6), k
        else:
            assert emd[k] == v, (k, emd[k], v)
    C.FUSED_EPILOGUE = False
    try:
        unfused = C.compute_cov_mmd_1nna(gen, ref, 512, ("cd", "emd"), verbose=False)
    finally:
        C.FUSED_EPILOGUE = True
    assert unfused == both


def test_fused_path_memory_grows_linearly():
    from dusty_gan_b200.utils.metrics import cov_mmd_1nna as C
    peaks = []
    for n in (40, 160):
        ref = torch.from_numpy(sampled_clouds(n, 8, 1)).cuda()
        gen = torch.from_numpy(sampled_clouds(n, 8, 2)).cuda()
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        C.emd_scores(gen, ref)
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
    # 4x the clouds: the keys grow by 24 B per stacked cloud; one (320 x 320) f32 matrix alone would be 400 KB
    assert peaks[1] - peaks[0] < 64 * 1024, peaks


WORKER = r'''
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["DUSTY_ROOT"]); sys.path.insert(0, os.path.join(os.environ["DUSTY_ROOT"], "tests"))
from helpers import sampled_clouds, lidar_like_clouds
torch.cuda.set_device(0)
from dusty_gan_b200.utils.metrics import cov_mmd_1nna as M
cases = [(sampled_clouds(11, 128, 1), sampled_clouds(9, 128, 2)),
         (lidar_like_clouds(8, 160, 3), sampled_clouds(7, 100, 4))]          # unequal point counts
cases = [(torch.from_numpy(g).cuda(), torch.from_numpy(r).cuda()) for g, r in cases]
single = [M.compute_cov_mmd_1nna(g, r, 512, ("emd",), verbose=False) for g, r in cases]
dist.init_process_group("gloo")
ok = True
for (g, r), s1 in zip(cases, single):
    ok = ok and M.compute_cov_mmd_1nna(g, r, 512, ("emd",), verbose=False) == s1 and len(s1) == 12
flags = [None] * dist.get_world_size(); dist.all_gather_object(flags, bool(ok))
if int(os.environ["RANK"]) == 0: print("RESULT", json.dumps({"ok": all(flags), "world": dist.get_world_size()}))
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_emd_scores_equal_unsharded_ranks_sharing_one_gpu(tmp_path, world):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, DUSTY_ROOT=ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", str(29570 + world), str(script)],
                         env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("RESULT")][-1]
    assert '"ok": true' in line and f'"world": {world}' in line, line
