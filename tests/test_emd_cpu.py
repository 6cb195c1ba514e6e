"""Approximate EMD without a GPU: the float64 oracle (oracle/emd.py) against exact transport, the C ABI's argument
checks, and the register budget of the EMD matrix kernel."""
import re
import subprocess

import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

from helpers import sampled_clouds
from oracle import emd


@pytest.mark.parametrize("n,seed", [(16, 0), (16, 1), (64, 2), (64, 3), (200, 4)])
def test_oracle_is_close_to_the_exact_assignment_cost(n, seed):
    """approxmatch's plan is feasible but not optimal. On FPS-like clouds of 16 to 200 points the first run measured
    its cost at 1.12 to 1.30 times the exact assignment cost (scipy linear_sum_assignment); the bounds below leave a
    margin on either side of that range."""
    a = sampled_clouds(1, n, seed)[0].astype(np.float64)
    b = sampled_clouds(1, n, 100 + seed)[0].astype(np.float64)
    d = np.sqrt(((a[:, None] - b[None]) ** 2).sum(-1))
    r, c = linear_sum_assignment(d)
    exact = d[r, c].sum()
    ratio = emd.cost(a, b) / exact
    assert 1.0 <= ratio <= 1.4, ratio


def test_translated_cloud_costs_n_times_the_shift():
    """Points on a lattice of spacing 0.1, shifted by |t| = 0.01: the steepest levels already match every point
    with its own image, so the cost is n |t| (measured within 0.1 %)."""
    g = np.arange(5) * 0.1
    a = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    t = np.array([0.006, -0.008, 0.0])
    assert abs(emd.cost(a, a + t) / (len(a) * np.linalg.norm(t)) - 1.0) < 1e-2


@pytest.mark.parametrize("n,m", [(40, 13), (13, 40), (30, 70)])
def test_unequal_point_counts_use_integer_multipliers(n, m):
    """multiL, multiR = (1, n // m) if n >= m else (m // n, 1): each point of the smaller cloud can absorb the
    integer multiple of mass, never more, and the plan moves almost all of it."""
    a = sampled_clouds(1, n, 1)[0]
    b = sampled_clouds(1, m, 2)[0]
    match = emd.approxmatch(a, b)
    mult_l, mult_r = (1, n // m) if n >= m else (m // n, 1)
    assert match.sum(1).max() <= mult_l * (1 + 1e-9) and match.sum(0).max() <= mult_r * (1 + 1e-9)
    capacity = min(n * mult_l, m * mult_r)
    assert match.sum() > 0.95 * capacity
    assert np.isclose(emd.grads(a, b)[0].sum(0), -emd.grads(a, b)[1].sum(0)).all()


def test_workspace_queries_and_argument_errors_without_a_gpu():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    assert lib.dusty_emd_forward_workspace_bytes(4, 2048, 2048) == 4 * 12 * 4096 * 4
    assert lib.dusty_emd_forward_workspace_bytes(1, 0, 5) == 0
    assert lib.dusty_emd_matrix_workspace_bytes(10, 2048, 10, 2048) == 296 * 12 * 4096 * 4
    # empty clouds: the reference divides by the point counts
    assert lib.dusty_emd_forward(None, None, 1, 0, 5, None, None, None, 0, None) == -1
    assert b"must hold points" in lib.dusty_last_error_string()
    assert lib.dusty_emd_backward(None, None, 1, 5, 0, None, None, None, None, None, 0, None) == -1
    def matrix(pa=8, pb=8, off_a=0, off_b=3, n_ref=3, n_total=7, keys=1):
        return lib.dusty_emd_matrix(None, 3, pa, None, 4, pb, 0, 3, 1, None, 0, off_a, off_b, n_ref, n_total,
                                    keys, None, 0, None)
    assert matrix(pa=0) == -1 and matrix(pb=0) == -1
    assert matrix(off_a=4, off_b=0, n_ref=4, n_total=7) == -1         # generated-by-reference: never needed
    assert b"generated-by-reference" in lib.dusty_last_error_string()
    assert matrix(off_a=2) == -1                                       # A straddles the reference/generated boundary
    assert matrix(n_total=6) == -1                                     # does not fit the stacked set


def test_earth_mover_distance_refuses_cpu_tensors():
    from dusty_gan_b200.utils.metrics.distance import earth_mover_distance
    with pytest.raises(RuntimeError, match="no CPU path"):
        earth_mover_distance(torch.zeros(1, 3, 8), torch.zeros(1, 3, 8))


def test_emd_matrix_kernel_keeps_its_occupancy_shape():
    """Two CTAs of 512 threads per SM (each 72 KB of shared memory): at most 64 registers, no local memory, in the
    matrix, forward and backward kernels."""
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-res-usage", _lib.LIB_PATH], text=True)
    usage = re.findall(r"Function (\S+):\s+REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)
    for frag in ("emd_matrix_kernel", "emd_forward_kernel", "emd_backward_kernel"):
        rows = [u for u in usage if frag in u[0]]
        assert len(rows) == 1, (frag, rows)
        _, reg, stack, local = rows[0]
        assert int(reg) <= 64 and int(stack) == 0 and int(local) == 0, (frag, reg, stack, local)
