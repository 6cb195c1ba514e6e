"""Float64 numpy restatement of the reference's approximate EMD (utils/metrics/distance/emd/: approxmatch +
matchcost + matchcostgrad1/2, the PSGN approxmatch of Fan et al. 2017). Same algorithm, exact exp and sqrt,
vectorised sums: the CPU-tier oracle; oracle/emd_reference.cu is the bit-level one."""
import numpy as np

LEVELS = [-(4.0 ** j) for j in range(7, -2, -1)] + [0.0]       # j = 7, 6, ..., -1, then level 0 for j = -2


def approxmatch(xyz1, xyz2):
    """One pair: xyz1 (n,3), xyz2 (m,3) -> match (n, m) float64 (the reference stores its transpose)."""
    p1 = np.asarray(xyz1, np.float64)
    p2 = np.asarray(xyz2, np.float64)
    n, m = len(p1), len(p2)
    if n == 0 or m == 0:
        raise ValueError("clouds must hold at least one point")
    multiL, multiR = (1.0, float(n // m)) if n >= m else (float(m // n), 1.0)
    remainL = np.full(n, multiL)
    remainR = np.full(m, multiR)
    d2 = ((p1[:, None, :] - p2[None, :, :]) ** 2).sum(-1)
    match = np.zeros((n, m))
    for level in LEVELS:
        e = np.exp(level * d2)
        ratioL = remainL / (1e-9 + e @ remainR)
        sumr = (e * ratioL[:, None]).sum(0) * remainR
        ratioR = np.minimum(remainR / (sumr + 1e-9), 1.0) * remainR
        remainR = np.maximum(0.0, remainR - sumr)
        w = e * ratioL[:, None] * ratioR[None, :]
        match += w
        remainL = np.maximum(0.0, remainL - w.sum(1))
    return match


def cost(xyz1, xyz2, match=None):
    p1 = np.asarray(xyz1, np.float64)
    p2 = np.asarray(xyz2, np.float64)
    if match is None:
        match = approxmatch(p1, p2)
    return float((np.sqrt(((p1[:, None, :] - p2[None, :, :]) ** 2).sum(-1)) * match).sum())


def earth_mover_distance(xyz1, xyz2):
    """(b,n,3) x (b,m,3) -> cost (b,) float64, the reference forward with transpose=False."""
    return np.array([cost(a, c) for a, c in zip(xyz1, xyz2)])


def grads(xyz1, xyz2, grad_cost=1.0):
    """d cost / d xyz1 (n,3) and d xyz2 (m,3) of one pair with the match held constant (as the reference)."""
    p1 = np.asarray(xyz1, np.float64)
    p2 = np.asarray(xyz2, np.float64)
    match = approxmatch(p1, p2)
    diff = p1[:, None, :] - p2[None, :, :]
    d = np.maximum(np.sqrt((diff ** 2).sum(-1)), 1e-20)
    c = (match / d)[:, :, None] * diff
    return grad_cost * c.sum(1), -grad_cost * c.sum(0)


def emd_matrix(A, B):
    """M[i,j] = cost(A[i], B[j]) / pa (compute_emd)."""
    pa = np.asarray(A).shape[1]
    return np.array([[cost(a, c) / pa for c in B] for a in A])
