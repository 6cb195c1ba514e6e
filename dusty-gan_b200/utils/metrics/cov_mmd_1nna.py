"""MMD / COV / 1-NNA over Chamfer distance on libdustyb200 (mirror of reference
utils/metrics/cov_mmd_1nna.py:19-139).

The reference fills each matrix with a Python double loop (one row, 512 columns per iteration,
>= 9 kernel launches each). Here one launch computes a whole matrix -- or, when the two sets have
the same number of points per cloud, ONE launch computes the upper triangle of the stacked
(N_ref+N_gen)^2 matrix that holds M_rr, M_rg and M_gg at once. ``compute_cov_mmd_1nna`` goes one step
further: the min / arg-min / top-1 reductions of ``_compute_cov_mmd`` and ``_compute_nna`` are fused into
that launch's epilogue, so no N x N tensor exists at all (``fused_scores``). When ``torch.distributed`` is
initialised with more than one rank the rows are sharded over the ranks and combined by a single
all-gather -- of the per-cloud (min, arg-min) vectors for the scores, of row blocks for the matrices
(see ``sharding.py``).

Distances are exactly the reference CUDA kernel's for finite inputs (csrc/chamfer.cu: the |b|^2 - 2 a.b
search is only trusted outside its own rounding window; inside it the tile is re-evaluated in the
reference's rounding), so arg-mins and the scores built on them do not flip on near-ties.
"""
import numpy as np
import torch

from ... import _lib, sharding
from .distance import chamfer_distance, earth_mover_distance


# When bench.py sets this to a list, every matrix launch appends a (start, end) CUDA event pair.
KERNEL_EVENTS = None


def compute_cd(pcs_1, pcs_2):
    dl, dr = chamfer_distance(pcs_1, pcs_2)
    return dl.mean(dim=1) + dr.mean(dim=1)


def compute_emd(pcs_1, pcs_2):
    """Approximate EMD per point (PointFlow's emd_approx): the match cost divided by the point count of pcs_1."""
    return earth_mover_distance(pcs_1, pcs_2, transpose=False) / pcs_1.size(1)


def _check_clouds(pcs, name):
    _lib.require_cuda(pcs, name)
    if pcs.dim() != 3 or pcs.size(2) != 3:
        raise ValueError(f"{name}: expected (B,P,3), got {tuple(pcs.shape)}")
    return pcs.contiguous()


# compute_cov_mmd_1nna: reductions fused into the matrix kernel's epilogue (no N x N tensor). False selects
# the round-1 path (matrices + finaliser kernels); both give bit-identical scores (tests/test_gpu_metrics.py).
FUSED_EPILOGUE = True

# Clouds with more points than this go through the sorted search (flag DUSTY_MATRIX_MERGE_ORIGIN of the C ABI): all
# exactly-zero points of a cloud -- the dropped pixels of an un-sampled range image (reference
# evaluate_reconstruction.py:124-131, SURVEY.md S7) -- are scanned as ONE point of that multiplicity, the other points
# are put in k-d order with a bounding box per 32 of them, and the kernel visits candidate chunks nearest first and
# skips every chunk that an exact box bound rules out. Results are unchanged (the bound is evaluated in the kernel's
# own rounding); on LiDAR clouds the search visits 1.7 % (un-sampled, of the kept pairs) to 8.2 % (2048 FPS samples)
# of the pairs: 5.4x the brute-force kernel on the 1000 vs 1000 x 2048 evaluation. The choice depends on the shape only, so a given input always takes the
# same path (and every row shard of a matrix the same one). Smaller clouds keep the brute-force kernel: its register
# tile, not pruning, is what pays there. Set it to a huge value to force the brute-force kernel (bench.py does, for
# the roofline of that kernel).
MERGE_ORIGIN_ABOVE = 256


def chamfer_matrix(pcs_1, pcs_2=None, rows=None, compact_rows=False, out=None, merge_origin=None, fused=None):
    """M[i,j] = compute_cd(pcs_1[i], pcs_2[j]) in one launch. ``pcs_2=None`` declares the symmetric
    case (upper triangle computed, mirrored unless ``compact_rows``). ``rows=(begin,end,stride)``
    restricts the computation to a row shard. ``merge_origin`` (default: by point count, see
    ``MERGE_ORIGIN_ABOVE``) collapses each cloud's exactly-zero points into one weighted point.
    ``fused=(keys, stacked_offset_1, stacked_offset_2, n_ref, n_total)`` also reduces every entry into the
    packed minima ``keys`` (int64, 3 n_total; see ``fused_scores``); with ``out=False`` the matrix is then
    not stored at all."""
    a = _check_clouds(pcs_1, "pcs_1")
    symmetric = pcs_2 is None
    b = a if symmetric else _check_clouds(pcs_2, "pcs_2")
    na, pa, _ = a.shape
    nb, pb, _ = b.shape
    begin, end, stride = rows if rows is not None else (0, na, 1)
    nrows = len(range(begin, end, stride))
    flags = 0
    if symmetric:
        flags |= _lib.MATRIX_SYMMETRIC
        if not compact_rows:
            flags |= _lib.MATRIX_MIRROR
    if compact_rows:
        flags |= _lib.MATRIX_COMPACT_ROWS
    if merge_origin is None:
        merge_origin = max(pa, pb) > MERGE_ORIGIN_ABOVE
    if merge_origin:
        flags |= _lib.MATRIX_MERGE_ORIGIN
    store = out is not False
    if not store and fused is None:
        raise ValueError("out=False needs fused=...")
    if out is None:
        out = torch.zeros(nrows if compact_rows else na, nb, device=a.device, dtype=torch.float32)
    if na == 0 or nb == 0 or nrows == 0:
        return out if store else None
    if pa == 0 or pb == 0:
        raise ValueError("clouds must hold at least one point")
    lib = _lib.load()
    nbytes = lib.dusty_chamfer_matrix_workspace_bytes(na, pa, 0 if symmetric else nb, pb)
    ws = _lib.workspace(nbytes, a.device)
    with torch.cuda.device(a.device):
        if KERNEL_EVENTS is not None:       # bench.py: device time of the launch on its own stream
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        m_ptr, ldm = (_lib.ptr(out), out.stride(0)) if store else (None, 0)
        if fused is None:
            _lib.check(lib.dusty_chamfer_matrix(_lib.ptr(a), na, pa, _lib.ptr(b), nb, pb, begin, end, stride, flags,
                                                m_ptr, ldm, _lib.ptr(ws), nbytes, _lib.stream_of(a)),
                       "dusty_chamfer_matrix")
        else:
            keys, off_1, off_2, n_ref, n_total = fused
            assert keys.dtype == torch.int64 and keys.numel() == 3 * n_total and keys.is_contiguous()
            _lib.check(lib.dusty_chamfer_matrix_fused(_lib.ptr(a), na, pa, _lib.ptr(b), nb, pb, begin, end, stride, flags,
                                                      m_ptr, ldm, off_1, off_2, n_ref, n_total, _lib.ptr(keys),
                                                      _lib.ptr(ws), nbytes, _lib.stream_of(a)),
                       "dusty_chamfer_matrix_fused")
        if KERNEL_EVENTS is not None:
            ev[1].record()
            KERNEL_EVENTS.append(ev)
    return out if store else None


def emd_matrix(pcs_1, pcs_2, rows=None, out=None, fused=None):
    """M[i,j] = compute_emd(pcs_1[i:i+1], pcs_2[j:j+1]) bit for bit, in one launch. EMD is not symmetric, so every
    entry is computed. ``rows=(begin,end,stride)`` restricts the computation to a row shard (other rows of ``out``
    are left as they are). ``fused=(keys, stacked_offset_1, stacked_offset_2, n_ref, n_total)`` also reduces every
    entry into the packed minima ``keys`` (int64, 3 n_total; see ``emd_scores``); with ``out=False`` the matrix is
    then not stored at all."""
    a = _check_clouds(pcs_1, "pcs_1")
    b = _check_clouds(pcs_2, "pcs_2")
    na, pa, _ = a.shape
    nb, pb, _ = b.shape
    begin, end, stride = rows if rows is not None else (0, na, 1)
    store = out is not False
    if not store and fused is None:
        raise ValueError("out=False needs fused=...")
    if out is None:
        out = torch.zeros(na, nb, device=a.device, dtype=torch.float32)
    if pa == 0 or pb == 0:
        raise ValueError("clouds must hold at least one point")
    if na == 0 or nb == 0 or len(range(begin, end, stride)) == 0:
        return out if store else None
    keys, off_1, off_2, n_ref, n_total = fused if fused is not None else (None, 0, 0, 0, 0)
    if keys is not None:
        assert keys.dtype == torch.int64 and keys.numel() == 3 * n_total and keys.is_contiguous()
    lib = _lib.load()
    nbytes = lib.dusty_emd_matrix_workspace_bytes(na, pa, nb, pb)
    ws = _lib.workspace(nbytes, a.device)
    with torch.cuda.device(a.device):
        if KERNEL_EVENTS is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        m_ptr, ldm = (_lib.ptr(out), out.stride(0)) if store else (None, 0)
        _lib.check(lib.dusty_emd_matrix(_lib.ptr(a), na, pa, _lib.ptr(b), nb, pb, begin, end, stride, m_ptr, ldm, off_1, off_2,
                                        n_ref, n_total, _lib.ptr(keys), _lib.ptr(ws), nbytes, _lib.stream_of(a)),
                   "dusty_emd_matrix")
        if KERNEL_EVENTS is not None:
            ev[1].record()
            KERNEL_EVENTS.append(ev)
    return out if store else None


def _pairwise_distance(pcs_1, pcs_2, batch_size, metrics=("cd",), verbose=True):
    """{"cd": (B_1,B_2)} like the reference (cov_mmd_1nna.py:24-51). ``batch_size`` (the reference's
    column block) and ``verbose`` (its tqdm bar) are accepted and have no effect."""
    # EMD matrices come from emd_matrix(pcs_1, pcs_2); this function keeps refusing "emd".
    if "emd" in metrics:
        raise NotImplementedError("EMD is not part of the path (the reference's extension does not build on "
                                  "torch>=2 and its callers pass metrics=('cd',))")
    distance = {}
    if "cd" in metrics:
        same = pcs_1 is pcs_2 or (pcs_1.data_ptr() == pcs_2.data_ptr() and pcs_1.shape == pcs_2.shape
                                  and pcs_1.stride() == pcs_2.stride())
        distance["cd"] = chamfer_matrix(pcs_1, None if same else pcs_2)
    return distance


def _compute_cov_mmd(M_rg):
    N_ref, N_gen = M_rg.shape
    mmd_gen, min_idx_gen = M_rg.min(dim=0)
    mmd_ref, _ = M_rg.min(dim=1)
    mmd = mmd_ref.mean().item()
    mmd_gen = mmd_gen.mean().item()
    cov = float(len(torch.unique(min_idx_gen))) / float(N_ref)
    return {"mmd": mmd, "mmd-sample": mmd_gen, "cov": cov}


def _nna_scores(tp, fp, fn, tn, total):
    s = {"tp": tp, "fp": fp, "fn": fn, "tn": tn}
    s.update({
        "precision": s["tp"] / (s["tp"] + s["fp"] + 1e-10),
        "recall": s["tp"] / (s["tp"] + s["fn"] + 1e-10),
        "accuracy_t": s["tp"] / (s["tp"] + s["fn"] + 1e-10),
        "accuracy_f": s["tn"] / (s["tn"] + s["fp"] + 1e-10),
        # torch.eq(label, pred).float().mean().item(): an f32 mean of 0/1 values
        "accuracy": float(np.float32(tp + tn) / np.float32(total)),
    })
    return s


def _finalize_device(M_rr, M_rg, M_gg):
    """COV/MMD/1-NNA (k=1) in three small kernels, one 28-byte read-back."""
    N_ref, N_gen = M_rg.shape
    M_rr, M_rg, M_gg = M_rr.contiguous(), M_rg.contiguous(), M_gg.contiguous()
    lib = _lib.load()
    nbytes = lib.dusty_cov_mmd_1nna_workspace_bytes(N_ref, N_gen)
    ws = _lib.workspace(nbytes, M_rg.device)
    out = torch.empty(7, device=M_rg.device, dtype=torch.float32)
    with torch.cuda.device(M_rg.device):
        _lib.check(lib.dusty_cov_mmd_1nna_finalize(_lib.ptr(M_rr), _lib.ptr(M_rg), _lib.ptr(M_gg), N_ref, N_gen,
                                                   _lib.ptr(out), _lib.ptr(ws), nbytes, _lib.stream_of(M_rg)),
                   "dusty_cov_mmd_1nna_finalize")
    o = [float(v) for v in out.tolist()]
    cov_mmd = {"mmd": o[0], "mmd-sample": o[1], "cov": float(o[2]) / float(N_ref)}
    return cov_mmd, _nna_scores(o[3], o[4], o[5], o[6], N_ref + N_gen)


def _compute_nna(M_rr, M_rg, M_gg, k, sqrt=False):
    """Leave-one-out k-NN two-sample test (reference cov_mmd_1nna.py:68-106) on the device kernels. ``sqrt`` only
    rescales the distances monotonically (``M.abs().sqrt()``), so the k nearest rows -- and every score -- are the
    same with or without it; it is accepted for signature compatibility."""
    if k == 1:
        return _finalize_device(M_rr, M_rg, M_gg)[1]
    N_ref, N_gen = M_rg.shape
    M_rr, M_rg, M_gg = M_rr.contiguous(), M_rg.contiguous(), M_gg.contiguous()
    lib = _lib.load()
    nbytes = lib.dusty_cov_mmd_1nna_workspace_bytes(N_ref, N_gen)
    ws = _lib.workspace(nbytes, M_rg.device)
    out = torch.empty(7, device=M_rg.device, dtype=torch.float32)
    with torch.cuda.device(M_rg.device):
        _lib.check(lib.dusty_cov_mmd_knna_finalize(_lib.ptr(M_rr), _lib.ptr(M_rg), _lib.ptr(M_gg), N_ref, N_gen, int(k),
                                                   _lib.ptr(out), _lib.ptr(ws), nbytes, _lib.stream_of(M_rg)),
                   "dusty_cov_mmd_knna_finalize")
    o = [float(v) for v in out.tolist()]
    return _nna_scores(o[3], o[4], o[5], o[6], N_ref + N_gen)


def pairwise_matrices(pcs_gen, pcs_ref):
    """(M_rr, M_rg, M_gg). Same point count: one stacked symmetric launch (row-sharded over the
    process group when there is one); otherwise three launches."""
    gen = _check_clouds(pcs_gen, "pcs_gen")
    ref = _check_clouds(pcs_ref, "pcs_ref")
    nr, ng = ref.size(0), gen.size(0)
    if ref.size(1) == gen.size(1):
        stacked = torch.cat([ref, gen], dim=0)
        M = sharding.symmetric_chamfer_matrix(stacked)
        return M[:nr, :nr], M[:nr, nr:], M[nr:, nr:]
    return chamfer_matrix(ref), chamfer_matrix(ref, gen), chamfer_matrix(gen)


def fused_scores(pcs_gen, pcs_ref, group=None):
    """(cov/mmd dict, 1-NNA dict) without ever storing a matrix: every entry the matrix kernel computes is
    reduced on the spot into three packed (value, index) minima per stacked cloud (reference first, then
    generated: the order of _compute_nna's matrix, reference cov_mmd_1nna.py:71-79). Ranks of ``group``
    work on a cyclic row shard each and all-gather those vectors (24 B per cloud and rank)."""
    gen = _check_clouds(pcs_gen, "pcs_gen")
    ref = _check_clouds(pcs_ref, "pcs_ref")
    nr, ng = ref.size(0), gen.size(0)
    n = nr + ng
    if nr == 0 or ng == 0:
        raise ValueError("both sets must hold at least one cloud")
    rank, G = sharding.world(group)
    lib = _lib.load()
    keys = torch.empty(3 * n, device=ref.device, dtype=torch.int64)
    with torch.cuda.device(ref.device):
        _lib.check(lib.dusty_nn_keys_reset(_lib.ptr(keys), n, _lib.stream_of(keys)), "dusty_nn_keys_reset")
    if ref.size(1) == gen.size(1):      # one stacked symmetric launch fills M_rr, M_rg and M_gg's reductions
        stacked = torch.cat([ref, gen], dim=0)
        chamfer_matrix(stacked, None, rows=sharding.owned_rows(n, rank, G), compact_rows=True, out=False,
                       fused=(keys, 0, 0, nr, n))
    else:
        chamfer_matrix(ref, None, rows=sharding.owned_rows(nr, rank, G), compact_rows=True, out=False, fused=(keys, 0, 0, nr, n))
        chamfer_matrix(ref, gen, rows=sharding.owned_rows(nr, rank, G), compact_rows=True, out=False, fused=(keys, 0, nr, nr, n))
        chamfer_matrix(gen, None, rows=sharding.owned_rows(ng, rank, G), compact_rows=True, out=False, fused=(keys, nr, nr, nr, n))
    return _scores_from_keys(keys, nr, ng, group)


def _scores_from_keys(keys, nr, ng, group):
    """All-gather every rank's packed minima and reduce them to (cov/mmd dict, 1-NNA dict)."""
    n = nr + ng
    lib = _lib.load()
    gathered = sharding.all_gather_keys(keys, group)
    nbytes = lib.dusty_cov_mmd_1nna_workspace_bytes(nr, ng)
    ws = _lib.workspace(nbytes, keys.device)
    out = torch.empty(7, device=keys.device, dtype=torch.float32)
    with torch.cuda.device(keys.device):
        _lib.check(lib.dusty_cov_mmd_1nna_from_keys(_lib.ptr(gathered), gathered.size(0), nr, ng, _lib.ptr(out), _lib.ptr(ws),
                                                    nbytes, _lib.stream_of(keys)), "dusty_cov_mmd_1nna_from_keys")
    o = [float(v) for v in out.tolist()]
    cov_mmd = {"mmd": o[0], "mmd-sample": o[1], "cov": float(o[2]) / float(nr)}
    return cov_mmd, _nna_scores(o[3], o[4], o[5], o[6], n)


def emd_pairwise_matrices(pcs_gen, pcs_ref):
    """(M_rr, M_rg, M_gg) of compute_emd, each computed in full (EMD is not symmetric; M_gr is never needed)."""
    gen = _check_clouds(pcs_gen, "pcs_gen")
    ref = _check_clouds(pcs_ref, "pcs_ref")
    return emd_matrix(ref, ref), emd_matrix(ref, gen), emd_matrix(gen, gen)


def emd_scores(pcs_gen, pcs_ref, group=None):
    """fused_scores for EMD: three launches (M_rr, M_rg, M_gg), each row-sharded over ``group``, reduce every entry
    into the packed minima of the column-wise 1-NN matrix [[M_rr, M_rg], [M_rg^T, M_gg]] and the cross-set minima;
    one all-gather of those vectors, no matrix stored."""
    gen = _check_clouds(pcs_gen, "pcs_gen")
    ref = _check_clouds(pcs_ref, "pcs_ref")
    nr, ng = ref.size(0), gen.size(0)
    n = nr + ng
    if nr == 0 or ng == 0:
        raise ValueError("both sets must hold at least one cloud")
    rank, G = sharding.world(group)
    lib = _lib.load()
    keys = torch.empty(3 * n, device=ref.device, dtype=torch.int64)
    with torch.cuda.device(ref.device):
        _lib.check(lib.dusty_nn_keys_reset(_lib.ptr(keys), n, _lib.stream_of(keys)), "dusty_nn_keys_reset")
    emd_matrix(ref, ref, rows=sharding.owned_rows(nr, rank, G), out=False, fused=(keys, 0, 0, nr, n))
    emd_matrix(ref, gen, rows=sharding.owned_rows(nr, rank, G), out=False, fused=(keys, 0, nr, nr, n))
    emd_matrix(gen, gen, rows=sharding.owned_rows(ng, rank, G), out=False, fused=(keys, nr, nr, nr, n))
    return _scores_from_keys(keys, nr, ng, group)


@torch.no_grad()
def compute_cov_mmd_1nna(pcs_gen, pcs_ref, batch_size, metrics=("cd",), verbose=True):
    assert isinstance(metrics, tuple)
    results = {}
    for metric in ("cd", "emd"):
        if metric not in metrics:
            continue
        if FUSED_EPILOGUE:
            cov_mmd, nna = (fused_scores if metric == "cd" else emd_scores)(pcs_gen, pcs_ref)
        else:       # the three matrices, then three small kernels over them (kept for A/B tests)
            M_rr, M_rg, M_gg = (pairwise_matrices if metric == "cd" else emd_pairwise_matrices)(pcs_gen, pcs_ref)
            cov_mmd, nna = _finalize_device(M_rr, M_rg, M_gg)
        for k, v in cov_mmd.items():
            results.update({"{}-{}".format(k, metric): v})
        for k, v in nna.items():
            results.update({"1-nn-{}-{}".format(k, metric): v})
    return results
