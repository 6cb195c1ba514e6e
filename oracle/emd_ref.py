"""ctypes front end of oracle/emd_reference.cu, the reference's EMD kernels restated (built with nvcc for sm_100a
into oracle/_build/libemd_ref.so with the library's flags). Inputs and outputs are CUDA torch tensors."""
import ctypes as C
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emd_reference.cu")
LIB = os.path.join(HERE, "_build", "libemd_ref.so")
# the flags of dusty-gan_b200/build.py that affect arithmetic: -O3, default -fmad / -prec-div / -prec-sqrt
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]
_lib = None


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the EMD reference oracle cannot be built")


def build(force=False):
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(SRC):
        subprocess.check_call([_nvcc(), *FLAGS, "-o", LIB, SRC, "-lcudart"])
    return LIB


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        for name in ("emd_ref_approxmatch", "emd_ref_matchcost", "emd_ref_matchcost_grad"):
            getattr(_lib, name).restype = C.c_int
    return _lib


def _p(t):
    return C.c_void_p(t.data_ptr())


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed with cudaError {rc}")


def approxmatch(xyz1, xyz2):
    """xyz1 (b,n,3), xyz2 (b,m,3) CUDA f32 -> match (b,m,n), the reference's dense matrix."""
    import torch
    a, c = xyz1.contiguous().float(), xyz2.contiguous().float()
    b, n, m = a.size(0), a.size(1), c.size(1)
    match = torch.empty(b, m, n, device=a.device, dtype=torch.float32)
    temp = torch.empty(32 * (n + m) * 2, device=a.device, dtype=torch.float32)
    with torch.cuda.device(a.device):
        _check(lib().emd_ref_approxmatch(b, n, m, _p(a), _p(c), _p(match), _p(temp)), "approxmatch")
    torch.cuda.synchronize(a.device)
    return match


def matchcost(xyz1, xyz2, match):
    import torch
    a, c = xyz1.contiguous().float(), xyz2.contiguous().float()
    b, n, m = a.size(0), a.size(1), c.size(1)
    out = torch.empty(b, device=a.device, dtype=torch.float32)
    with torch.cuda.device(a.device):
        _check(lib().emd_ref_matchcost(b, n, m, _p(a), _p(c), _p(match), _p(out)), "matchcost")
    torch.cuda.synchronize(a.device)
    return out


def matchcost_grad(xyz1, xyz2, match, grad_cost):
    import torch
    a, c = xyz1.contiguous().float(), xyz2.contiguous().float()
    b, n, m = a.size(0), a.size(1), c.size(1)
    g1, g2 = torch.zeros_like(a), torch.zeros_like(c)
    g = grad_cost.contiguous().float()
    with torch.cuda.device(a.device):
        _check(lib().emd_ref_matchcost_grad(b, n, m, _p(g), _p(a), _p(c), _p(match), _p(g1), _p(g2)), "matchcost_grad")
    torch.cuda.synchronize(a.device)
    return g1, g2


def earth_mover_distance(xyz1, xyz2):
    """The reference's forward: cost (b,) of (b,n,3) x (b,m,3) CUDA clouds."""
    return matchcost(xyz1, xyz2, approxmatch(xyz1, xyz2))


def emd_matrix(A, B):
    """M[i,j] = reference cost(A[i], B[j]) / pa, the reference compute_emd, one pair batch per row."""
    import torch
    na, pa = A.size(0), A.size(1)
    nb = B.size(0)
    M = torch.empty(na, nb, device=A.device, dtype=torch.float32)
    for i in range(na):
        M[i] = earth_mover_distance(A[i:i + 1].expand(nb, -1, -1), B) / pa
    return M
