"""ctypes binding of libdustyb200.so (the C ABI declared in include/dusty_b200.h).

This is the stub a reference maintainer would add in place of the two
``torch.utils.cpp_extension.load`` calls (reference cd/chamfer_distance.py:7-13,
fps/furthest_point_sampling.py:10-16). The library is looked up in-tree only
(``dusty-gan_b200/lib``); if it is missing the import of any op fails loudly -- there is no fallback.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdustyb200.so")

c_float_p = C.c_void_p
c_int_p = C.c_void_p


class Gate(C.Structure):
    _fields_ = [("mode", C.c_int32), ("hard", C.c_int32), ("noise_a", C.c_void_p), ("noise_b", C.c_void_p),
                ("batch_stride", C.c_int64), ("pixel_stride", C.c_int64), ("inv_tau", C.c_float), ("eps", C.c_float)]


class HeadParams(C.Structure):
    _fields_ = [("b", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("conf_channels", C.c_int32),
                ("gate_pixel", Gate), ("gate_image", Gate),
                ("threshold", C.c_float), ("drop_const", C.c_float),
                ("tol", C.c_float), ("disp_scale", C.c_float), ("disp_shift", C.c_float), ("min_depth", C.c_float),
                ("inv_range", C.c_float), ("range", C.c_float), ("inv_max_depth", C.c_float),
                ("points_layout", C.c_int32)]


class ScanParams(C.Structure):
    _fields_ = [("b", C.c_int32), ("hs", C.c_int32), ("ws", C.c_int32), ("channels", C.c_int32),
                ("h", C.c_int32), ("w", C.c_int32), ("scale_h", C.c_float), ("scale_w", C.c_float),
                ("min_depth", C.c_float), ("max_depth", C.c_float), ("range", C.c_float),
                ("disp_lo", C.c_float), ("inv_disp_range", C.c_float), ("drop_const", C.c_float)]


ABI_VERSION = 3          # DUSTY_B200_ABI_VERSION of include/dusty_b200.h
NOISE_NONE, NOISE_LOGISTIC, NOISE_UNIFORM = 0, 1, 2
MATRIX_SYMMETRIC, MATRIX_MIRROR, MATRIX_COMPACT_ROWS, MATRIX_PREPARED, MATRIX_MERGE_ORIGIN = 1, 2, 4, 8, 16

# name -> (restype, argtypes); kept in one table so the symbol-export test can walk it
SIGNATURES = {
    "dusty_abi_version": (C.c_int, []),
    "dusty_last_error_string": (C.c_char_p, []),
    "dusty_launch_count": (C.c_uint64, []),
    "dusty_chamfer_forward_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_chamfer_forward": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_int, c_float_p, c_float_p,
                                        c_int_p, c_int_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_chamfer_backward_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_chamfer_backward": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_int, c_float_p, c_float_p,
                                         c_int_p, c_int_p, c_float_p, c_float_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_chamfer_matrix_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "dusty_chamfer_matrix": (C.c_int, [c_float_p, C.c_int, C.c_int, c_float_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, c_float_p, C.c_longlong, C.c_void_p, C.c_size_t,
                                       C.c_void_p]),
    "dusty_nn_keys_bytes": (C.c_size_t, [C.c_int]),
    "dusty_nn_keys_reset": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "dusty_chamfer_matrix_fused": (C.c_int, [c_float_p, C.c_int, C.c_int, c_float_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, c_float_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_cov_mmd_1nna_from_keys": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, c_float_p, C.c_void_p, C.c_size_t,
                                               C.c_void_p]),
    "dusty_symmetric_from_shards": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, c_float_p, C.c_longlong, C.c_void_p]),
    "dusty_cov_mmd_1nna_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "dusty_cov_mmd_1nna_finalize": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, C.c_int, c_float_p,
                                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_cov_mmd_knna_finalize": (C.c_int, [c_float_p, c_float_p, c_float_p, C.c_int, C.c_int, C.c_int, c_float_p,
                                              C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_emd_forward_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_emd_forward": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_int, c_float_p, c_float_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    "dusty_emd_backward": (C.c_int, [c_float_p, c_float_p, C.c_int, C.c_int, C.c_int, c_float_p, c_float_p, c_float_p,
                                     c_float_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_emd_matrix_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "dusty_emd_matrix": (C.c_int, [c_float_p, C.c_int, C.c_int, c_float_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   c_float_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_size_t, C.c_void_p]),
    "dusty_jsd_vote":(C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_int, c_float_p, c_int_p, c_float_p, C.c_float,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "dusty_jsd_from_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, c_float_p, C.c_void_p]),
    "dusty_swd_descriptors_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "dusty_swd_descriptors": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_int_p, C.c_int,
                                        c_float_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_swd_sliced_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_swd_sliced": (C.c_int, [c_float_p, c_float_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, c_float_p, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_depth_metrics_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_depth_metrics": (C.c_int, [C.POINTER(HeadParams), c_float_p, c_float_p, C.c_void_p, c_float_p, c_float_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_fps_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_fps": (C.c_int, [c_float_p, C.c_int, C.c_int, C.c_int, c_int_p, c_float_p, C.c_void_p, C.c_size_t,
                            C.c_void_p]),
    "dusty_gather_points": (C.c_int, [c_float_p, c_int_p, C.c_int, C.c_int, C.c_int, C.c_int, c_float_p, C.c_void_p]),
    "dusty_gather_points_grad": (C.c_int, [c_float_p, c_int_p, C.c_int, C.c_int, C.c_int, C.c_int, c_float_p,
                                           C.c_void_p]),
    "dusty_logistic_noise": (C.c_int, [c_float_p, c_float_p, C.c_float, C.c_size_t, c_float_p, C.c_void_p]),
    "dusty_gumbel_sigmoid": (C.c_int, [c_float_p, C.POINTER(Gate), C.c_float, C.c_int, C.c_int, c_float_p, C.c_void_p]),
    "dusty_head_project_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_head_project": (C.c_int, [C.POINTER(HeadParams), c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                     c_float_p, c_int_p, c_int_p, c_float_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dusty_head_project_backward_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "dusty_head_project_backward": (C.c_int, [C.POINTER(HeadParams), c_float_p, c_float_p, c_float_p, c_float_p,
                                              c_float_p, c_float_p, c_float_p, c_float_p, c_float_p, C.c_void_p,
                                              C.c_size_t, C.c_void_p]),
    "dusty_inv_to_xyz": (C.c_int, [C.POINTER(HeadParams), c_float_p, c_float_p, c_float_p, C.c_void_p]),
    "dusty_scan_preprocess": (C.c_int, [C.POINTER(ScanParams), c_float_p, c_float_p, c_float_p, c_float_p, c_float_p,
                                        c_float_p, C.c_void_p]),
    "dusty_chamfer_count_pairs": (C.c_int, [C.c_int, C.POINTER(C.c_uint64)]),
    "dusty_probe_fp32_peak": (C.c_int, [C.c_int, c_float_p, C.POINTER(C.c_double), C.c_void_p]),
}

_lib = None


def load():
    """Load the shared object (once) and attach the prototypes. Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python dusty-gan_b200/build.py` "
            "(or __graft_entry__.build()). dusty-gan_b200 has no CPU/PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.dusty_abi_version() != ABI_VERSION:
        raise RuntimeError("libdustyb200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def check(rc, what):
    """Turn a non-zero C-ABI return into a RuntimeError (the reference only printf'ed kernel errors)."""
    if rc != 0:
        msg = load().dusty_last_error_string().decode(errors="replace")
        raise RuntimeError(f"{what} failed with code {rc}: {msg}")


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_of(t):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def require_cuda(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: dusty-gan_b200 runs on B200 only (no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")


def workspace(nbytes, device):
    """Scratch owned by the caller side of the ABI: a plain torch allocation (512-byte aligned)."""
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)


def launch_count():
    return int(load().dusty_launch_count())
