"""The C-ABI boundary without a GPU: the library loads, exports exactly what include/dusty_b200.h
declares, the ctypes table covers every symbol, and ops refuse to run without CUDA tensors."""
import os
import re
import subprocess

import pytest
import torch

from conftest import ROOT


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dusty_b200.h")).read()
    return sorted(set(re.findall(r"^DUSTY_API [\w \*]+?\**\s*(dusty_\w+)\(", text, flags=re.M)))


def test_header_declares_the_documented_entry_points():
    syms = declared_symbols()
    for must in ("dusty_chamfer_forward", "dusty_chamfer_matrix", "dusty_fps", "dusty_gather_points",
                 "dusty_head_project", "dusty_inv_to_xyz", "dusty_gumbel_sigmoid", "dusty_logistic_noise",
                 "dusty_cov_mmd_1nna_finalize", "dusty_chamfer_backward", "dusty_scan_preprocess"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = sorted(set(re.findall(r" T (dusty_\w+)", out)))
    assert exported == declared_symbols()
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    lib = _lib.load()
    assert lib.dusty_abi_version() == _lib.ABI_VERSION == 3
    assert lib.dusty_launch_count() == 0 or lib.dusty_launch_count() > 0


def test_library_is_sm100a_only_and_uses_tma_and_packed_fp32():
    from dusty_gan_b200 import _lib
    elf = subprocess.check_output(["cuobjdump", "-lelf", _lib.LIB_PATH], text=True)
    archs = set(re.findall(r"sm_(\d+a?)", elf))
    assert archs == {"100a"}, archs
    sass = subprocess.check_output(["cuobjdump", "-sass", _lib.LIB_PATH], text=True)
    assert "UBLKCP" in sass            # 1-D TMA bulk copies feed the Chamfer tiles
    assert "FFMA2" in sass             # packed FP32 FMA in the search loop
    assert "FMNMX3" in sass            # 3-input min
    assert "SYNCS" in sass             # mbarrier transactions


def test_workspace_queries_without_a_gpu():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    assert lib.dusty_chamfer_forward_workspace_bytes(2, 2048, 2048) == 2 * 2 * 2048 * 16
    assert lib.dusty_chamfer_forward_workspace_bytes(0, 5, 5) == 0
    assert lib.dusty_chamfer_matrix_workspace_bytes(10, 33, 0, 33) == 10 * 64 * 16 + 256 + 768 + 10 * 64 * 16      # scan copies + per-cloud meta + chunk boxes + block boxes (32 x 2 float4 per cloud)
    assert lib.dusty_fps_workspace_bytes(3, 1001, 16) >= 3 * 4 * 1004 * 4
    assert lib.dusty_head_project_workspace_bytes(256, 64, 512) >= 256 * 8 * 4
    assert lib.dusty_cov_mmd_1nna_workspace_bytes(1000, 1000) > 0


def test_argument_errors_are_reported_not_printed():
    from dusty_gan_b200 import _lib
    lib = _lib.load()
    rc = lib.dusty_chamfer_forward(None, None, -1, 4, 4, None, None, None, None, None, 0, None)
    assert rc == -1
    assert b"negative size" in lib.dusty_last_error_string()
    with pytest.raises(RuntimeError, match="code -1"):
        _lib.check(rc, "dusty_chamfer_forward")
    assert lib.dusty_fps(None, 1, 0, 4, None, None, None, 0, None) == -1
    p = _lib.ScanParams()
    p.b, p.hs, p.ws, p.channels, p.h, p.w = 1, 64, 2048, 2, 64, 512
    assert lib.dusty_scan_preprocess(p, None, None, None, None, None, None, None) == -1
    assert b"bad shape" in lib.dusty_last_error_string()


def test_ops_refuse_cpu_tensors():
    from dusty_gan_b200.utils.sampling.fps import furthest_point_sampling
    from dusty_gan_b200.utils.metrics.cov_mmd_1nna import compute_cov_mmd_1nna
    from dusty_gan_b200.utils.lidar import LiDAR, synthetic_hdl64e_angles
    with pytest.raises(RuntimeError, match="no CPU path"):
        furthest_point_sampling(torch.zeros(1, 8, 3), 2)
    with pytest.raises(RuntimeError, match="no CPU path"):
        compute_cov_mmd_1nna(torch.zeros(2, 8, 3), torch.zeros(2, 8, 3), 512, ("cd",))
    lidar = LiDAR(8, 32, 0.9, 120.0, angle=synthetic_hdl64e_angles())
    assert lidar.angle.shape == (1, 2, 8, 32)
    with pytest.raises(RuntimeError, match="no CPU path"):
        lidar.inv_to_xyz(torch.zeros(1, 1, 8, 32))


def test_missing_library_fails_loudly(monkeypatch):
    from dusty_gan_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libdustyb200.so")
    with pytest.raises(RuntimeError, match="no CPU/PyTorch fallback"):
        _lib.load()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "dusty-gan_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "/root/reference" not in text, f


def _build_c_demo(tmp_path):
    from dusty_gan_b200 import _lib
    exe = str(tmp_path / "c_abi_demo")
    libdir = os.path.dirname(_lib.LIB_PATH)
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(cuda, "include"), os.path.join(ROOT, "examples", "c_abi_demo.c"),
                           "-L", libdir, "-ldustyb200", "-L", os.path.join(cuda, "lib64"), "-lcudart", "-lm",
                           "-Wl,-rpath," + libdir, "-o", exe])
    return exe


def test_header_is_plain_c_and_a_c_program_links(tmp_path):
    """The boundary is C: the header parses as pedantic C99 and a program without Python or torch links
    against the shared object (it runs in tests/test_gpu_c_abi.py)."""
    subprocess.check_call(["gcc", "-std=c99", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c",
                           os.path.join(ROOT, "include", "dusty_b200.h")])
    assert os.path.exists(_build_c_demo(tmp_path))


def test_struct_layouts_match_the_ctypes_mirrors(tmp_path):
    """Every Python call passes the parameter structs by pointer through the ctypes mirrors in _lib.py: their size and
    each field's offset must be what a C compiler makes of include/dusty_b200.h."""
    import ctypes
    from dusty_gan_b200 import _lib
    mirrors = {"dusty_gate": _lib.Gate, "dusty_head_params": _lib.HeadParams, "dusty_scan_params": _lib.ScanParams}
    lines = ["#include <stddef.h>", "#include <stdio.h>", '#include "dusty_b200.h"', "int main(void) {"]
    want = []
    for cname, cls in mirrors.items():
        lines.append(f'  printf("{cname} sizeof %zu\\n", sizeof({cname}));')
        want.append(f"{cname} sizeof {ctypes.sizeof(cls)}")
        for field, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{field} %zu\\n", offsetof({cname}, {field}));')
            want.append(f"{cname}.{field} {getattr(cls, field).offset}")
    lines += ["  return 0;", "}"]
    src, exe = tmp_path / "layout.c", str(tmp_path / "layout")
    src.write_text("\n".join(lines) + "\n")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe])
    assert subprocess.check_output([exe], text=True).splitlines() == want


def test_hot_kernels_keep_their_occupancy_shape():
    """Register budgets the measured numbers depend on (cuobjdump -res-usage): the dense Chamfer kernel at 128
    registers without local memory (two CTAs of 256 threads per SM), the head kernel at 32 (2048 threads per SM),
    the FPS throughput kernel within three CTAs per SM, and no stack or local memory in any of them."""
    from dusty_gan_b200 import _lib
    out = subprocess.check_output(["cuobjdump", "-res-usage", _lib.LIB_PATH], text=True)
    usage = dict(re.findall(r"Function (\S+):\s+REG:(\d+) STACK:\d+ SHARED:\d+ LOCAL:\d+", out))
    local = dict(re.findall(r"Function (\S+):\s+REG:\d+ STACK:(\d+) SHARED:\d+ LOCAL:\d+", out))

    def one(fragment):
        names = [n for n in usage if fragment in n]
        assert len(names) == 1, (fragment, names)
        return names[0]
    dense = one("nn_kernelILi8ELb1ELb0ELi256")
    assert int(usage[dense]) <= 128 and int(local[dense]) == 0
    for frag in ("nn_kernelILi8ELb1ELb0ELi128", "nn_kernelILi8ELb1ELb0ELi64", "nn_kernelILi8ELb1ELb0ELi32"):
        n = one(frag)
        assert int(usage[n]) <= 128 and int(local[n]) == 0, frag
    pair = one("nn_pair_split_kernel")                                 # resident-pair kernel: three 8-warp CTAs per SM
    assert int(usage[pair]) <= 85 and int(local[pair]) <= 16           # (the stack bytes belong to the double-division subroutine of the epilogue)
    assert int(usage[one("head_project_kernelILi1ELb0E")]) <= 32         # 8 CTAs of 256 threads per SM
    assert int(usage[one("head_project_kernelILi2ELb0E")]) <= 36         # DUSty-II: 7 CTAs per SM
    assert int(usage[one("head_project_kernelILi1ELb1E")]) <= 48         # with compaction: 5 CTAs per SM, 16 KB smem each
    assert int(usage[one("fps_multi_kernelILb1E")]) <= 84                # three clouds of 256 threads per SM, distances on chip
    assert int(usage[one("fps_multi_kernelILb0E")]) <= 40                # the six-per-SM layout kept for A/B runs
    assert int(usage[one("scan_preprocess_kernel")]) <= 40
