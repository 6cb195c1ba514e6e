"""Build libdustyb200.so in-tree with nvcc for sm_100a (and nothing else).

    python dusty-gan_b200/build.py [--force]

The shared object lands in dusty-gan_b200/lib/ (git-ignored, but shipped to the GPU box with the
working tree). No torch headers are involved: the library's ABI is include/dusty_b200.h.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libdustyb200.so")
SOURCES = ["api.cu", "chamfer.cu", "fps.cu", "head_project.cu", "metrics.cu", "jsd.cu", "scan_preprocess.cu", "emd.cu", "swd.cu",
           "depth_metrics.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "-I", os.path.join(ROOT, "include"), "-I", CSRC,
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdustyb200.so cannot be built")


def _fingerprint():
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in sorted(os.listdir(CSRC)) + ["../../include/dusty_b200.h"]:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every .cu of the library for sm_100a; returns the path of the shared object."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "libdustyb200.stamp")
    fp = _fingerprint()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == fp:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lcudart"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libdustyb200.so failed")
    with open(stamp, "w") as fh:
        fh.write(fp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
