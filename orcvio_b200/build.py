"""Builds liborcvio_b200.so in-tree with nvcc for sm_100a.

    python -m orcvio_b200.build [--force] [--verbose]

The library is compiled file by file (objects cached by mtime under orcvio_b200/lib/obj)
and linked with `nvcc -shared`.  tri_kernel.cu is compiled with --fmad=false because the
Levenberg-Marquardt accept/reject decisions must follow the oracle's IEEE operation order.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(LIBDIR, "obj")
LIB = os.path.join(LIBDIR, "liborcvio_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
          "-Xcompiler", "-fno-strict-aliasing"]
SOURCES = {
    "tri_kernel.cu": ["--fmad=false"],
    "jac_kernel.cu": [],
    "project_kernel.cu": [],
    "info_kernel.cu": [],
    "peak_kernel.cu": [],
    "prop_kernel.cu": [],
    "zupt_kernel.cu": [],
    "obj_kernel.cu": [],
    "ekf_kernel.cu": [],
    "hybrid_kernel.cu": [],
    "metrics_kernel.cu": [],
    "consistency_kernel.cu": [],
    "kabsch_kernel.cu": [],
    "objlm_kernel.cu": [],
    "lm.cpp": [],
    "batch.cu": [],
    "objects.cu": [],
    "capi.cu": [],
    "config.cpp": [],
    "formats.cpp": [],
}


def _newer(src, obj, headers):
    if not os.path.exists(obj):
        return True
    t = os.path.getmtime(obj)
    return any(os.path.getmtime(p) > t for p in [src] + headers)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    os.makedirs(OBJDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "orcvio_b200.h"))
    objs = []
    rebuilt = False
    for src, extra in SOURCES.items():
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(OBJDIR, src + ".o")
        objs.append(obj)
        if force or _newer(path, obj, headers):
            cmd = [nvcc] + ARCH + COMMON + extra + ["-c", path, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas")
                cmd.insert(2, "-v")
                print(" ".join(cmd))
            subprocess.check_call(cmd)
            rebuilt = True
    if rebuilt or not os.path.exists(LIB):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB


def exported_symbols():
    """Names of every function declared in include/orcvio_b200.h (the C-ABI contract)."""
    import re
    hdr = open(os.path.join(HERE, "..", "include", "orcvio_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(orcvio_[a-z0-9_]+)\s*\(", hdr)))


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
