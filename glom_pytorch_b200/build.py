"""Build libglom_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m glom_pytorch_b200.build          # or __graft_entry__.build()
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libglom_b200.so")
SOURCES = ["glom_api.cu", "simt_kernels.cu", "tc_kernels.cu", "islands.cu", "bwd_kernels.cu", "tc_bwd_kernels.cu",
           "contrastive.cu"]
HEADERS = ["engine.h", "ptx.cuh", os.path.join("..", "..", "include", "glom_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-cudart", "static",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def is_stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force=False, verbose=False, out_dir=None):
    """Compile every CUDA source of the engine into one shared library. Returns its path.
    out_dir: write the objects and the library there instead of into the package (always builds)."""
    if out_dir is None and not force and not is_stale():
        return LIB
    lib_path = LIB if out_dir is None else os.path.join(out_dir, os.path.basename(LIB))
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(CSRC if out_dir is None else out_dir, s.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static",
            "-Xcompiler", "-fPIC", *objs, "-o", lib_path]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("nvcc link failed")
    return lib_path


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
