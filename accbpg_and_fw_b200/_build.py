"""Build recipe for libaccbpg_b200.so (sm_100a only, in-tree, no torch linkage).

    python accbpg_and_fw_b200/_build.py          # or  __graft_entry__.build()
    (run it by path: importing the package requires an up-to-date library)

nvcc cross-compiles without a GPU.  The shared object is written next to this file so
it travels with the repo snapshot to the GPU box; it links cudart statically and has
no other dependency than libcuda at run time.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libaccbpg_b200.so")
BUILD_DIR = os.path.join(HERE, "csrc", "build")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]
# files whose scalar expressions must round exactly like NumPy's (no FMA contraction)
SOURCES = {
    "vecops.cu": ["-fmad=false"],
    "linreg.cu": ["-fmad=false"],
    "linreg_small.cu": ["-fmad=false"],
    "fw.cu": ["-fmad=false"],
    "dopt.cu": [],
    "chol.cu": [],
    "sparse.cu": [],
    "small.cu": [],
    "prof.cu": [],
}


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a and link the C-ABI shared library.  Returns its path."""
    os.makedirs(BUILD_DIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "dmma.cuh"),
               os.path.join(HERE, "..", "include", "accbpg_b200.h"),
               os.path.abspath(__file__)]
    objs = []
    for src, extra in SOURCES.items():
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            raise RuntimeError(f"missing CUDA source {path}")
        obj = os.path.join(BUILD_DIR, src.replace(".cu", ".o"))
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + ARCH + COMMON + extra + ["-c", path, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            subprocess.run(cmd, check=True)
        objs.append(obj)
    if force or _stale(LIB, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-cudart", "static"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
