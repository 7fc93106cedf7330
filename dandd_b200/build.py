"""Build the CUDA hot path (dandd_b200/csrc/*.cu) into an in-tree shared library for sm_100a.

nvcc cross-compiles without a GPU, so this runs in the build container; the resulting
libdandd_b200.so is git-ignored but travels to the GPU box with the repository snapshot."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libdandd_b200.so")
SOURCES = ["pack.cu", "sketch.cu", "card.cu", "planes.cu", "lattice.cu", "exact.cu", "leaveout.cu", "greedy.cu", "cover.cu", "api.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "hist.cuh", "swar.cuh", os.path.join("..", "..", "include", "dandd_b200.h")]
NVCC_FLAGS = ["-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"] + os.environ.get("DD_NVCC_EXTRA", "").split()


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the CUDA extension cannot be built")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu for sm_100a (-lineinfo for ncu source view) and link the C-ABI library."""
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stderr.write(out)
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    link = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
