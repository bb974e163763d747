"""Build libri_b200.so (the C-ABI library of include/ri_b200.h) in-tree with nvcc for sm_100a.

    python build.py            incremental (per-file objects under csrc/build/)
    python build.py --force    rebuild everything

nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels to the GPU box.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "libri_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SOURCES = ["abi.cu", "knn.cu", "knn_warp.cu", "ppf.cu", "prologue.cu", "voxelize.cu", "devox.cu", "grad.cu", "knn_grid.cu", "matcher.cu", "ballquery.cu", "localmlp.cu", "gridsub.cu", "pose.cu", "lrf.cu", "icp.cu", "normals.cu", "fgr.cu", "fpfh.cu", "teaser.cu", "fps.cu", "iss.cu"]

FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _compile(src, force, verbose):
    path = os.path.join(CSRC, src)
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    if force or _stale(obj, [path] + headers):
        cmd = [NVCC] + FLAGS + ["-I", os.path.join(HERE, "..", "include"), "-c", path, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(obj + ".log", "w") as f:
            f.write(log)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, log))
        if verbose:
            print(log)
        return True
    return False


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        changed = list(ex.map(lambda s: _compile(s, force, verbose), srcs))
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if any(changed) or _stale(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcudart", "-lcuda"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
