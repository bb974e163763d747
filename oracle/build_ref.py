"""Build the UNMODIFIED reference CUDA backend into oracle/_ref/ (test infrastructure only).

The reference (`/root/reference/PVCNN/modules/functional/backend.py:14-39`) JIT-compiles 21
sources into one pybind11 module `_multi_shape_pvcnn_backend`.  This recipe compiles the very
same files *where they lie* under /root/reference for sm_100a and drops the resulting .so into
`oracle/_ref/` (git-ignored, but shipped to the GPU box by gpurun).  No reference source is
copied into this repository.

The .so is the executable specification used by `tests/` (GPU parity), by
`oracle/make_golden.py` (golden fixture generation) and by `bench.py --impl reference-cuda`.
It is never imported by the product package.

Usage:  python oracle/build_ref.py            (no-op if /root/reference is absent or .so is fresh)
"""
import os
import sys
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
REF_SRC = "/root/reference/PVCNN/modules/functional/src"
OUT_DIR = os.path.join(HERE, "_ref")
NAME = "_multi_shape_pvcnn_backend"

# the exact list of backend.py:17-37
SOURCES = [
    'ball_query/ball_query.cpp', 'ball_query/ball_query.cu',
    'grouping/grouping.cpp', 'grouping/grouping.cu',
    'interpolate/neighbor_interpolate.cpp', 'interpolate/neighbor_interpolate.cu',
    'interpolate/trilinear_devox.cpp', 'interpolate/trilinear_devox.cu',
    'sampling/sampling.cpp', 'sampling/sampling.cu',
    'voxelization/vox.cpp', 'voxelization/vox.cu',
    'interpolate/spherical_trilinear_devox.cpp', 'interpolate/spherical_trilinear_devox.cu',
    'spherical_voxelization/spherical_vox.cpp', 'spherical_voxelization/spherical_vox.cu',
    'spherical_ppf/ppf.cpp', 'spherical_ppf/ppf.cu',
    'knn/knn.cpp', 'knn/knn.cu',
    'bindings.cpp',
]


def so_path():
    return os.path.join(OUT_DIR, NAME + ".so")


def build(force=False, verbose=False):
    if not os.path.isdir(REF_SRC):
        return None  # GPU box: only the prebuilt file is used
    if os.path.exists(so_path()) and not force:
        return so_path()
    os.makedirs(OUT_DIR, exist_ok=True)
    os.environ["TORCH_CUDA_ARCH_LIST"] = "10.0a"
    os.environ.setdefault("MAX_JOBS", str(os.cpu_count() or 8))
    from torch.utils.cpp_extension import load
    build_dir = os.path.join(OUT_DIR, "build")
    os.makedirs(build_dir, exist_ok=True)
    load(name=NAME,
         extra_cflags=['-O3', '-std=c++17'],          # same as backend.py:15
         sources=[os.path.join(REF_SRC, f) for f in SOURCES],
         build_directory=build_dir, verbose=verbose, is_python_module=False)
    shutil.copy2(os.path.join(build_dir, NAME + ".so"), so_path())
    shutil.rmtree(build_dir, ignore_errors=True)
    return so_path()


GRIDSUB_DIR = "/root/reference/cpp_wrappers/cpp_subsampling"
GRIDSUB_SO = os.path.join(OUT_DIR, "libgridsub_ref.so")


def build_gridsub(force=False):
    """The reference's CPU grid subsampling (cpp_wrappers/cpp_subsampling/grid_subsampling/grid_subsampling.cpp +
    cpp_utils/cloud/cloud.cpp, compiled where they lie with the flags of cpp_subsampling/setup.py) behind the C shim
    oracle/gridsub_ref_shim.cpp -> oracle/_ref/libgridsub_ref.so.  Returns the path, or None when the reference tree is
    absent and no prebuilt file exists."""
    if not os.path.isdir(GRIDSUB_DIR):
        return GRIDSUB_SO if os.path.exists(GRIDSUB_SO) else None
    if os.path.exists(GRIDSUB_SO) and not force:
        return GRIDSUB_SO
    import subprocess
    os.makedirs(OUT_DIR, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++11", "-fPIC", "-shared", "-I", GRIDSUB_DIR,
                           os.path.join(HERE, "gridsub_ref_shim.cpp"),
                           os.path.join(GRIDSUB_DIR, "grid_subsampling", "grid_subsampling.cpp"),
                           os.path.join(GRIDSUB_DIR, "..", "cpp_utils", "cloud", "cloud.cpp"),
                           "-o", GRIDSUB_SO])
    return GRIDSUB_SO


def ref_grid_subsampling(points, features=None, labels=None, grid_size=0.1):
    """Run the reference's own grid_subsampling() (unordered_map output order).  numpy in / out; None if unavailable."""
    import ctypes
    import numpy as np
    p = build_gridsub()
    if p is None:
        return None
    lib = ctypes.CDLL(p)
    pts = np.ascontiguousarray(points, np.float32)
    N = pts.shape[0]
    f = None if features is None else np.ascontiguousarray(features, np.float32).reshape(N, -1)
    l = None if labels is None else np.ascontiguousarray(labels, np.int32).reshape(N, -1)
    fdim = 0 if f is None else f.shape[1]
    ldim = 0 if l is None else l.shape[1]
    op = np.empty((N, 3), np.float32); of = np.empty((N, max(fdim, 1)), np.float32); ol = np.empty((N, max(ldim, 1)), np.int32)
    vp = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    lib.ref_grid_subsampling.restype = ctypes.c_int
    lib.ref_grid_subsampling.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3 + [ctypes.c_float] + [ctypes.c_void_p] * 3
    M = lib.ref_grid_subsampling(vp(pts), vp(f), vp(l), N, fdim, ldim, float(grid_size), vp(op), vp(of), vp(ol))
    return op[:M], (of[:M, :fdim] if fdim else None), (ol[:M, :ldim] if ldim else None)


def load_ref():
    """Import the prebuilt reference backend (needs `import torch` first). Returns module or None."""
    p = so_path()
    if not os.path.exists(p):
        return None
    import torch  # noqa: F401  (libtorch symbols)
    import importlib.util
    spec = importlib.util.spec_from_file_location(NAME, p)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("reference backend:", p)
    print("reference grid subsampling:", build_gridsub(force="--force" in sys.argv))
