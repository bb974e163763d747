"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports exactly what include/*.h declares,
the ctypes signature table matches the header, and the reference-named `_backend` surface is complete.
No kernel is launched here."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "ri_b200.h")
PKG = os.path.join(ROOT, "point-cloud-registration-based-on-rotation-invariant-feature_b200")


def header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(int|size_t)\s+(ri_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = [a.strip() for a in m.group(3).split(",")]
        if args == ["void"]:
            args = []
        out[m.group(2)] = (m.group(1), args)
    return out


@pytest.fixture(scope="module")
def built_lib():
    import __graft_entry__ as ge
    ge.build_library()
    return ctypes.CDLL(os.path.join(PKG, "libri_b200.so"))


def test_header_declares_something():
    fns = header_functions()
    assert len(fns) >= 14
    for must in ("ri_knn_f32", "ri_ppf_f32", "ri_ppf_gather_f32", "ri_sph_voxelize_f32", "ri_cube_voxelize_f32",
                 "ri_trilinear_devox_f32", "ri_sph_trilinear_devox_f32", "ri_voxel_edge_gather_f32"):
        assert must in fns


def test_library_exports_every_declared_symbol(built_lib):
    for name in header_functions():
        assert hasattr(built_lib, name), "libri_b200.so does not export %s" % name


def test_ctypes_table_matches_header(built_lib):
    import ri_b200
    table = ri_b200._lib.SIGNATURES
    fns = header_functions()
    assert set(table) == set(fns), (set(table) ^ set(fns))
    for name, (ret, args) in fns.items():
        res, argtypes = table[name]
        assert len(argtypes) == len(args), name
        assert (res is ctypes.c_size_t) == (ret == "size_t"), name
        for a, t in zip(args, argtypes):
            if a.startswith("const char*"):
                assert t is ctypes.c_char_p, (name, a)
            elif "*" in a:
                assert t is ctypes.c_void_p, (name, a)
            elif a.startswith("size_t"):
                assert t is ctypes.c_size_t, (name, a)
            elif a.startswith("unsigned long long"):
                assert t is ctypes.c_ulonglong, (name, a)
            elif a.startswith("long long"):
                assert t is ctypes.c_longlong, (name, a)
            elif a.startswith("float"):
                assert t is ctypes.c_float, (name, a)
            else:
                assert t is ctypes.c_int, (name, a)


def test_abi_version_and_workspace_query(built_lib):
    built_lib.ri_abi_version.restype = ctypes.c_int
    assert built_lib.ri_abi_version() >= 1
    built_lib.ri_voxelize_workspace_bytes.restype = ctypes.c_size_t
    built_lib.ri_voxelize_workspace_bytes.argtypes = [ctypes.c_int] * 4
    small = built_lib.ri_voxelize_workspace_bytes(1, 64, 1024, 32)
    big = built_lib.ri_voxelize_workspace_bytes(32, 64, 1024, 32)
    # per cloud: ~5 int tables of N entries + the compact means table C * N floats
    assert 4 * 1024 * 4 + 64 * 1024 * 4 <= small < big <= 32 * (6 * 1024 * 4 + 64 * 1024 * 4 + 1024)


def test_spherical_devox_refuses_r_below_4_before_any_launch(built_lib):
    """The spherical devoxelizer's corner indices reach r^2 + 7r + 4, past the r^3 grid for r = 2 and 3: the entry point
    returns RI_ERR_UNSUPPORTED (-3) before touching a pointer or the device (null pointers, no GPU needed here)."""
    fn = built_lib.ri_sph_trilinear_devox_f32
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 4 + [ctypes.c_void_p] * 4
    for r in (2, 3):
        assert fn(None, None, None, 2, 5, 100, r, None, None, None, None) == -3, r
    assert fn(None, None, None, 2, 5, 100, 4, None, None, None, None) == -1     # r = 4 passes the guard (null g_inds: bad arg)


def test_backend_has_reference_function_names():
    """The hot-path subset of src/bindings.cpp:13-56."""
    import ri_b200
    for fn in ("knn_forward_cuda", "knn_backward_cuda", "spherical_ppf_forward", "avg_voxelize_forward",
               "avg_voxelize_backward", "spherical_avg_voxelize_forward", "spherical_avg_voxelize_backward",
               "trilinear_devoxelize_forward", "trilinear_devoxelize_backward",
               "spherical_trilinear_devoxelize_forward", "spherical_trilinear_devoxelize_backward"):
        assert callable(getattr(ri_b200._backend, fn))
    for fn in ("k_nearest_neighbor", "ppf", "avg_voxelize", "spherical_avg_voxelize", "trilinear_devoxelize",
               "spherical_trilinear_devoxelize"):
        assert callable(getattr(ri_b200.functional, fn))
    for cls in ("Voxelization", "Spherical_Voxelization", "knnModule", "PVConv"):
        assert hasattr(ri_b200.modules, cls)


def test_ops_refuse_cpu_tensors():
    """No CPU fallback: a CPU tensor is an error, exactly like the reference's CHECK_CUDA (utils.hpp:15)."""
    import torch
    import ri_b200  # noqa: F401
    x = torch.randn(1, 3, 16)
    with pytest.raises(RuntimeError):
        torch.ops.ri.knn(x, x, 2)
    with pytest.raises(RuntimeError):
        torch.ops.ri.ppf(x, x, x, x)
    with pytest.raises(RuntimeError):
        ri_b200.FrontEnd(1, 16, 4, device="cpu")


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "cpu_oracle" not in text and "ri_oracle" not in text and "oracle." not in text, f
