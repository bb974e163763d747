"""ctypes binding of libri_b200.so (include/ri_b200.h).  No fallback: if the library is missing or a symbol
is absent, importing this module raises — the ops of this package exist only as sm_100a CUDA kernels."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libri_b200.so")

_P = ctypes.c_void_p
_I = ctypes.c_int
_Z = ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/ri_b200.h one to one
SIGNATURES = {
    "ri_abi_version": (_I, []),
    "ri_debug_stamp": (_I, [_P, _P]),
    "ri_debug_set_knob": (_I, [ctypes.c_char_p, _I]),
    "ri_knn_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ri_knn_thread_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ri_knn_bilateral_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "ri_knn_grid_workspace_bytes": (_Z, [_I, _I, _I]),
    "ri_knn_grid_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "ri_knn_backward_f32": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "ri_ppf_f32": (_I, [_P, _P, _P, _P, _I, _I, _P, _P]),
    "ri_ppf_gather_f32": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "ri_knn_ppf_f32": (_I, [_P, _P, ctypes.c_longlong, _I, _I, _I, _P, _P, _P, _P]),
    "ri_vox_prologue_f32": (_I, [_P, _I, _P, _I, _I, _I, _I, ctypes.c_float, _I, _P, _P, _P, _P, _P]),
    "ri_split_xyz_normals_f32": (_I, [_P, _I, _I, _P, _P, _P, _P]),
    "ri_ppf_gather_packed_f32": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "ri_voxelize_workspace_bytes": (_Z, [_I, _I, _I, _I]),
    "ri_sph_voxelize_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "ri_cube_voxelize_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _Z, _P]),
    "ri_sph_voxelize_edge_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_cube_voxelize_edge_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_sph_voxelize_prepare_f32": (_I, [_P, _I, _I, _I, _I, _P, _P, _Z, _P]),
    "ri_cube_voxelize_prepare_f32": (_I, [_P, _I, _I, _I, _I, _P, _P, _Z, _P]),
    "ri_voxelize_means_f32": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _P, _Z, _P]),
    "ri_voxelize_fill_f32": (_I, [_I, _I, _I, _I, _I, _I, _P, _P, _P, _Z, _P]),
    "ri_vox_front_f32": (_I, [_P, _I, _P, _P, _I, _I, _I, _I, _I, ctypes.c_float, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_voxelize_backward_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ri_trilinear_devox_f32": (_I, [_P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ri_sph_trilinear_devox_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "ri_devox_backward_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "ri_voxel_edge_gather_f32": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ri_ball_query_f32": (_I, [_P, _P, _I, _I, _I, ctypes.c_float, _I, _P, _P]),
    "ri_local_ppf_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "ri_local_ppf_mlp_max_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _I, _P, _P, _I, _P, _P]),
    "ri_grouping_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "ri_grouping_backward_f32": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "ri_grid_subsample_workspace_bytes": (_Z, [_I]),
    "ri_grid_subsample_f32": (_I, [_P, _P, _P, _I, _I, _I, ctypes.c_float, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_pose_from_matches_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, ctypes.c_float, ctypes.c_float, _I,
                                     ctypes.c_ulonglong, _P, _P, _P, _P]),
    "ri_registration_metrics_f32": (_I, [_P, _P, _P, _I, _I, _P, _P]),
    "ri_lrf_change_coords_f32": (_I, [_P, _I, _P, _I, _I, _I, _P, _P, _P, _P]),
    "ri_icp_workspace_bytes": (_Z, [_I, _I, _I]),
    "ri_icp_f32": (_I, [_P, _P, _P, _P, _I, _I, _I, ctypes.c_float, _I, _I, ctypes.c_float, ctypes.c_float,
                        _P, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_generalized_icp_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, ctypes.c_float, ctypes.c_float, _I, ctypes.c_float,
                                    ctypes.c_float, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_robust_icp_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, ctypes.c_float, _I, ctypes.c_float, _I, ctypes.c_float,
                               _I, ctypes.c_float, ctypes.c_float, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_estimate_normals_f32": (_I, [_P, _I, _I, ctypes.c_float, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_fgr_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, ctypes.c_float, _I, ctypes.c_float, _I, _I, _I,
                        ctypes.c_float, _I, ctypes.c_ulonglong, ctypes.c_float, _P, _P, _P, _P, _P]),
    "ri_teaser_workspace_bytes": (_Z, [_I, _I]),
    "ri_teaser_f32": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _I, ctypes.c_float, ctypes.c_float, ctypes.c_float, _I,
                           ctypes.c_float, ctypes.c_longlong, ctypes.c_float, _P, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_fpfh_workspace_bytes": (_Z, [_I, _I, _I]),
    "ri_compute_fpfh_f32": (_I, [_P, _P, _I, _I, ctypes.c_float, _I, _P, _P, _P, _P, _Z, _P]),
    "ri_furthest_point_sample_f32": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "ri_iss_workspace_bytes": (_Z, [_I, _I]),
    "ri_iss_keypoints_f32": (_I, [_P, _I, _I, ctypes.c_float, ctypes.c_float, _P, _I, _P, _P, _P, _P, _P, _Z, _P]),
    "ri_mutual_nn_workspace_bytes":(_Z, [_I, _I, _I, _I]),
    "ri_mutual_nn_tf32x3": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _Z, _P]),
}


FPS_MAX_POINTS = 131072     # RI_FPS_MAX_POINTS


class RiError(RuntimeError):
    pass


_ERR = {-1: "bad argument", -2: "workspace missing or too small", -3: "unsupported size/configuration"}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libri_b200.so not found at %s — build it with `python %s` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for these ops." % (LIB_PATH, os.path.join(HERE, "build.py")))
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library is stale
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc, what):
    """Turn a non-zero return code of the C ABI into a Python RuntimeError (the reference's TORCH_CHECK /
    CUDA_CHECK_ERRORS role, utils.hpp:15-28, cuda_utils.cuh:28-37 — but never exit())."""
    if rc == 0:
        return
    if rc < 0:
        raise RiError("%s: %s (code %d)" % (what, _ERR.get(rc, "error"), rc))
    raise RiError("%s: CUDA error %d" % (what, rc))
