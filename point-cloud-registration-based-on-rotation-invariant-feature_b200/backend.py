"""`_backend`: the reference's pybind11 module surface for the hot path, served by libri_b200.so.

The reference's Python wrappers call `_backend.<fn>(at::Tensor...)` on the JIT-built module
`_multi_shape_pvcnn_backend` (/root/reference/PVCNN/modules/functional/backend.py:14-39, functions listed in
src/bindings.cpp:13-56).  This object exposes the SAME function names, positional signatures, return arity,
dtypes and shapes for every hot-path function, so the reference's functional/*.py files run unchanged when
their `from PVCNN.modules.functional.backend import _backend` resolves to it (INTEGRATION.md).

ball_query / grouping (SURVEY.md §8f row f1) and sampling (furthest_point_sampling, gather_features_*; row f12) are served
too.  Only 3-NN interpolation (SURVEY.md §2 row 14) is not provided here and raises AttributeError.
"""
import torch

from . import ops as _ops  # noqa: F401  (registers torch.ops.ri.*)

_ri = torch.ops.ri


class _Backend:
    # knn/knn.cpp:6-25
    @staticmethod
    def knn_forward_cuda(xyz1, xyz2, k):
        return list(_ri.knn(xyz1, xyz2, int(k)))

    # knn/knn.cpp:27-52
    @staticmethod
    def knn_backward_cuda(xyz1, xyz2, graddist1, graddist2, idx1, idx2):
        return list(_ri.knn_backward(xyz1, xyz2, graddist1, graddist2, idx1, idx2))

    # spherical_ppf/ppf.cpp:17-36
    @staticmethod
    def spherical_ppf_forward(coords, center, normals, center_normal):
        return _ri.ppf(coords, center, normals, center_normal)

    # voxelization/vox.cpp:17-43 -> [out (b,c,s), ind (b,n), cnt (b,s)]
    @staticmethod
    def avg_voxelize_forward(features, coords, resolution):
        return list(_ri.cube_voxelize(features, coords, int(resolution)))

    # voxelization/vox.cpp:54-78
    @staticmethod
    def avg_voxelize_backward(grad_y, indices, cnt):
        return _ri.voxelize_backward(grad_y, indices, cnt)

    # spherical_voxelization/spherical_vox.cpp:17-46
    @staticmethod
    def spherical_avg_voxelize_forward(features, coords, resolution):
        return list(_ri.sph_voxelize(features, coords, int(resolution)))

    # spherical_voxelization/spherical_vox.cpp:57-81
    @staticmethod
    def spherical_avg_voxelize_backward(grad_y, indices, cnt):
        return _ri.voxelize_backward(grad_y, indices, cnt)

    # interpolate/trilinear_devox.cpp:18-55 (is_training is ignored by the reference too: inds/wgts always returned)
    @staticmethod
    def trilinear_devoxelize_forward(r, is_training, coords, features):
        return list(_ri.trilinear_devox(coords, features, int(r)))

    # interpolate/trilinear_devox.cpp:67-90
    @staticmethod
    def trilinear_devoxelize_backward(grad_y, indices, weights, r):
        return _ri.devox_backward(grad_y, indices, weights, int(r), False)

    # interpolate/spherical_trilinear_devox.cpp:19-56
    @staticmethod
    def spherical_trilinear_devoxelize_forward(r, is_training, coords, features, g_inds):
        return list(_ri.sph_trilinear_devox(coords, features, g_inds, int(r)))

    # interpolate/spherical_trilinear_devox.cpp:68-91
    @staticmethod
    def spherical_trilinear_devoxelize_backward(grad_y, indices, weights, r):
        return _ri.devox_backward(grad_y, indices, weights, int(r), True)

    # ball_query/ball_query.cpp:6-30 (bindings.cpp name: ball_query)
    @staticmethod
    def ball_query(centers_coords, points_coords, radius, num_neighbors):
        return _ri.ball_query(centers_coords, points_coords, float(radius), int(num_neighbors))

    # grouping/grouping.cpp
    @staticmethod
    def grouping_forward(features, indices):
        return _ri.grouping(features, indices)

    @staticmethod
    def grouping_backward(grad_y, indices, n):
        return _ri.grouping_backward(grad_y, indices, int(n))

    # sampling/sampling.cpp: furthest_point_sampling(coords [B,3,N], num_samples) -> indices [B,M] int32
    @staticmethod
    def furthest_point_sampling(coords, num_samples):
        return _ri.furthest_point_sample(coords, None, int(num_samples))

    # gather_features_forward(features [B,C,N], indices [B,M]) -> [B,C,M]: grouping with one neighbour per centre
    @staticmethod
    def gather_features_forward(features, indices):
        B, C, _ = features.shape
        return _ri.grouping(features, indices.unsqueeze(-1)).view(B, C, indices.shape[1])

    # gather_features_backward(grad_y [B,C,M], indices [B,M], n) -> [B,C,n], contributions of repeated indices summed
    @staticmethod
    def gather_features_backward(grad_y, indices, n):
        return _ri.grouping_backward(grad_y.unsqueeze(-1), indices.unsqueeze(-1), int(n))


_backend = _Backend()

__all__ = ['_backend']
