"""Functional API — the hot-path names of /root/reference/PVCNN/modules/functional/__init__.py:1-11
(avg_voxelize, spherical_avg_voxelize, trilinear_devoxelize, spherical_trilinear_devoxelize, ppf,
k_nearest_neighbor) plus the fused forms this package adds (knn_ppf, voxel_edge_features, knn_indices) and the normal
estimation, descriptors and keypoints xyz-only inputs need (estimate_normals, compute_fpfh_feature,
compute_iss_keypoints, keypoint_batch) and the reference's sampling (furthest_point_sample, gather)."""
from .devoxelization import trilinear_devoxelize, spherical_trilinear_devoxelize
from .voxelization import avg_voxelize, spherical_avg_voxelize, avg_voxelize_edge, spherical_avg_voxelize_edge
from .ppf import ppf, knn_ppf, knn_ppf_fused
from .knn import k_nearest_neighbor, knn_indices
from .edge import voxel_edge_features
from .ball_query import ball_query, grouping, local_ppf, ball_local_ppf, fold_fuser, local_ppf_features
from .lrf import change_coords, global_ppf
from .normals import estimate_normals
from .fpfh import compute_fpfh_feature
from .sampling import furthest_point_sample, gather
from .keypoints import compute_iss_keypoints, keypoint_batch
