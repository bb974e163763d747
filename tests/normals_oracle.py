"""CPU reference of normal estimation (row f6), for the tests and tools/bench_normals.py only.

Open3D's estimate_normals with KDTreeSearchParamHybrid (the reference calls it in utils/open3d_func.py:77-83), restated in
numpy fp64 + scipy's k-d tree, with the rules of csrc/normals.cu:
    C = S2/n - mu mu^T over the differences p - q of the neighbour list; normal = eigenvector of the smallest eigenvalue;
    (0,0,1) when n < 3 or trace(C) is not positive and finite; flipped when n.(camera - q) < 0 or n.prior < 0.
Clouds are point-major [N,3] here.  The product package never imports this module.
"""
import numpy as np
from scipy.spatial import cKDTree


def normals_from_neighbours(xyz, idx, count, camera=None, prior=None):
    """xyz [N,3]; idx [N,K] neighbour indices, the first count[i] of row i used; camera [3] or prior [N,3] (at most one)
    -> (normals [N,3] fp64, C [N,3,3] fp64 covariances, eigenvalues [N,3] ascending)."""
    xyz = np.asarray(xyz, np.float64)
    idx = np.asarray(idx, np.int64)
    count = np.asarray(count, np.int64)
    N, K = idx.shape
    D = xyz[np.clip(idx, 0, max(N - 1, 0))] - xyz[:, None, :]           # [N,K,3] p - q
    D = D * (np.arange(K)[None, :] < count[:, None])[:, :, None]
    n = np.maximum(count, 1).astype(np.float64)
    mu = D.sum(1) / n[:, None]
    C = np.einsum('nki,nkj->nij', D, D) / n[:, None, None] - mu[:, :, None] * mu[:, None, :]
    tr = np.trace(C, axis1=1, axis2=2)
    ok = (count >= 3) & np.isfinite(tr) & (tr > 0)
    w = np.zeros((N, 3)); nrm = np.tile(np.array([0.0, 0.0, 1.0]), (N, 1))
    if ok.any():
        w[ok], V = np.linalg.eigh(C[ok])
        nrm[ok] = V[:, :, 0]
    if camera is not None:
        dot = np.sum(nrm * (np.asarray(camera, np.float64)[None, :] - xyz), 1)
    elif prior is not None:
        dot = np.sum(nrm * np.asarray(prior, np.float64), 1)
    else:
        dot = np.ones(N)
    nrm[dot < 0] *= -1.0
    return nrm, C, w


def hybrid_neighbours(xyz, r, max_nn):
    """KDTreeSearchParamHybrid: the max_nn nearest points (the query included) with distance < r, fp64.
    -> (idx [N,max_nn] int64, -1 beyond count; count [N]; dist [N,max_nn] Euclidean, inf beyond count)."""
    xyz = np.asarray(xyz, np.float64)
    d, j = cKDTree(xyz).query(xyz, k=list(range(1, max_nn + 1)))
    ok = d < r
    count = ok.sum(1)
    return np.where(ok, j, -1), count, np.where(ok, d, np.inf)


def estimate_normals(xyz, r, max_nn=30, camera=None, prior=None):
    """xyz [N,3] -> (normals [N,3] fp64, count [N])."""
    idx, count, _ = hybrid_neighbours(xyz, r, max_nn)
    nrm, _, _ = normals_from_neighbours(xyz, idx, count, camera, prior)
    return nrm, count
