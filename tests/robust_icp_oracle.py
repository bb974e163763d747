"""CPU reference of the robust kernels of point-to-plane and generalized ICP (row f11), for the tests and
tools/bench_robust_icp.py only.

Open3D's TransformationEstimationPointToPlane(loss) and TransformationEstimationForGeneralizedICP(epsilon, loss), one pair at a
time, numpy fp64 + scipy's k-d tree, written out the way Open3D sums them:
  point-to-plane  r = (q - t).n_t, J = [q x n_t, n_t]; H = sum w(r) J^T J, g = sum w(r) J^T r.
  generalized     M = C_t + R C_s R^T, W = (M^-1)^(1/2) by an eigendecomposition, r = W d, J = W J0; each of the three rows
                  k is weighted by w(r_k): H = sum_k w(r_k) J_k^T J_k, g = sum_k w(r_k) J_k^T r_k (the explicit per-row sum,
                  not csrc/icp.cu's A = W diag(w) W shortcut, so that the tests check the kernel's reduction).
Then tests/gicp_oracle.update (identity when |det H| < 1e-6).  The loop, the correspondences and the stopping rule are those of
tests/icp_oracle.py; the source is transformed by the accumulated T.  The product package never imports this module.
"""
import numpy as np
from scipy.spatial import cKDTree

import gicp_oracle as go
from icp_oracle import _evaluate

KERNELS_WITH_K = ('huber', 'cauchy', 'gm', 'tukey')


def weight(kernel, r):
    """Open3D's RobustKernel::Weight (recalled from its RobustKernel.cpp, not verified) of residuals r, in fp64.
    kernel: 'l2', 'l1' or (name, k), name in KERNELS_WITH_K.  'l1' gives 0 at r = 0 exactly (Open3D: +inf)."""
    r = np.asarray(r, np.float64)
    e = np.abs(r)
    name, k = (kernel, None) if isinstance(kernel, str) else (kernel[0], float(kernel[1]))
    if name == 'l2':
        return np.ones_like(r)
    if name == 'l1':
        return np.where(e > 0, 1.0 / np.where(e > 0, e, 1.0), 0.0)
    if name == 'huber':
        return k / np.maximum(e, k)
    if name == 'cauchy':
        return 1.0 / (1.0 + (r / k) ** 2)
    if name == 'gm':
        return k / (k + r * r) ** 2
    if name == 'tukey':
        return np.where(e <= k, (1.0 - (e / k) ** 2) ** 2, 0.0)
    raise ValueError(kernel)


def whitening(M):
    """W = (M^-1)^(1/2) (principal root) of symmetric positive definite M [m,3,3], by eigh."""
    lam, V = np.linalg.eigh(M)
    return V @ (lam[:, :, None] ** -0.5 * np.swapaxes(V, 1, 2))


def plane_moments(q, t, nt, kernel):
    """(H [6,6], g [6]) of robust point-to-plane over correspondences q -> t [m,3] with target normals nt [m,3]."""
    J = np.concatenate([np.cross(q, nt), nt], 1)
    res = np.sum((q - t) * nt, 1)
    w = weight(kernel, res)
    return np.einsum('m,ma,mb->ab', w, J, J), np.einsum('m,ma,m->a', w, J, res)


def gicp_moments(q, t, Cs_rot, Ct, kernel):
    """(H [6,6], g [6]) of robust generalized ICP: the per-row weighted sum of the whitened rows."""
    W = whitening(Ct + Cs_rot)
    J = W @ go.jacobian0(q)                              # [m,3,6]
    r = np.einsum('mij,mj->mi', W, q - t)                # [m,3]
    w = weight(kernel, r)
    return np.einsum('mk,mka,mkb->ab', w, J, J), np.einsum('mk,mka,mk->a', w, J, r)


def _loop(src, tgt, r, init, moments, max_iter, relative_fitness, relative_rmse):
    tgt = np.asarray(tgt, np.float64)
    tree = cKDTree(tgt)
    T = np.eye(4) if init is None else np.asarray(init, np.float64).copy()
    fitness, rmse, corr, q = _evaluate(src, tree, r, T)
    iters, min_eig = 0, []
    for i in range(max_iter):
        ok = corr >= 0
        H, g = moments(T, q[ok], tgt[corr[ok]], ok, corr[ok])
        min_eig.append(float(np.linalg.eigvalsh(H)[0]))
        T = go.update(H, g) @ T
        prev = (fitness, rmse)
        fitness, rmse, corr, q = _evaluate(src, tree, r, T)
        iters = i + 1
        if abs(prev[0] - fitness) < relative_fitness and abs(prev[1] - rmse) < relative_rmse:
            break
    return T, fitness, rmse, iters, corr, min_eig


def icp_point_to_plane(src, tgt, tgt_normals, r, kernel, init=None, max_iter=30, relative_fitness=1e-6,
                       relative_rmse=1e-6):
    """-> (T [4,4] fp64, fitness, inlier_rmse, iterations, corr [n1], min_eig: smallest eigenvalue of H per update)."""
    nt = np.asarray(tgt_normals, np.float64)
    mom = lambda T, q, t, ok, j: plane_moments(q, t, nt[j], kernel)
    return _loop(src, tgt, r, init, mom, max_iter, relative_fitness, relative_rmse)


def generalized_icp_normals(src, tgt, src_normals, tgt_normals, r, kernel, epsilon=1e-3, init=None, max_iter=30,
                            relative_fitness=1e-6, relative_rmse=1e-6):
    """Robust generalized ICP with the covariances built from normals (gicp_oracle.covariances_from_normals).
    -> (T [4,4] fp64, fitness, inlier_rmse, iterations, corr [n1], min_eig)."""
    Cs = go.covariances_from_normals(src_normals, epsilon)
    Ct = go.covariances_from_normals(tgt_normals, epsilon)

    def mom(T, q, t, ok, j):
        R = T[:3, :3]
        return gicp_moments(q, t, R @ Cs[ok] @ R.T, Ct[j], kernel)
    return _loop(src, tgt, r, init, mom, max_iter, relative_fitness, relative_rmse)
