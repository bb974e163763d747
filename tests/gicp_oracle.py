"""CPU reference of generalized ICP (row f9), for the tests and tools/bench_gicp.py only.

Open3D's registration_generalized_icp (Segal, Haehnel, Thrun, RSS 2009), one pair at a time, numpy fp64 + scipy's k-d tree,
written the way Open3D writes its update: per correspondence M = C_t + R C_s R^T, W = (M^-1)^(1/2) by an eigendecomposition,
r = W d, J = W J0 with J0 = [-[q]x, I3], and H = sum J^T J, g = sum J^T r; then the point-to-plane solve (identity when
|det H| < 1e-6) and U = Rz(x2) Ry(x1) Rx(x0), translation x3..5.  The loop, the correspondences and the stopping rule are
those of tests/icp_oracle.py; the source is transformed by the accumulated T.  The product package never imports this module.
"""
import numpy as np
from scipy.spatial import cKDTree

from icp_oracle import _evaluate


def covariances_from_normals(normals, epsilon):
    """C = I - (1 - eps) n^ n^T per row of normals [m,3] (n^ = n / |n|; I for a zero-length or non-finite normal)
    -> [m,3,3].  Equal to Open3D's R_{e1->n} diag(eps, 1, 1) R_{e1->n}^T."""
    n = np.asarray(normals, np.float64)
    l = np.linalg.norm(n, axis=1, keepdims=True)
    ok = np.isfinite(l) & (l > 0)
    u = np.where(ok, n / np.where(ok, l, 1.0), 0.0)
    return np.eye(3)[None] - (1.0 - epsilon) * u[:, :, None] * u[:, None, :]


def covariances_open3d_knn(xyz, epsilon, knn=20):
    """Open3D's path for a cloud without normals or covariances: the covariance of each point's knn nearest points (itself
    included), its SVD, and the singular values replaced by (1, 1, eps) -> [m,3,3]."""
    x = np.asarray(xyz, np.float64)
    _, idx = cKDTree(x).query(x, k=min(knn, len(x)))
    nb = x[idx]
    d = nb - nb.mean(1, keepdims=True)
    C = np.einsum('mki,mkj->mij', d, d) / nb.shape[1]
    U, _, Vt = np.linalg.svd(C)
    return U @ (np.array([1.0, 1.0, epsilon])[None, :, None] * Vt)


def _skew(q):
    S = np.zeros(q.shape + (3,))
    S[:, 0, 1], S[:, 0, 2], S[:, 1, 2] = -q[:, 2], q[:, 1], -q[:, 0]
    S[:, 1, 0], S[:, 2, 0], S[:, 2, 1] = q[:, 2], -q[:, 1], q[:, 0]
    return S


def jacobian0(q):
    """J0 = [-[q]x, I3] per row of q [m,3] -> [m,3,6]: d(U q)/dx at x = 0 for U = [Rz(x2) Ry(x1) Rx(x0) | x3..5]."""
    return np.concatenate([-_skew(q), np.broadcast_to(np.eye(3), q.shape[:1] + (3, 3))], 2)


def moments(q, t, Cs_rot, Ct, form='sqrt'):
    """(H [6,6], g [6]) of correspondences q -> t [m,3] with the source covariances already rotated (R C_s R^T) and the
    target's.  form='sqrt': Open3D's W = (M^-1)^(1/2) (eigh), H = sum (W J0)^T (W J0), g = sum (W J0)^T (W d);
    form='inv': H = sum J0^T M^-1 J0, g = sum J0^T M^-1 d (what csrc/icp.cu accumulates)."""
    M = Ct + Cs_rot
    Minv = np.linalg.inv(M)
    J0 = jacobian0(q)
    d = q - t
    if form == 'inv':
        return np.einsum('mka,mkl,mlb->ab', J0, Minv, J0), np.einsum('mka,mkl,ml->a', J0, Minv, d)
    w, V = np.linalg.eigh(Minv)
    W = V @ (np.sqrt(w)[:, :, None] * np.swapaxes(V, 1, 2))
    J = W @ J0
    r = np.einsum('mij,mj->mi', W, d)
    return np.einsum('mka,mkb->ab', J, J), np.einsum('mka,mk->a', J, r)


def update(H, g):
    """x = -H^-1 g, identity when |det H| < 1e-6 or x is not finite; -> U [4,4] = [Rz(x2) Ry(x1) Rx(x0) | x3..5]."""
    det = np.linalg.det(H)
    if not np.isfinite(det) or abs(det) < 1e-6:
        return np.eye(4)
    x = np.linalg.solve(H, -g)
    if not np.all(np.isfinite(x)):
        return np.eye(4)
    ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
    Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]])
    Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
    Rz = np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]])
    U = np.eye(4); U[:3, :3] = Rz @ Ry @ Rx; U[:3, 3] = x[3:]
    return U


def generalized_icp(src, tgt, r, Cs, Ct, init=None, max_iter=30, relative_fitness=1e-6, relative_rmse=1e-6,
                    form='sqrt'):
    """src [n1,3], tgt [n2,3], source / target covariances Cs [n1,3,3], Ct [n2,3,3] (each in its cloud's own frame).
    -> (T [4,4] fp64, fitness, inlier_rmse, iterations, corr [n1], min_eig: the smallest eigenvalue of H of every update)."""
    tgt = np.asarray(tgt, np.float64)
    tree = cKDTree(tgt)
    T = np.eye(4) if init is None else np.asarray(init, np.float64).copy()
    fitness, rmse, corr, q = _evaluate(src, tree, r, T)
    iters, min_eig = 0, []
    for i in range(max_iter):
        ok = corr >= 0
        R = T[:3, :3]
        H, g = moments(q[ok], tgt[corr[ok]], R @ Cs[ok] @ R.T, Ct[corr[ok]], form)
        min_eig.append(float(np.linalg.eigvalsh(H)[0]))
        T = update(H, g) @ T
        prev = (fitness, rmse)
        fitness, rmse, corr, q = _evaluate(src, tree, r, T)
        iters = i + 1
        if abs(prev[0] - fitness) < relative_fitness and abs(prev[1] - rmse) < relative_rmse:
            break
    return T, fitness, rmse, iters, corr, min_eig


def generalized_icp_normals(src, tgt, src_normals, tgt_normals, r, epsilon=1e-3, init=None, max_iter=30,
                            relative_fitness=1e-6, relative_rmse=1e-6, form='sqrt'):
    """generalized_icp with the covariances built from normals (covariances_from_normals)."""
    return generalized_icp(src, tgt, r, covariances_from_normals(src_normals, epsilon),
                           covariances_from_normals(tgt_normals, epsilon), init, max_iter, relative_fitness,
                           relative_rmse, form)
