"""CPU reference of ICP refinement and registration evaluation (row f5), for the tests and tools/bench_icp.py only.

Open3D's evaluate_registration / registration_icp (the reference wraps them in utils/open3d_func.py), one pair at a time,
numpy fp64 + scipy's k-d tree, written as the loop of csrc/icp.cu:
    T = init; res = evaluate(T); per iteration U = solve(res); T = U T; res = evaluate(T);
    stop when both |d fitness| < relative_fitness and |d rmse| < relative_rmse.
The source is transformed by the accumulated T.  The product package never imports this module.
"""
import numpy as np
from scipy.spatial import cKDTree


def kabsch(a, b):
    """Least-squares rigid transform mapping a [m,3] onto b [m,3] (rotation + translation, no scale), fp64 SVD."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    ca, cb = a.mean(0), b.mean(0)
    U, _, Vt = np.linalg.svd((a - ca).T @ (b - cb))
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))])
    R = Vt.T @ D @ U.T
    T = np.eye(4); T[:3, :3] = R; T[:3, 3] = cb - R @ ca
    return T


def _evaluate(src, tree, r, T):
    q = np.asarray(src, np.float64) @ T[:3, :3].T + T[:3, 3]
    d, j = tree.query(q, k=1, distance_upper_bound=r)
    ok = np.isfinite(d) & (d < r)
    corr = np.where(ok, j, -1).astype(np.int64)
    n = int(ok.sum())
    fitness = n / len(q)
    rmse = float(np.sqrt(np.sum(d[ok] ** 2) / n)) if n else 0.0
    return fitness, rmse, corr, q


def evaluate_registration(src, tgt, r, T=None):
    """src [n1,3], tgt [n2,3], T [4,4] -> (fitness, inlier_rmse, corr [n1] int: target index or -1)."""
    T = np.eye(4) if T is None else np.asarray(T, np.float64)
    fitness, rmse, corr, _ = _evaluate(src, cKDTree(np.asarray(tgt, np.float64)), r, T)
    return fitness, rmse, corr


def _solve_point_to_point(q, t, nt):
    return kabsch(q, t) if len(q) else np.eye(4)


def _solve_point_to_plane(q, t, nt):
    """Open3D's TransformationEstimationPointToPlane: r = (q - t).n, J = [q x n, n], J^T J x = -J^T r, identity when
    |det J^T J| < 1e-6; U = Rz(x2) Ry(x1) Rx(x0), translation x3..5."""
    J = np.concatenate([np.cross(q, nt), nt], 1)
    res = np.sum((q - t) * nt, 1)
    A, b = J.T @ J, -J.T @ res
    det = np.linalg.det(A)
    if not np.isfinite(det) or abs(det) < 1e-6:
        return np.eye(4)
    x = np.linalg.solve(A, b)
    if not np.all(np.isfinite(x)):
        return np.eye(4)
    ca, sa, cb, sb, cg, sg = np.cos(x[0]), np.sin(x[0]), np.cos(x[1]), np.sin(x[1]), np.cos(x[2]), np.sin(x[2])
    Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]])
    Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
    Rz = np.array([[cg, -sg, 0], [sg, cg, 0], [0, 0, 1]])
    U = np.eye(4); U[:3, :3] = Rz @ Ry @ Rx; U[:3, 3] = x[3:]
    return U


def _icp(src, tgt, tgt_normals, r, init, solve, max_iter, relative_fitness, relative_rmse):
    tgt = np.asarray(tgt, np.float64)
    nrm = None if tgt_normals is None else np.asarray(tgt_normals, np.float64)
    tree = cKDTree(tgt)
    T = np.eye(4) if init is None else np.asarray(init, np.float64).copy()
    fitness, rmse, corr, q = _evaluate(src, tree, r, T)
    iters = 0
    for i in range(max_iter):
        ok = corr >= 0
        U = solve(q[ok], tgt[corr[ok]], None if nrm is None else nrm[corr[ok]])
        T = U @ T
        prev = (fitness, rmse)
        fitness, rmse, corr, q = _evaluate(src, tree, r, T)
        iters = i + 1
        if abs(prev[0] - fitness) < relative_fitness and abs(prev[1] - rmse) < relative_rmse:
            break
    return T, fitness, rmse, iters, corr


def icp_point_to_point(src, tgt, r, init=None, max_iter=30, relative_fitness=1e-6, relative_rmse=1e-6):
    """-> (T [4,4] fp64, fitness, inlier_rmse, iterations, corr [n1])."""
    return _icp(src, tgt, None, r, init, _solve_point_to_point, max_iter, relative_fitness, relative_rmse)


def icp_point_to_plane(src, tgt, tgt_normals, r, init=None, max_iter=30, relative_fitness=1e-6, relative_rmse=1e-6):
    """-> (T [4,4] fp64, fitness, inlier_rmse, iterations, corr [n1])."""
    return _icp(src, tgt, tgt_normals, r, init, _solve_point_to_plane, max_iter, relative_fitness, relative_rmse)
